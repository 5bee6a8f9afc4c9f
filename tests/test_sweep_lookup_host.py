"""Host side of the sweep lookup (sweep.pack_queries / covers, nmb_sweep_lookup): the counters a packed record addresses
against a brute-force restatement that expands each motif into its concrete motifs and places them with the header's
formulas, the coverage rules, the record layout, and the entry point's argument checks (no GPU needed)."""
import itertools
import os
import re

import numpy as np
import pytest

from nanomotif_b200 import _lib
from nanomotif_b200.sweep import LOOKUP_REASONS, covers, pack_queries

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LETTERS = "ATGCRYSWKMBDHVN"
STATES = {"A": "A", "T": "T", "G": "G", "C": "C", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC",
          "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ATGCx"}  # x: a non-ACGT contig letter
DIGIT = {"A": 0, "T": 1, "G": 2, "C": 3, "x": 4}
SHAPES = ((3, 3), (3, 4), (4, 3), (4, 4))


def _contiguous_counters(motif, mp):
    """nmb200.h: block of length k at sum_{j<k} j*2*5^j, [o][class][5^k], window = letters as base-5 digits."""
    k = len(motif)
    first = sum(j * 2 * 5 ** j for j in range(4, k))
    out = []
    for concrete in itertools.product(*(STATES[ch] for ch in motif)):
        w = 0
        for ch in concrete:
            w = w * 5 + DIGIT[ch]
        out += [first + (mp * 2 + cls) * 5 ** k + w for cls in (0, 1)]
    return out


def _bipartite_counters(motif, mp):
    """nmb200.h: g major, then (3,3) (3,4) (4,3) (4,4); block [o][class][4^(a+b)], window xL | yL<<a | xR<<2a |
    yR<<(2a+b), letter i of a part at bit i."""
    left, gap, right = re.fullmatch(r"([^N]+)(N+)([^N]+)", motif).groups()
    a, g, b = len(left), len(gap), len(right)
    block = lambda x, y: (x + y) * 2 * 4 ** (x + y)
    first = (g - 4) * sum(block(*s) for s in SHAPES) + sum(block(*s) for s in SHAPES[:SHAPES.index((a, b))])
    o = mp if mp < a else mp - g
    out = []
    for concrete in itertools.product(*(STATES[ch] for ch in left + right)):
        d = [DIGIT[ch] for ch in concrete]
        xl = sum((d[i] >> 1) << i for i in range(a))
        yl = sum((d[i] & 1) << i for i in range(a))
        xr = sum((d[a + i] >> 1) << i for i in range(b))
        yr = sum((d[a + i] & 1) << i for i in range(b))
        code = xl | yl << a | xr << 2 * a | yr << (2 * a + b)
        out += [first + (o * 2 + cls) * 4 ** (a + b) + code for cls in (0, 1)]
    return out


def _addressed(rec):
    """The counters a record addresses: every cell's class-0 and class-1 counter, in the kernel's mixed radix."""
    n = int(rec["n_pos"])
    out = []
    for ds in itertools.product(*(range(int(rec["n_states"][p])) for p in range(n))):
        c0 = int(rec["base"]) + sum(int(rec["offset"][p][d]) for p, d in enumerate(ds))
        out += [c0, c0 + int(rec["class_step"])]
    return out


def _cells(rec):
    return int(np.prod(rec["n_states"][:rec["n_pos"]].astype(np.int64)))


def _random_cases(rng):
    cases = []
    for k in range(4, 9):
        for _ in range(25):
            s = list(rng.choice(list(LETTERS), k, p=[0.1] * 4 + [0.04] * 10 + [0.2]))
            s[int(rng.integers(k))] = "ACGT"[int(rng.integers(4))]
            s = "".join(s)
            cases += [(s, mp, 0) for mp in range(k) if s[mp] in "ACGT"]
    for g in range(4, 9):
        for a, b in SHAPES:  # every bipartite (a, g, b)
            for _ in range(4):
                halves = list(rng.choice(list(LETTERS[:14]), a + b))
                halves[int(rng.integers(a + b))] = "ACGT"[int(rng.integers(4))]
                s = "".join(halves[:a]) + "N" * g + "".join(halves[a:])
                cases += [(s, mp, 1) for mp in range(len(s)) if (mp < a or mp >= a + g) and s[mp] in "ACGT"]
    return cases


def test_records_address_the_concrete_motifs():
    cases = _random_cases(np.random.default_rng(5))
    records, status = pack_queries([c[0] for c in cases], [c[1] for c in cases])
    assert (status == 0).all()
    kinds = set()
    for (motif, mp, kind), rec in zip(cases, records):
        assert int(rec["kind"]) == kind and 0 <= int(rec["n_pos"]) <= 7
        want = (_contiguous_counters if kind == 0 else _bipartite_counters)(motif, mp)
        got = _addressed(rec)
        assert len(got) == len(set(got)) == 2 * _cells(rec), motif
        assert sorted(got) == sorted(want), (motif, mp)
        kinds.add((kind, len(motif)))
    assert {k for _, k in kinds} == set(range(4, 9)) | set(range(10, 17))


def test_cells_of_concrete_and_wildcard_motifs():
    records, status = pack_queries(["GATC", "NNNANNNN", "CCWGG", "GAANNNNNNRTCG", "ACGTNNNNTGCA"], [1, 3, 1, 2, 0])
    assert (status == 0).all()
    assert [_cells(r) for r in records] == [1, 5 ** 7, 2, 2, 1]
    assert [int(r["n_pos"]) for r in records] == [0, 7, 1, 1, 0]
    assert sorted(_addressed(records[1])) == sorted(_contiguous_counters("NNNANNNN", 3))


COVERAGE = [  # (motif, mod_pos, status)
    ("GATC", 1, 0), ("GATCNNNN", 0, 0), ("NGATC", 2, 0), ("CCWGG", 1, 0), ("NNNANNNN", 3, 0),
    ("GAANNNNNNRTCG", 2, 0), ("GAANNNNNNRTCG", 12, 0), ("ACGNNNNTGC", 9, 0), ("ACGTNNNNNNNNTGCA", 15, 0),
    ("GAT", 1, 2),                   # length 3
    ("GATCGATCG", 1, 2),             # contiguous length 9
    ("GANNNNNNNRTCG", 1, 2),          # N inside a half (left half of 2 letters + N)
    ("GAANNNNNNNRNCG", 1, 2),         # N inside the right half
    ("GAANNNNNNNNNRTCG", 1, 2),       # gap 9
    ("GAANNNRTCG", 1, 2),             # gap 3
    ("GAATNNNNNNRTCGA", 1, 2),        # half of 5
    ("GNTC", 1, 5), ("GRTC", 1, 5),   # N or R at the modified position
    ("GAANNNNNNRTCG", 9, 5),          # R at the modified position of a half
    ("GAANNNNNNRTCG", 5, 4),          # modified position in the gap
    ("GATC", 4, 3), ("GATC", -1, 3), ("GAANNNNNNRTCG", 13, 3),
    ("GAUC", 1, 1), ("gatc", 1, 1), ("GA TC", 0, 1), ("GA*C", 0, 1), ("GAÄC", 0, 1),  # unknown letters
    ("", 0, 2),                      # empty string
]


def test_coverage_table():
    motifs, mps, want = zip(*COVERAGE)
    records, status = pack_queries(list(motifs), list(mps))
    assert status.tolist() == list(want)
    assert covers(list(motifs), list(mps)).tolist() == [w == 0 for w in want]
    assert (records["kind"][status != 0] == -1).all()  # nmb_sweep_lookup answers these with -1
    assert set(want) - {0} == set(LOOKUP_REASONS)
    assert covers([], []).shape == (0,) and pack_queries([], [])[0].dtype == _lib.SWEEP_QUERY_DTYPE
    with pytest.raises(ValueError):
        pack_queries(["GATC"], [1, 2])


def test_query_dtype_matches_header():
    text = open(os.path.join(ROOT, "include", "nmb200.h")).read()
    m = re.search(r"typedef struct nmb_sweep_query \{(.*?)\} nmb_sweep_query; /\* (\d+) bytes \*/", text, re.S)
    assert m and int(m.group(2)) == _lib.SWEEP_QUERY_DTYPE.itemsize == 168
    fields = re.findall(r"(int32_t|int64_t|uint8_t) (\w+)", m.group(1))
    assert [f for _, f in fields] == list(_lib.SWEEP_QUERY_DTYPE.names)
    assert _lib.SWEEP_QUERY_DTYPE.fields["offset"][1] == 28 and _lib.SWEEP_QUERY_DTYPE.fields["base"][1] == 8


def test_lookup_refuses_bad_arguments():
    lib = _lib.lib
    p = np.zeros(64, dtype=np.uint32).ctypes.data
    q = np.zeros(1, dtype=_lib.SWEEP_QUERY_DTYPE).ctypes.data
    out = np.zeros(2, dtype=np.int64).ctypes.data
    cases = [  # (hist, slots, n_rows, queries, n_queries, out, message)
        (None, None, 1, q, 1, out, b"bad argument"),
        (p, None, -1, q, 1, out, b"bad argument"),
        (p, None, 65536, q, 1, out, b"bad argument"),
        (p, None, 1, q, -1, out, b"bad argument"),
        (p, None, 1, None, 1, out, b"null queries"),
        (p, None, 1, q, 1, None, b"null output"),
    ]
    for hist, slots, n_rows, queries, n_queries, o, msg in cases:
        assert lib.nmb_sweep_lookup(hist, None, slots, n_rows, queries, n_queries, o, None) == -1
        assert msg in lib.nmb_last_error() and b"nmb_sweep_lookup" in lib.nmb_last_error()
    # nothing to compute: accepted without a launch
    assert lib.nmb_sweep_lookup(p, None, None, 0, q, 1, None, None) == 0
    assert lib.nmb_sweep_lookup(p, None, None, 65535, None, 0, None, None) == 0
