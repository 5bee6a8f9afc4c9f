"""Host side of the degenerate bipartite sweep (halves over the 14 IUPAC letters other than N), no GPU needed: the
vectorised decoder inverts SweepIndex.bipartite_iupac_index; a numpy restatement of slice + 4-state -> 14-letter
subset sum equals brute-force summation over the concrete motifs; the C entry points refuse bad arguments before
any CUDA call."""
import itertools

import numpy as np
import pytest

from nanomotif_b200 import _lib
from nanomotif_b200.sweep import BIP_LETTERS, SweepIndex, bip_iupac_scratch_bytes, decode_bipartite_iupac

SHAPES = [(3, 3), (3, 4), (4, 3), (4, 4)]
CONCRETE = {"A": "A", "T": "T", "G": "G", "C": "C", "R": "AG", "Y": "CT", "S": "GC", "W": "AT", "K": "GT", "M": "AC",
            "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG"}
DIGIT = {"A": 0, "T": 1, "G": 2, "C": 3}


def _code(letters, a, b):
    """Bit-planar window index of concrete halves (SweepIndex.bipartite_index of the split)."""
    return SweepIndex.bipartite_index("".join(letters[:a]), "".join(letters[a:]))


def restate_table(block, a, b, o, canonical):
    """numpy restatement of nmb_sweep_bip_iupac_slice + nmb_sweep_bip_iupac_expand over one finished
    [4^(a+b)] block of one (shape, offset, class): slice to base-4 digits (first letter most significant), then the
    14-letter subset sum axis by axis, last axis first."""
    n = a + b - 1
    w = np.arange(4 ** n)
    code = np.zeros(w.size, dtype=np.int64)
    rest = w.copy()
    for p in reversed(range(a + b)):
        if p == o:
            d = np.full(w.size, DIGIT[canonical])
        else:
            d, rest = rest % 4, rest // 4
        xbit, ybit = (p, a + p) if p < a else (2 * a + p - a, 2 * a + b + p - a)
        code |= (d >> 1) << xbit | (d & 1) << ybit
    t = block[code].astype(np.int64)
    sums = np.array([[int(c in CONCRETE[l]) for c in "ATGC"] for l in BIP_LETTERS])  # [14][4]
    for step in range(n):
        outer, inner = 4 ** (n - 1 - step), 14 ** step
        t = np.einsum("lj,ojr->olr", sums, t.reshape(outer, 4, inner)).reshape(-1)
    return t


def test_decode_inverts_index():
    rng = np.random.default_rng(31)
    for g in range(4, 9):
        for a, b in SHAPES:
            for o in range(a + b):
                mp = o if o < a else o + g
                canon = "ATGC"[int(rng.integers(0, 4))]
                idx = rng.integers(0, 14 ** (a + b - 1), 60)
                got = decode_bipartite_iupac(a, g, b, mp, idx, canon)
                for i, s in zip(idx.tolist(), got.tolist()):
                    left, right = s[:a], s[a + g:]
                    assert s == left + "N" * g + right and (left + right)[o] == canon
                    assert SweepIndex.bipartite_iupac_index(left, right, o) == i
    # every letter appears at every free half position
    got = decode_bipartite_iupac(3, 4, 3, 1, np.arange(14 ** 5), "A")
    halves = np.array([list(s[:3] + s[7:]) for s in got])
    for p in (0, 2, 3, 4, 5):
        assert set(halves[:, p]) == set(BIP_LETTERS)
    assert set(halves[:, 1]) == {"A"}
    assert decode_bipartite_iupac(4, 8, 4, 0, np.zeros(0, np.int64)).size == 0


@pytest.mark.parametrize("a,b", SHAPES)
def test_restated_zeta_equals_brute_force(a, b):
    rng = np.random.default_rng(32 + a * 10 + b)
    block = rng.integers(0, 1000, 4 ** (a + b)).astype(np.int64)
    for o in (0, a - 1, a, a + b - 1):
        canon = "ATGC"[o % 4]
        table = restate_table(block, a, b, o, canon)
        assert table.size == 14 ** (a + b - 1)
        idx = rng.integers(0, table.size, 400)
        for i in idx.tolist():
            letters, rest = [], i
            for _ in range(a + b - 1):
                letters.append(BIP_LETTERS[rest % 14])
                rest //= 14
            letters = letters[::-1]
            letters.insert(o, canon)
            want = sum(int(block[_code(c, a, b)]) for c in itertools.product(*(CONCRETE[l] for l in letters)))
            assert table[i] == want, (a, b, o, "".join(letters))
        # concrete halves: the entry is the counter itself
        concrete = [l for l in itertools.product("ATGC", repeat=a + b - 1)][:200]
        for c in concrete:
            full = list(c)
            full.insert(o, canon)
            i = SweepIndex.bipartite_iupac_index("".join(full[:a]), "".join(full[a:]), o)
            assert table[i] == block[_code(full, a, b)]


def test_scratch_per_bin():
    assert bip_iupac_scratch_bytes() == 2 * 4 * (16 * 14 ** 5 + 4 * 14 ** 6) == 309_786_624


def test_slice_expand_and_filter_refuse_bad_arguments():
    lib = _lib.lib
    buf = np.zeros(16, dtype=np.uint32)
    p = buf.ctypes.data

    def slice_(a=3, g=4, b=3, mp=0, cls=0, canon=0, hist=p, dst=p, n_slots=1):
        return lib.nmb_sweep_bip_iupac_slice(hist, n_slots, a, g, b, mp, cls, canon, dst, None)

    for kw in ({"a": 2}, {"a": 5}, {"b": 5}, {"g": 3}, {"g": 9}, {"mp": 3}, {"mp": 6}, {"mp": -1}, {"mp": 10},
               {"canon": 4}, {"canon": -1}, {"cls": 2}, {"hist": None}, {"dst": None}, {"n_slots": 0}):
        assert slice_(**kw) == -1, kw
        assert b"nmb_sweep_bip_iupac_slice" in lib.nmb_last_error()
    assert slice_(mp=5) == -1 and b"outside the halves" in lib.nmb_last_error()
    assert lib.nmb_sweep_bip_iupac_expand(None, p, 1, 1, None) == -1
    assert lib.nmb_sweep_bip_iupac_expand(p, p, 0, 1, None) == -1
    f = lib.nmb_sweep_bip_iupac_expand_filter
    n_out = np.zeros(1, dtype=np.int64).ctypes.data
    for prune in (0, 1):
        assert f(p, p, 1, 14, 0.7, 5, prune, None, 10, n_out, None) == -1  # null output with room for records
        assert b"null output" in lib.nmb_last_error()
        assert f(p, p, 1, 14, 0.7, 5, prune, p, 10, None, None) == -1
        assert f(p, p, 1, 14 ** 9, 0.7, 5, prune, p, 10, n_out, None) == -1  # table index past 32 bits
        assert f(p, p, 1, 14, 0.7, -1, prune, p, 10, n_out, None) == -1
