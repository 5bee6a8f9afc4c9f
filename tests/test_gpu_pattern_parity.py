"""K5 (contig x motif methylation-pattern table) cell by cell against the written-spec oracle, at the shapes it runs in
production: 70 motifs (batches of 64 + 6, motif blocks of 32 + 32 + 6), many contigs per warp, contig edges inside
warps that hold a non-ACGT letter, occurrences across tile boundaries, segments of exactly 1..65 observations around the
32/33 switch of the median kernel, the read-coverage filter boundaries and 32-bit payload sums that carry.

The oracle is a vectorised restatement of `oracle.restate.methylation_pattern` (the regex oracle loops over rows in
Python and would take minutes here), pinned to it on eight of the motifs."""
import ctypes as C
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O

MIN_COV, MIN_FRAC = 3, 0.8
BIG = 1 << 31  # rows with n_valid_cov or n_mod >= 2^31 do not fit the int32 payload and are dropped by the index build
MOD_TYPES = ("a", "m", "21839")
EDGE_SPECS = ["NGATC_a_2", "GATCN_a_1", "NA_a_1", "AN_a_0", "NGATCN_a_2", "NGAT" + "N" * 30 + "CN_a_33"]
POLY_A = (1, 2, 31, 32, 33, 64, 65)  # exact segment sizes of A_a_0; 32 holds one fraction only
TILE_BOUNDARIES = (65536, 131072)


def _specs():
    """70 specs of mod type 'a': the first batch of 64 includes motifs of 33-62 positions (H = 2), the last 6 do not."""
    fixed = ["A_a_0", "AC_a_0", "GATC_a_1", "CCGG_a_0", "GATC_a_0", "GATC_a_3", "TCGA_a_3", "CCWGG_a_2", "RGATCY_a_2",
             "GRNGAAGY_a_5", "TTCRAA_a_3", "BDHV_a_1", "GCANNNNNNTGC_a_2", "CAYNNNNRTG_a_1", "GAANNNNTTC_a_1",
             "NNGATC_a_3", "GATCNN_a_1", "NNA_a_2", "ANN_a_0", "NGATC_a_0",
             "C" + "N" * 33 + "AT_a_34", "GA" + "N" * 40 + "TC_a_42", "AC" + "N" * 56 + "GT_a_58", "A" + "N" * 60 + "T_a_61",
             "GAT" + "N" * 30 + "C_a_32"] + EDGE_SPECS
    rng = np.random.default_rng(70)
    rand = set()
    while len(fixed) + len(rand) < 64:
        L = int(rng.integers(3, 9))
        s = "".join(rng.choice(list("ACGTACGTACGTRYWSN"), size=L))
        if s[0] != "N" and s[-1] != "N":
            rand.add(f"{s}_a_{int(rng.integers(0, L))}")
    tail = ["C_a_0", "NTA_a_2", "TAN_a_0", "GATC_a_2", "YA_a_1", "CNG_a_1"]  # batch 2: short motifs only
    out = fixed + sorted(rand) + tail
    assert len(out) == len(set(out)) == 70
    return out


EXTRA_SPECS = ["CCGG_m_0", "GATC_m_3", "C_m_0", "NCG_m_1", "CGN_m_0", "CCGG_21839_1", "C_21839_0", "GNC_21839_2",
               "GATC_m_1"]


class Host:
    pass


@functools.lru_cache(maxsize=1)
def _host():
    """Seeded assembly (contig order fixes which warp of 32 chunks = 16 kbp each contig lands in) and pileup rows."""
    from nanomotif_b200 import _lib, synth
    from nanomotif_b200.device import plan_layout

    rng = np.random.default_rng(20261020)

    def rand(n, n_runs=0.0):
        return synth.random_sequence(rng, n, 0.5, n_runs).tobytes().decode()

    contigs = {}
    # one long contig across two tile boundaries, planted occurrences straddling them (both strands, modified base on
    # either side): GATC with A / T left / right of the boundary and long motifs with mod_pos >= 32
    s = bytearray(rand(150000).encode())
    b0, b1 = TILE_BOUNDARIES
    s[b0 - 2:b0 + 2] = b"GATC"                            # '+' A at b0-1 (left), '-' T at b0 (right)
    s[b1 - 3:b1 + 1] = b"GATC"                            # '+' A at b1-2, '-' T at b1-1 (both left)
    s[b0 - 20] = ord("C")
    s[b0 + 14:b0 + 16] = b"AT"                            # C N33 AT starting at b0-20: '+' mod at b0+14 (right)
    contigs["long"] = s.decode()
    contigs["mid0"] = rand(13000)  # the next contig starts at a warp boundary (163840)
    # warp A (32 chunks): 22 one-chunk contigs, one of them holds an N letter, then a 10-chunk filler
    ends = [("GATC", "GATC"), ("A", "T"), ("T", "A"), ("GATCA", "TGATC")]
    lens_a = [1, 2, 5, 17, 40, 70, 448, 300, 120, 9, 64, 33, 200, 448, 3, 61, 250, 8, 100, 31, 400]
    for i, L in enumerate(lens_a):
        a, z = ends[i % 4]
        contigs[f"wa{i:02d}"] = (a + rand(max(0, L - len(a) - len(z))) + z)[:L] if L >= len(a) + len(z) else rand(L)
        if i == 10:
            contigs["edgeN"] = "GATC" + rand(100) + "N" + rand(100) + "GATC"
    contigs["fillA"] = rand(10 * 512 - 64)
    # warp B (no N letter in reach): the same edge layout, poly-A segments, carries, 2^31 rows, filter boundaries
    contigs["edge"] = "GATC" + rand(100) + "A" + rand(100) + "GATC"
    for n in POLY_A:
        contigs[f"polyA{n}"] = "A" * n
    contigs["carry"] = "A" * 48 + rand(100)
    contigs["bigcov"] = "A" * 20 + rand(80)
    for i, L in enumerate([9, 66, 448, 129]):
        a, z = ends[i % 4]
        contigs[f"wb{i}"] = a + rand(L - len(a) - len(z)) + z
    contigs["mid1"] = rand(40000)
    contigs["mid2"] = rand(40000, 3e-4)  # N runs inside a long contig
    names = list(contigs)
    lengths = np.array([len(contigs[n]) for n in names], dtype=np.int64)
    starts, n_tiles = plan_layout(lengths)
    assert n_tiles >= 5 and int(starts[names.index("wa00")]) % (32 * _lib.CHUNK_BP) == 0

    # pileup rows
    cols = {k: [] for k in ("contig", "position", "strand", "mod_type", "n_mod", "Nvalid_cov", "n_diff", "kind")}

    def add(name, pos, strand, mt, n_mod, cov, diff, kind="random"):
        n = len(pos)
        for k, v in (("contig", name), ("strand", strand), ("mod_type", mt), ("kind", kind)):
            cols[k].append(np.full(n, v, dtype=object))
        for k, v in (("position", pos), ("n_mod", n_mod), ("Nvalid_cov", cov), ("n_diff", diff)):
            cols[k].append(np.broadcast_to(np.asarray(v, dtype=np.int64), (n,)).copy())

    def random_rows(name, pos, strand, mt):
        n = len(pos)
        cov = rng.choice(np.array([2, 3, 3, 4, 4, 5, 5, 8, 12, 30, 79]), size=n)
        diff = rng.choice(np.array([0, 0, 0, 1, 1, 2, 5, 20]), size=n)
        add(name, pos, strand, mt, rng.integers(0, cov + 1), cov, diff)

    special = {"polyA%d" % n for n in POLY_A} | {"carry", "bigcov"}
    for name in names:
        seq = np.frombuffer(contigs[name].encode(), dtype=np.uint8)
        L = len(seq)
        dense = L <= 448 or name == "fillA"
        for st in "+-":
            if name in special:
                continue
            if dense:
                pos = np.arange(L)
            else:  # 30 % of the positions, plus every position within 200 bp of a tile boundary
                pos = np.flatnonzero(rng.random(L) < 0.3)
                if name == "long":
                    near = np.concatenate([np.arange(b - 200, b + 200) for b in TILE_BOUNDARIES])
                    pos = np.union1d(pos, near)
            random_rows(name, pos, st, "a")
            c = ord("C") if st == "+" else ord("G")  # rows of two more mod types at the same C positions
            cpos = np.flatnonzero(seq == c)
            if not dense:
                cpos = cpos[rng.random(len(cpos)) < 0.3]
            random_rows(name, cpos, st, "m")
            random_rows(name, cpos, st, "21839")
    for n in POLY_A:  # '+' rows on every base, n_valid_cov in {4, 5}: heavily tied fractions
        cov = rng.choice(np.array([4, 5]), size=n)
        if n == 32:  # one segment of identical fractions
            cov, n_mod = np.full(n, 4), np.full(n, 2)
        else:
            n_mod = rng.integers(0, cov + 1)
        add(f"polyA{n}", np.arange(n), "+", "a", n_mod, cov, 0, "poly")
    k = np.arange(48)
    add("carry", k, "+", "a", BIG - 2 - k, BIG - 1 - k, 0, "carry")  # 16-bit halves of the warp sums carry
    add("bigcov", np.arange(10), "+", "a", 1, 5, 0)
    add("bigcov", [10], "+", "a", 3, BIG, 0, "big")       # n_valid_cov = 2^31
    add("bigcov", [11], "+", "a", BIG, 5, 0, "big")       # n_mod = 2^31
    add("bigcov", [12], "+", "a", 2, BIG - 1, 0)           # largest value that fits
    # exact filter boundaries at motif occurrences (a GATC starts wb0, edge, wa04, wa08): cov == min, cov one below,
    # cov / (cov + diff) == 0.8 exactly and one step below (39 / 49)
    for name, cov, diff, kind in (("wb0", 3, 0, "cov_at_min"), ("edge", 2, 0, "cov_below_min"),
                                  ("wa04", 4, 1, "frac_at_min"), ("wa08", 39, 10, "frac_below_min")):
        add(name, [1], "+", "m", 1, cov, diff, kind)  # the A of GATC_m_1; mod type 'm' has no other row at an A
    # rows that must be ignored: unknown contig, position == length, past the end, negative
    add("ghost", np.arange(5), "+", "a", 2, 5, 0, "ignored")
    add("wa03", [17, 20], "+", "a", 2, 5, 0, "ignored")
    add("wa05", [-1], "-", "a", 2, 5, 0, "ignored")
    c = {k: np.concatenate(v) for k, v in cols.items()}
    H = Host()
    H.contigs, H.names, H.lengths, H.starts, H.n_tiles = contigs, names, lengths, starts, n_tiles
    H.rows = c
    H.specs, H.all_specs = _specs(), _specs() + EXTRA_SPECS
    H.visible = (c["Nvalid_cov"] < BIG) & (c["n_mod"] < BIG) & (c["n_mod"] >= 0)
    H.want = oracle_table(contigs, c, H.all_specs, H.visible)
    return H


def oracle_table(contigs: dict, rows: dict, specs, keep=None):
    """(stats int64 [n_specs, n_contigs, 3] = n_motif_obs / sum n_mod / sum n_valid_cov, median float64 [n_specs,
    n_contigs], NaN without observations, per-spec row hit masks) of oracle.restate.methylation_pattern, vectorised:
    occurrences by O.subseq_indices_np per (contig, strand), rows joined with np.isin."""
    names = list(contigs)
    contig = np.asarray(rows["contig"]).astype(str)
    pos, strand = rows["position"], np.asarray(rows["strand"]).astype(str)
    mt = np.asarray(rows["mod_type"]).astype(str)
    n_mod, cov, diff = rows["n_mod"], rows["Nvalid_cov"], rows["n_diff"]
    with np.errstate(divide="ignore", invalid="ignore"):
        ok = (cov >= MIN_COV) & ((cov / (cov + diff)) >= MIN_FRAC)
    if keep is not None:
        ok &= keep
    by_contig = {n: np.flatnonzero(contig == n) for n in names}
    seqs = {n: np.frombuffer(contigs[n].encode(), dtype=np.uint8) for n in names}
    stats = np.zeros((len(specs), len(names), 3), dtype=np.int64)
    med = np.full((len(specs), len(names)), np.nan)
    at_occ = np.zeros((len(specs), len(pos)), dtype=bool)  # the row sits at an occurrence (filters not applied)
    for si, spec in enumerate(specs):
        iupac, want_mt, mp = spec.rsplit("_", 2)
        mp = int(mp)
        rx = "".join(O.IUPAC_TO_REGEX[ch] for ch in iupac)
        rc_rx, rc_mp = O.reverse_complement_motif(rx, mp)
        for ci, name in enumerate(names):
            r = by_contig[name]
            r = r[mt[r] == want_mt]
            if not len(r):
                continue
            fwd = O.subseq_indices_np(rx, seqs[name]) + mp
            rev = O.subseq_indices_np(rc_rx, seqs[name]) + rc_mp
            hit = np.where(strand[r] == "+", np.isin(pos[r], fwd), (strand[r] == "-") & np.isin(pos[r], rev))
            at_occ[si, r[hit]] = True
            h = r[hit & ok[r]]
            if not len(h):
                continue
            stats[si, ci] = (len(h), int(n_mod[h].sum()), int(cov[h].sum()))
            med[si, ci] = float(np.median(n_mod[h] / cov[h]))
    return stats, med, at_occ


def _mismatches(got_stats, got_med, want_stats, want_med, specs, names, limit=8):
    bad = (got_stats != want_stats).any(axis=2)
    if got_med is not None:
        bad |= ~((got_med == want_med) | (np.isnan(got_med) & np.isnan(want_med)))
    out = []
    for m, c in np.argwhere(bad)[:limit]:
        g = tuple(int(x) for x in got_stats[m, c])
        w = tuple(int(x) for x in want_stats[m, c])
        gm = "" if got_med is None else f" median {got_med[m, c]!r}"
        out.append(f"{specs[m]} @ {names[c]}: got (obs, sum n_mod, sum cov) {g}{gm}, oracle {w} median {want_med[m, c]!r}")
    return int(bad.sum()), out


def _assert_exact(got_stats, got_med, want_stats, want_med, specs, names):
    n, cells = _mismatches(got_stats, got_med, want_stats, want_med, specs, names)
    assert n == 0, f"{n} cells differ from the oracle:\n" + "\n".join(cells)


@pytest.fixture(scope="module")
def world():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from nanomotif_b200.device import DeviceAssembly, _to_device
    from nanomotif_b200.pattern import PatternIndex

    H = _host()
    asm = DeviceAssembly.from_sequences(H.contigs)
    assert asm.names == H.names and np.array_equal(asm.starts, H.starts) and asm.n_tiles == H.n_tiles
    d = asm.device
    r = H.rows
    cid = np.array([asm.index.get(n, -1) for n in r["contig"]], dtype=np.int32)
    mt = np.array([MOD_TYPES.index(m) for m in r["mod_type"]], dtype=np.uint8)
    strand = np.where(r["strand"] == "+", 0, 1).astype(np.uint8)
    rows_d = dict(contig_id=_to_device(cid, d), position=_to_device(r["position"], d), strand=_to_device(strand, d),
                  mod_type=_to_device(mt, d), n_mod=_to_device(r["n_mod"], d), Nvalid_cov=_to_device(r["Nvalid_cov"], d),
                  n_diff=_to_device(r["n_diff"], d))
    index = PatternIndex(asm, rows_d, MOD_TYPES.index("a"), MIN_COV, MIN_FRAC)

    _assert_coverage(asm, H)
    return dict(asm=asm, index=index, H=H)


def _assert_coverage(asm, H):
    """Every case the fixture claims is present, and the oracle sees it."""
    from nanomotif_b200 import _lib

    r, (stats, _med, at_occ) = H.rows, H.want
    si, ci = H.all_specs.index, H.names.index
    with np.errstate(divide="ignore", invalid="ignore"):
        passes = (r["Nvalid_cov"] >= MIN_COV) & (r["Nvalid_cov"] / (r["Nvalid_cov"] + r["n_diff"]) >= MIN_FRAC) & H.visible

    def row(name, p, st, mt="a"):
        i = np.flatnonzero((r["contig"] == name) & (r["position"] == p) & (r["strand"] == st) & (r["mod_type"] == mt))
        assert len(i) == 1, (name, p, st, mt)
        return int(i[0])

    # flanking wildcards at contig edges: in a warp with an N letter (chunk_info bit 30) and in one without
    info = asm.seq_records.view(asm.n_tiles, _lib.SEQ_REC_WORDS)[:, 2 * _lib.SEQ_PLANE_WORDS:].reshape(-1).cpu().numpy()
    chunk = {n: int(H.starts[ci(n)]) // _lib.CHUNK_BP for n in ("edgeN", "edge")}
    assert info[chunk["edgeN"]] >= 0 and info[chunk["edgeN"]] & (1 << 30)
    w = chunk["edge"] // 32 * 32
    assert info[chunk["edge"]] & (1 << 29) and not any(x >= 0 and x & (1 << 30) for x in info[w:w + 32].tolist())
    for name in ("edgeN", "edge"):
        L = len(H.contigs[name])
        # GATC at both ends: NGATC's A at 1 ('+') and its T at L-2 ('-'), GATCN's A at L-3 and T at 2 hang over the edge
        for spec, p, st in (("NGATC_a_2", 1, "+"), ("NGATC_a_2", L - 2, "-"), ("GATCN_a_1", L - 3, "+"),
                            ("GATCN_a_1", 2, "-")):
            assert not at_occ[si(spec), row(name, p, st)]
            assert at_occ[si("GATC_a_1"), row(name, p, st)]  # the GATC itself is there
        for spec in ("NA_a_1", "AN_a_0"):
            assert stats[si(spec), ci(name), 0] > 0
    # many short contigs per warp, hits off the warp's first contig
    assert sum(1 for n in H.names if H.lengths[ci(n)] <= 70 and stats[si("A_a_0"), ci(n), 0] > 0) >= 8
    assert sum(H.lengths <= 448) >= 30
    # occurrences across tile boundaries, both strands, modified base on either side
    b0, b1 = TILE_BOUNDARIES
    for spec, p, st in (("GATC_a_1", b0 - 1, "+"), ("GATC_a_1", b0, "-"), ("GATC_a_1", b1 - 2, "+"),
                        ("GATC_a_1", b1 - 1, "-"), ("C" + "N" * 33 + "AT_a_34", b0 + 14, "+")):
        assert at_occ[si(spec), row("long", p, st)], (spec, p, st)
    assert stats[si("A" + "N" * 60 + "T_a_61"), ci("long"), 0] > 0
    assert H.lengths[ci("wa03")] < 62  # a contig shorter than the longest motif
    # exact segment sizes around the 32/33 switch of the median kernel
    for n in POLY_A:
        assert stats[si("A_a_0"), ci(f"polyA{n}"), 0] == n
    # filter boundaries
    for kind, counted in (("cov_at_min", True), ("frac_at_min", True), ("cov_below_min", False), ("frac_below_min", False)):
        i = int(np.flatnonzero(r["kind"] == kind)[0])
        assert at_occ[si("GATC_m_1"), i] and passes[i] == counted, kind
    # ignored rows sit where an occurrence would be if they counted, but none is joined
    assert not at_occ[:, r["kind"] == "ignored"].any()
    # several mod types at one position (rows of a, m and 21839 at the C positions of wa20), each joined and kept
    cs = np.flatnonzero(np.frombuffer(H.contigs["wa20"].encode(), np.uint8) == ord("C")).tolist()
    assert any(all(at_occ[si(f"C_{mt}_0"), row("wa20", p, "+", mt)] and passes[row("wa20", p, "+", mt)] for mt in MOD_TYPES)
               for p in cs)
    # 32-bit sums that carry, and rows beyond int32
    assert stats[si("A_a_0"), ci("carry"), 0] >= 48 and stats[si("A_a_0"), ci("carry"), 2] > (1 << 36)
    assert (r["kind"] == "big").sum() == 2 and not H.visible[r["kind"] == "big"].any()


def _motifs(specs):
    from nanomotif_b200.motif import Motif
    from nanomotif_b200.pattern import parse_motif_spec

    return [Motif(iupac, mp).from_iupac() for iupac, _mt, mp in map(parse_motif_spec, specs)]


def _want(H, specs):
    stats, med, _ = H.want
    idx = [H.all_specs.index(s) for s in specs]
    return stats[idx], med[idx]


def _table(H):
    from nanomotif_b200.pileup import PileupTable

    r = H.rows
    return PileupTable(r["contig"], r["position"], r["strand"], np.zeros(len(r["position"])), r["mod_type"], r["Nvalid_cov"],
                       {"n_mod": r["n_mod"], "n_diff": r["n_diff"]})


def test_vectorised_oracle_equals_spec_oracle():
    """The restatement used below == oracle.restate.methylation_pattern (regex, one row at a time) on eight motifs."""
    H = _host()
    specs = ["NGATC_a_2", "GATCN_a_1", "NA_a_1", "A_a_0", "GATC_a_1", "C" + "N" * 33 + "AT_a_34", "GATC_m_1", "CCGG_21839_1"]
    r, v = H.rows, H.visible
    rows = O.methylation_pattern(H.contigs, r["contig"][v], r["position"][v], r["strand"][v], r["mod_type"][v],
                                 r["n_mod"][v], r["Nvalid_cov"][v], r["n_diff"][v], specs)
    stats, med = _want(H, specs)
    want = {}
    for name, iupac, mt, mp, value, cov, n in rows:
        want[(f"{iupac}_{mt}_{mp}", name)] = (n, cov, value)
    got = {(s, H.names[c]): (int(stats[i, c, 0]), stats[i, c, 2] / stats[i, c, 0], med[i, c])
           for i, s in enumerate(specs) for c in np.flatnonzero(stats[i, :, 0] > 0)}
    assert got == want and len(want) > 100


@pytest.mark.parametrize("median", [True, False], ids=["median", "weighted"])
@pytest.mark.parametrize("mode", ["host64", "host16", "device"])
@pytest.mark.parametrize("mpi", [1, 3, 32, None], ids=["mpi1", "mpi3", "mpi32", "mpi_default"])
def test_pattern_table_exact(world, mpi, mode, median):
    """pattern_table == oracle in every (motif, contig) cell: batches of 64 + 6 or 16 x 4 + 6 (both pinned slots reused),
    or on the device; motif blocks of 1, 3, 32 (32 + 32 + 6) or the default."""
    from nanomotif_b200.pattern import pattern_table

    H = world["H"]
    batch = 16 if mode == "host16" else 64
    stats, val = pattern_table(world["index"], _motifs(H.specs), median=median, batch=batch, motifs_per_item=mpi,
                               on_device=mode == "device")
    if mode == "device":
        stats, val = stats.cpu().numpy(), (val.cpu().numpy() if median else None)
    want_stats, want_med = _want(H, H.specs)
    _assert_exact(stats, val if median else None, want_stats, want_med, H.specs, H.names)


def _scan_on_device(index, motifs, mpi, grid_ctas, static):
    """pattern_table's on-device branch for ONE launch of all motifs: phase 0 -> nmb_segment_offsets -> phase 1 ->
    nmb_segment_median, through the static entry point (items blockIdx.x + k * gridDim.x) or the balanced one."""
    import torch

    from nanomotif_b200._lib import check, lib, ptr
    from nanomotif_b200.device import MotifPrograms, _stream, _work_counter

    asm = index.asm
    d, nc, nb = asm.device, asm.n_contigs, len(motifs)
    progs = MotifPrograms(motifs, d, strip=False)
    view = asm.view()
    stats = torch.zeros((nb * nc, 3), dtype=torch.int64, device=d)

    def scan(phase, offsets=None, cursor=None, fractions=None):
        args = (C.byref(view), ptr(index.valid), ptr(index.rank_dir), ptr(index.payload), ptr(progs.programs), nb, mpi,
                progs.max_len, phase, ptr(stats), ptr(offsets), ptr(cursor), ptr(fractions), grid_ctas)
        if static:
            check(lib.nmb_pattern_scan(*args, _stream()), "nmb_pattern_scan")
        else:
            check(lib.nmb_pattern_scan_balanced(*args, ptr(_work_counter(d)), _stream()), "nmb_pattern_scan_balanced")

    scan(0)
    offsets = torch.empty(nb * nc + 1, dtype=torch.int64, device=d)
    cursor = torch.empty(nb * nc, dtype=torch.int32, device=d)
    check(lib.nmb_segment_offsets(ptr(stats), nb * nc, ptr(offsets), ptr(cursor), _stream()), "nmb_segment_offsets")
    fractions = torch.empty(max(1, int(offsets[-1].item())), dtype=torch.float64, device=d)
    scan(1, offsets, cursor, fractions)
    med = torch.empty(nb * nc, dtype=torch.float64, device=d)
    check(lib.nmb_segment_median(ptr(fractions), ptr(offsets), nb * nc, ptr(med), _stream()), "nmb_segment_median")
    return stats.view(nb, nc, 3).cpu().numpy(), med.view(nb, nc).cpu().numpy()


@pytest.mark.parametrize("grid_ctas", [1, 7])
@pytest.mark.parametrize("static", [True, False], ids=["static", "balanced"])
def test_entry_points_and_counter_rearm(world, static, grid_ctas):
    """All 70 motifs in one launch (blocks of 32 + 32 + 6, H = 2): grid_ctas = 1 makes one CTA walk all 15 items in
    sequence (mbarrier phases, queue reset between items).  Run twice: the balanced launches draw from the same work
    counter, which the last CTA re-arms."""
    H = world["H"]
    want_stats, want_med = _want(H, H.specs)
    first = _scan_on_device(world["index"], _motifs(H.specs), 32, grid_ctas, static)
    _assert_exact(*first, want_stats, want_med, H.specs, H.names)
    again = _scan_on_device(world["index"], _motifs(H.specs), 32, grid_ctas, static)
    np.testing.assert_array_equal(again[0], first[0])
    np.testing.assert_array_equal(again[1], first[1])


def test_row_driven_path_equals_oracle_on_edge_motifs(world):
    """methylation_pattern_rows (row-driven kernels over K3 match planes) against the oracle, not just against the
    tile-driven path: flanking wildcards at contig edges in warps with and without an N letter."""
    from nanomotif_b200.pattern import methylation_pattern_rows

    H = world["H"]
    table = _table(H)
    v = H.visible  # the row-driven path narrows the payload to int32 without the index build's range check
    table = type(table)(table.contig[v], table.position[v], table.strand[v], table.fraction_mod[v], table.mod_type[v],
                        table.Nvalid_cov[v], {k: x[v] for k, x in table.extra.items()})
    specs = EDGE_SPECS + ["GATC_a_1", "A" + "N" * 60 + "T_a_61"]
    want_stats, want_med = _want(H, specs)
    got = [methylation_pattern_rows(table, H.contigs, s) for s in specs]
    _assert_exact(np.stack([g[0] for g in got]), np.stack([g[1] for g in got]), want_stats, want_med, specs, H.names)


def test_rows_beyond_int32_are_dropped(world):
    """Documented limit: rows with n_valid_cov or n_mod >= 2^31 take no part (the payload is int32); the oracle would
    count them."""
    from nanomotif_b200.pattern import pattern_table

    H = world["H"]
    stats, _ = pattern_table(world["index"], _motifs(["A_a_0"]))
    full, _, _ = oracle_table(H.contigs, H.rows, ["A_a_0"])
    c = H.names.index("bigcov")
    assert stats[0, c, 0] == _want(H, ["A_a_0"])[0][0, c, 0] == full[0, c, 0] - 2


def _expected_frame(H, specs, weighted):
    import pandas as pd

    from nanomotif_b200.pattern import COLUMNS, parse_motif_spec

    stats, med = _want(H, specs)
    mi, ci = np.nonzero(stats[:, :, 0] > 0)
    parsed = [parse_motif_spec(s) for s in specs]
    with np.errstate(divide="ignore", invalid="ignore"):
        value = stats[:, :, 1] / stats[:, :, 2] if weighted else med
    obs = stats[mi, ci, 0]
    return pd.DataFrame({
        "contig": np.array(H.names, dtype=object)[ci],
        "motif": np.array([p[0] for p in parsed], dtype=object)[mi],
        "mod_type": np.array([p[1] for p in parsed], dtype=object)[mi],
        "mod_position": np.array([p[2] for p in parsed], dtype=np.int8)[mi],
        "methylation_value": value[mi, ci],
        "mean_read_cov": stats[mi, ci, 2] / obs,
        "n_motif_obs": obs.astype(np.int32),
    }, columns=COLUMNS)


@pytest.mark.parametrize("weighted", [False, True], ids=["median", "weighted"])
def test_methylation_pattern_frame_and_bedmethyl_file(world, tmp_path, weighted):
    """The public frame for three mod types (several at one position) == the oracle's frame exactly; the same pileup
    written as bedMethyl and the assembly as FASTA give the same frame."""
    import pandas as pd

    from nanomotif_b200.pattern import MethylationOutput, methylation_pattern

    H = world["H"]
    out = MethylationOutput.WeightedMean if weighted else MethylationOutput.Median
    df = methylation_pattern(_table(H), H.contigs, H.all_specs, output_type=out)
    pd.testing.assert_frame_equal(df, _expected_frame(H, H.all_specs, weighted), check_exact=True)
    # bedMethyl rows have a non-negative start and a known contig; the rows without one are ignored either way
    r = H.rows
    keep = (r["contig"] != "ghost") & (r["position"] >= 0) & H.visible
    path = tmp_path / "p.bed"
    with open(path, "w") as f:
        for i in np.flatnonzero(keep).tolist():
            pos, cov = int(r["position"][i]), int(r["Nvalid_cov"][i])
            row = [r["contig"][i], pos, pos + 1, r["mod_type"][i], cov, r["strand"][i], pos, pos + 1, "255,0,0", cov,
                   f"{100 * r['n_mod'][i] / cov:.2f}", int(r["n_mod"][i]), 0, 0, 0, 0, int(r["n_diff"][i]), 0]
            f.write("\t".join(str(x) for x in row) + "\n")
    fa = tmp_path / "a.fasta"
    fa.write_text("".join(f">{n}\n{s}\n" for n, s in H.contigs.items()))
    pd.testing.assert_frame_equal(methylation_pattern(str(path), str(fa), H.all_specs, output_type=out), df,
                                  check_exact=True)
