"""Sweep lookup (BinSweep.count_matrix, SweepIndex.count_many, nmb_sweep_lookup) on the device: the gathered counts of
every listed motif in every bin equal the expanded tables, the candidate frames, K2's scans and the oracle's tables.
Every comparison first checks that the exact sum fits uint32 (so the table entry, a uint32 sum, is not wrapped), then
exact equality."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O

MOD_TYPES = ["a", "m", "21839"]
CANON = {"a": "A", "m": "C", "21839": "C"}
# the fixture of tests/test_gpu_bin_sweep.py: consecutive bins share a tile at their boundary, bin_0 spans several
# tiles, bin_2 has no pileup rows, bin_6 holds only short contigs (checked against the oracle); N and R in contigs
BINS = {
    "bin_0": ((150000, 7), (("GATC", 1, "a"), ("CC[AT]GG", 1, "m"))),
    "bin_1": ((250000, 3), (("GAATTC", 2, "a"), ("GCAC......GTT", 2, "a"))),
    "bin_2": ((20000, 5), ()),
    "bin_3": ((60000, 5), (("TCGA", 3, "a"), ("CCGG", 0, "21839"))),
    "bin_4": ((120000, 2600), (("G[AG].GAAG[CT]", 5, "a"), ("GGCC", 2, "m"))),
    "bin_5": ((120000, 7), (("CTGCAG", 4, "a"), ("GGA......TCC", 2, "a"))),
    "bin_6": ((2600, 7, 3, 5), (("GAGG", 1, "a"),)),
}
NO_ROWS = "bin_2"
MIN_MEAN, MIN_MOD = 0.7, 5


@pytest.fixture(scope="module")
def world():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb
    from nanomotif_b200 import synth

    rng = np.random.default_rng(21)
    bins, cols = {}, {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    for b, (lengths, planted) in BINS.items():
        bins[b] = {}
        for j, L in enumerate(lengths):
            name = f"{b}_c{j}"
            seq = synth.random_sequence(rng, L, 0.35 + 0.04 * len(bins), 3e-5)
            if L > 1000:
                seq[rng.integers(0, L, 15)] = ord("N")  # isolated non-ACGT letters
                seq[rng.integers(0, L, 15)] = ord("R")
                seq[-1] = ord("R")
            bins[b][name] = seq.tobytes().decode()
            if b == NO_ROWS:
                continue
            p = synth.synth_pileup(seq, rng, planted=planted, depth=12, mod_types=tuple(MOD_TYPES))
            cols["contig"].append(np.full(len(p["position"]), name, dtype=object))
            cols["position"].append(p["position"])
            cols["strand"].append(np.where(p["strand"] == 0, "+", "-"))
            cols["mod_type"].append(np.asarray(MOD_TYPES, dtype=object)[p["mod_type"]])
            cols["fraction_mod"].append(p["fraction_mod"])
    pile = {k: np.concatenate(v) for k, v in cols.items()}
    scorer = nmb.MultiBinScorer(pile, bins, MOD_TYPES, 0.3, 0.7)
    return scorer, bins, pile


@pytest.fixture(scope="module")
def sweeps(world):
    from nanomotif_b200.sweep import BinSweep

    return {mt: BinSweep(world[0], mt) for mt in MOD_TYPES}


def _equal(got, want, what):
    """got: exact int64 sums; want: uint32 table entries (any integer dtype, taken mod 2^32)."""
    got, want = np.asarray(got), np.asarray(want).astype(np.int64) & 0xFFFFFFFF
    assert got.dtype == np.int64 and got.shape == want.shape, what
    assert (got >= 0).all() and (got < 1 << 32).all(), what
    bad = np.flatnonzero(got.ravel() != want.ravel())
    assert not bad.size, f"{what}: {bad.size} differ, first at {bad[0]}: {got.ravel()[bad[0]]} != {want.ravel()[bad[0]]}"


def _entries(t, idx):
    import torch

    return t[torch.as_tensor(idx, device=t.device)].cpu().numpy()


def _table_indices(rng, k, n):
    """n table indices of the (k, mod_pos) tables: half of them N-heavy (each letter N with probability 0.4)."""
    digits = rng.integers(0, 15, (n, k - 1))
    heavy = rng.random((n, k - 1)) < 0.4
    heavy[: n // 2] = False
    digits[heavy] = 14
    return (digits * 15 ** np.arange(k - 2, -1, -1)).sum(1)


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_iupac_tables(world, sweeps, mt):
    """Whole (4, mod_pos) tables of every bin, and about 20 000 sampled motifs per (k, mod_pos) for k = 5..8."""
    from nanomotif_b200.sweep import decode_motifs

    sw, canon = sweeps[mt], CANON[mt]
    rng = np.random.default_rng(40 + MOD_TYPES.index(mt))
    nonzero = 0
    for k in range(4, 9):
        for mp in range(k):
            idx = np.arange(15 ** 3) if k == 4 else np.unique(_table_indices(rng, k, 20000))
            n_mod, n_nomod = sw.count_matrix(decode_motifs(k, mp, idx, canon), np.full(idx.size, mp))
            assert n_mod.shape == (len(BINS), idx.size)
            for s, b in enumerate(sw.bins):
                tm, tn = sw.index(b).table(k, mp, canon)
                _equal(n_mod[s], _entries(tm, idx), f"{b} n_mod ({k}, {mp})")
                _equal(n_nomod[s], _entries(tn, idx), f"{b} n_nomod ({k}, {mp})")
            nonzero += int((n_mod > 0).sum())
    assert nonzero > 1000


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_bipartite_tables(world, sweeps, mt):
    """Every ACGT-half motif of one shape per gap (bipartite_table), and sampled IUPAC-half motifs
    (bipartite_iupac_table)."""
    from nanomotif_b200.sweep import BIP_LETTERS, SweepIndex, decode_bipartite, decode_bipartite_iupac

    sw, canon = sweeps[mt], CANON[mt]
    rng = np.random.default_rng(50 + MOD_TYPES.index(mt))
    nonzero = 0
    for g, (a, b) in zip(range(4, 9), ((3, 3), (3, 4), (4, 3), (4, 4), (4, 4))):
        first, n = SweepIndex.bipartite_block(a, g, b)
        counters = np.concatenate([first + o * 2 * n + np.arange(n) for o in range(a + b)])
        motifs, mps = decode_bipartite(counters)
        n_mod, n_nomod = sw.count_matrix(motifs, mps)
        for o in range(a + b):
            mp = o if o < a else o + g
            cols = slice(o * n, (o + 1) * n)
            for s, bin_name in enumerate(sw.bins):
                tm, tn = sw.index(bin_name).bipartite_table(a, g, b, mp)
                _equal(n_mod[s, cols], tm.cpu().numpy(), f"{bin_name} ({a}, {g}, {b}) mod_pos {mp}")
                _equal(n_nomod[s, cols], tn.cpu().numpy(), f"{bin_name} ({a}, {g}, {b}) mod_pos {mp}")
        nonzero += int((n_mod > 0).sum())
    for _ in range(6):
        a, b = (int(x) for x in rng.choice([3, 4], 2))
        g = int(rng.integers(4, 9))
        o = int(rng.integers(a + b))
        mp = o if o < a else o + g
        idx = np.unique(rng.integers(0, 14 ** (a + b - 1), 5000))
        motifs = decode_bipartite_iupac(a, g, b, mp, idx, canon)
        assert set("".join(motifs)) <= set(BIP_LETTERS + "N")
        n_mod, n_nomod = sw.count_matrix(motifs, np.full(idx.size, mp))
        for s, bin_name in enumerate(sw.bins):
            tm, tn = sw.index(bin_name).bipartite_iupac_table(a, g, b, mp, canon)
            _equal(n_mod[s], _entries(tm, idx), f"{bin_name} IUPAC halves ({a}, {g}, {b}) mod_pos {mp}")
            _equal(n_nomod[s], _entries(tn, idx), f"{bin_name} IUPAC halves ({a}, {g}, {b}) mod_pos {mp}")
    assert nonzero > 100


VARIANTS = ({}, {"prune": True}, {"bipartite_letters": "IUPAC"}, {"bipartite_letters": "IUPAC", "prune": True},
            {"ks": [5, 7], "bipartite": False})


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_candidate_frames(world, sweeps, mt):
    """count_matrix on a frame's (motif, mod_position) gives the frame's n_mod / n_nomod in the row's bin: the fused
    filters and the gather are two independent device paths."""
    sw = sweeps[mt]
    rows = 0
    for kw in VARIANTS:
        df = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, **kw)
        n_mod, n_nomod = sw.count_matrix(df["motif"].tolist(), df["mod_position"].to_numpy())
        at = np.array([sw.slot[b] for b in df["bin"]], dtype=np.int64)
        cols = np.arange(len(df))
        _equal(n_mod[at, cols], df["n_mod"].to_numpy(), f"candidates({kw}) n_mod")
        _equal(n_nomod[at, cols], df["n_nomod"].to_numpy(), f"candidates({kw}) n_nomod")
        rows += len(df)
    assert rows > 50


def _sample(rng, canon, n):
    """(motif, mod_pos): IUPAC 4..8-mers without flanking N and ACGT bipartite motifs, the canonical base at mod_pos."""
    out = []
    while len(out) < n:
        if rng.random() < 0.7:
            s = "".join(rng.choice(list("ACGTRYSWKMBDHVN"), size=int(rng.integers(4, 9))))
            if s[0] == "N" or s[-1] == "N":
                continue
        else:
            s = "".join(rng.choice(list("ACGT"), size=int(rng.integers(3, 5)))) + "N" * int(rng.integers(4, 9)) + \
                "".join(rng.choice(list("ACGT"), size=int(rng.integers(3, 5))))
        pos = [i for i, ch in enumerate(s) if ch == canon]
        if pos:
            out.append((s, int(rng.choice(pos))))
    return out


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_counts_match_scan(world, sweeps, mt):
    import nanomotif_b200 as nmb

    scorer = world[0]
    sw = sweeps[mt]
    rng = np.random.default_rng(60 + MOD_TYPES.index(mt))
    sample = _sample(rng, CANON[mt], 300)
    motifs, mps = [s for s, _ in sample], [p for _, p in sample]
    n_mod, n_nomod = sw.count_matrix(motifs, mps)
    for s, b in enumerate(sw.bins):
        want = scorer.context(b, mt).score([nmb.Motif(m, p).from_iupac() for m, p in sample])
        _equal(n_mod[s], want[:, 0], f"{b} n_mod against K2")
        _equal(n_nomod[s], want[:, 1], f"{b} n_nomod against K2")
    assert int((n_mod > 0).sum()) > 100


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_short_contigs_against_the_oracle(world, sweeps, mt):
    from nanomotif_b200.sweep import decode_motifs

    _, bins, pile = world
    small = bins["bin_6"]
    sel = np.isin(pile["contig"], list(small)) & (pile["mod_type"] == mt)
    total = 0
    for k, mp in ((4, 0), (5, 2), (6, 5)):
        want_mod, want_nomod = O.sweep_table(small, pile["contig"][sel], pile["position"][sel], pile["strand"][sel],
                                             pile["fraction_mod"][sel], k, mp, CANON[mt])
        idx = np.arange(want_mod.size)
        n_mod, n_nomod = sweeps[mt].count_matrix(decode_motifs(k, mp, idx, CANON[mt]), np.full(idx.size, mp),
                                                 bins=["bin_6"])
        _equal(n_mod[0], want_mod, f"bin_6 ({k}, {mp}) n_mod")
        _equal(n_nomod[0], want_nomod, f"bin_6 ({k}, {mp}) n_nomod")
        total += int(want_mod.sum() + want_nomod.sum())
    assert total > 0


def _mixed_motifs(canon):
    """Queries of 1, 2, < 32 and >= 32 cells, contiguous and bipartite, in one list."""
    return [("GATC".replace("A", canon), 1), ("NNN" + canon + "NNNN", 3), ("CCWGG", 1 if canon == "C" else None),
            ("RN" + canon + "NY", 2), ("N" + canon + "NNNNNN", 1), ("GAANNNNNNRTCG", 2 if canon == "A" else 11),
            ("BDH" + canon + "NNNNVKMS", 3), ("ACG" + canon + "NNNNNNNNTGCA", 3), (canon + "TCNNNNNNGAT", 0),
            ("SWNN" + canon + "NN", 4), ("HHH" + canon, 3)]


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_invariants(world, sweeps, mt):
    """Column sums over all bins equal one SweepIndex over the whole assembly; the bin without rows gives zeros;
    bins= subsets and order are honoured; queries of >= 32 and < 32 cells mixed in one launch give what each gives
    alone."""
    from nanomotif_b200.sweep import SweepIndex, covers

    scorer = world[0]
    sw, canon = sweeps[mt], CANON[mt]
    sample = [(m, p) for m, p in _mixed_motifs(canon) if p is not None]
    sample += _sample(np.random.default_rng(70 + MOD_TYPES.index(mt)), canon, 200)
    motifs, mps = [m for m, _ in sample], [p for _, p in sample]
    assert covers(motifs, mps).all()
    n_mod, n_nomod = sw.count_matrix(motifs, mps)
    whole = SweepIndex(scorer.assembly, scorer.pileup, MOD_TYPES.index(mt)).add().add_bipartite()
    w_mod, w_nomod = whole.count_many(motifs, mps)
    np.testing.assert_array_equal(n_mod.sum(0), w_mod)
    np.testing.assert_array_equal(n_nomod.sum(0), w_nomod)
    assert w_mod.sum() > 0
    s = sw.slot[NO_ROWS]
    assert not n_mod[s].any() and not n_nomod[s].any()
    sub = ["bin_5", NO_ROWS, "bin_0", "bin_6"]
    m_sub, u_sub = sw.count_matrix(motifs, mps, bins=sub)
    rows = [sw.slot[b] for b in sub]
    np.testing.assert_array_equal(m_sub, n_mod[rows])
    np.testing.assert_array_equal(u_sub, n_nomod[rows])
    for j, (m, p) in enumerate(sample[:11]):  # each query alone, and the single-motif path
        alone = sw.count_matrix([m], [p])
        np.testing.assert_array_equal(alone[0][:, 0], n_mod[:, j])
        np.testing.assert_array_equal(alone[1][:, 0], n_nomod[:, j])
        if len(m) <= 8 or set(m) <= set("ACGTN"):
            for b in ("bin_0", "bin_6"):
                assert sw.counts(b, m, p) == (int(n_mod[sw.slot[b], j]), int(n_nomod[sw.slot[b], j])), (b, m, p)
    for b in ("bin_1", "bin_4"):  # one bin's SweepIndex reads the same histograms
        i_mod, i_nomod = sw.index(b).count_many(motifs, mps)
        np.testing.assert_array_equal(i_mod, n_mod[sw.slot[b]])
        np.testing.assert_array_equal(i_nomod, n_nomod[sw.slot[b]])


def test_argument_errors(world, sweeps):
    from nanomotif_b200.sweep import BinSweep, SweepIndex

    scorer = world[0]
    sw = sweeps["a"]
    with pytest.raises(ValueError, match=r"motif 1 \('GANNNNNNNRTCG', mod_position 1\)"):
        sw.count_matrix(["GATC", "GANNNNNNNRTCG"], [1, 1])
    for motifs, mps in ((["GATCGATCG"], [1]), (["GRTC"], [1]), (["GATC"], [7]), (["GAANNNNNNRTCG"], [5]),
                        ([""], [0]), (["GAXC"], [1])):
        with pytest.raises(ValueError):
            sw.count_matrix(motifs, mps)
    with pytest.raises(ValueError):
        sw.count_matrix(["GATC"], [1, 2])
    flat = BinSweep(scorer, "a", bins=["bin_0", "bin_3"], bipartite=False)
    with pytest.raises(ValueError, match="bipartite=False"):
        flat.count_matrix(["GATC", "GAANNNNNNRTCG"], [1, 2])
    got = flat.count_matrix(["GATC"], [1])[0]
    assert got.shape == (2, 1) and got[0, 0] == sw.count_matrix(["GATC"], [1], bins=["bin_0"])[0][0, 0]
    index = SweepIndex(scorer.assembly, scorer.pileup, 0).add(*scorer._ranges["bin_3"])
    with pytest.raises(ValueError, match="no bipartite histogram"):
        index.count_many(["GAANNNNNNRTCG"], [2])
    assert index.count_many(["GATC"], [1])[0][0] == sw.counts("bin_3", "GATC", 1)[0]
    with pytest.raises(KeyError):
        sw.count_matrix(["GATC"], [1], bins=["bin_0", "no_such_bin"])
    with pytest.raises(ValueError, match="twice"):
        sw.count_matrix(["GATC"], [1], bins=["bin_0", "bin_0"])
    for m, u in (sw.count_matrix([], []), sw.count_matrix(["GATC"], [1], bins=[]), sw.count_matrix([], [], bins=[])):
        assert m.dtype == u.dtype == np.int64 and m.size == u.size == 0
    assert sw.count_matrix([], [])[0].shape == (len(BINS), 0)
    assert index.count_many([], [])[0].shape == (0,)


def test_unreadable_records_give_minus_one(world, sweeps):
    """Records the kernel cannot read safely (here: an uncovered motif's kind -1, an offset past the histogram) and
    negative slots are answered without a read outside the histograms."""
    import torch

    from nanomotif_b200 import _lib
    from nanomotif_b200.sweep import HIST_SIZE, _lookup, pack_queries

    sw = sweeps["a"]
    records, status = pack_queries(["GATC", "GRTC", "NNNANNNN"], [1, 1, 3])
    assert status.tolist() == [0, 5, 0]
    records = np.concatenate([records, records[:1]])
    records["base"][3] = HIST_SIZE - 1
    d = sw.asm.device
    slots = torch.tensor([0, -1, 3], dtype=torch.int32, device=d)
    with torch.cuda.device(d):
        out = _lookup(sw.hist, None, slots, 3, records).cpu().numpy()
    want0 = sw.count_matrix(["GATC", "NNNANNNN"], [1, 3], bins=[sw.bins[0], sw.bins[3]])
    assert out[0, 0].tolist() == [want0[0][0, 0], want0[1][0, 0]]
    assert out[2, 2].tolist() == [want0[0][1, 1], want0[1][1, 1]]
    assert (out[:, 1] == -1).all() and (out[:, 3] == -1).all()
    assert (out[1] == np.array([[0, 0], [-1, -1], [0, 0], [-1, -1]])).all()
    assert _lib.SWEEP_QUERY_DTYPE.itemsize == 168
