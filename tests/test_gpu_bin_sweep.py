"""Per-bin sweep (sweep.BinSweep): the histograms of all bins from one launch equal, bin for bin and bit for bit, those of
one SweepIndex per bin; its counts equal K2's scans; its candidate frame equals the union of the per-bin SweepIndex
candidates plus the bipartite hits, however the bins are chunked."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O

MOD_TYPES = ["a", "m", "21839"]
CANON = {"a": "A", "m": "C", "21839": "C"}
# bin -> (contig lengths, planted motifs (regex, mod_pos, mod type)); consecutive bins share a tile at their boundary,
# bin_0 spans several tiles, bin_2 has no pileup rows, bin_6 holds only short contigs (checked against the oracle)
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


def _iupac(regex):
    """The sweep's spelling of a planted regex motif: classes -> IUPAC letters, '.' -> N."""
    sets = {"AG": "R", "CT": "Y", "AT": "W", "CG": "S", "GT": "K", "AC": "M"}
    out = []
    for tok in __import__("re").findall(r"\[[^\]]*\]|.", regex):
        out.append("N" if tok == "." else sets["".join(sorted(tok[1:-1]))] if tok.startswith("[") else tok)
    return "".join(out)


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
    asm = scorer.assembly
    assert asm.tile_span(*scorer._ranges["bin_0"])[1] >= 3
    t5, n5 = asm.tile_span(*scorer._ranges["bin_5"])
    assert t5 + n5 - 1 == asm.tile_span(*scorer._ranges["bin_6"])[0]  # bin_5 ends in the tile that holds bin_6
    return scorer, bins, pile


@pytest.fixture(scope="module")
def sweeps(world):
    from nanomotif_b200.sweep import BinSweep

    scorer = world[0]
    return {mt: BinSweep(scorer, mt) for mt in MOD_TYPES}


def _own_index(scorer, b, mt):
    from nanomotif_b200.sweep import SweepIndex

    lo, hi = scorer._ranges[b]
    return SweepIndex(scorer.assembly, scorer.pileup, MOD_TYPES.index(mt)).add(lo, hi).add_bipartite(lo, hi)


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_histograms_equal_one_index_per_bin(world, sweeps, mt):
    import torch

    from nanomotif_b200.sweep import BIP_SIZE, HIST_SIZE

    scorer = world[0]
    sw = sweeps[mt]
    assert sw.bins == list(BINS)
    raw, bip_raw = sw.raw.view(-1, HIST_SIZE), sw.bip_raw.view(-1, BIP_SIZE)
    total = 0
    for s, b in enumerate(sw.bins):
        own = _own_index(scorer, b, mt)
        assert torch.equal(raw[s], own.raw), b
        assert torch.equal(bip_raw[s], own.bip_raw), b
        assert torch.equal(sw.hist[s], own.hist), b
        assert torch.equal(sw.bip[s], own.bip), b
        if b == NO_ROWS:
            assert int(raw[s].abs().sum()) == 0 and int(bip_raw[s].abs().sum()) == 0
        total += int(raw[s].long().sum())
    assert total > 0


def test_subset_and_skipped_slots_through_the_slot_map(world):
    """bins= sweeps a subset; a contig mapped to -1 counts nowhere, so slots no contig maps to stay zero."""
    import ctypes as C

    import torch

    from nanomotif_b200 import _lib
    from nanomotif_b200.sweep import HIST_SIZE, BinSweep

    scorer = world[0]
    sub = ["bin_5", "bin_1", "bin_6"]
    sw = BinSweep(scorer, "a", bins=sub, bipartite=False)
    assert sw.raw.numel() == 3 * HIST_SIZE and sw.bip_raw is None
    for s, b in enumerate(sub):
        assert torch.equal(sw.raw.view(-1, HIST_SIZE)[s], _own_index(scorer, b, "a").raw), b
    # the entry point itself: slots 0..6 for the bins in order, only bin_1 and bin_4 mapped
    asm = scorer.assembly
    slot_of = np.full(asm.n_contigs, -1, dtype=np.int32)
    for b in ("bin_1", "bin_4"):
        lo, hi = scorer._ranges[b]
        slot_of[lo:hi] = list(BINS).index(b)
    d = asm.device
    hist = torch.zeros(len(BINS) * HIST_SIZE, dtype=torch.int32, device=d)
    cmap = torch.from_numpy(slot_of).to(d)
    base = _lib.ptr(scorer.pileup.class_records)
    _lib.check(_lib.lib.nmb_sweep_hist(C.byref(asm.view()), base, 0, asm.n_tiles, 0, 0, _lib.ptr(cmap), len(BINS),
                                       _lib.ptr(hist), None))
    torch.cuda.synchronize()
    hist = hist.view(len(BINS), HIST_SIZE)
    for s, b in enumerate(BINS):
        if b in ("bin_1", "bin_4"):
            assert torch.equal(hist[s], _own_index(scorer, b, "a").raw), b
        else:
            assert int(hist[s].abs().sum()) == 0, b


def _sample(rng, canon, n):
    iupac = "ACGTRYSWKMBDHVN"
    out = []
    while len(out) < n:
        if rng.random() < 0.7:
            s = "".join(rng.choice(list(iupac), size=int(rng.integers(4, 9))))
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

    scorer, bins, pile = world
    sw = sweeps[mt]
    rng = np.random.default_rng(22 + MOD_TYPES.index(mt))
    nonzero = n = 0
    for b in BINS:
        sample = _sample(rng, CANON[mt], 50)
        want = scorer.context(b, mt).score([nmb.Motif(s, p).from_iupac() for s, p in sample])
        for (s, p), w in zip(sample, want):
            assert sw.counts(b, s, p) == tuple(int(x) for x in w), (b, s, p)
            nonzero += int(w.sum()) > 0
            n += 1
    assert n >= 300 and nonzero > 100
    # whole tables of the bin of short contigs against the oracle's histogram + subset sums
    small = bins["bin_6"]
    sel = np.isin(pile["contig"], list(small)) & (pile["mod_type"] == mt)
    index = sw.index("bin_6")
    for k, mp in ((4, 0), (5, 2), (6, 5)):
        want_mod, want_nomod = O.sweep_table(small, pile["contig"][sel], pile["position"][sel], pile["strand"][sel],
                                             pile["fraction_mod"][sel], k, mp, CANON[mt])
        got_mod, got_nomod = index.table(k, mp, CANON[mt])
        np.testing.assert_array_equal(got_mod.cpu().numpy(), want_mod)
        np.testing.assert_array_equal(got_nomod.cpu().numpy(), want_nomod)
        assert want_mod.sum() + want_nomod.sum() > 0


def _expected_frame(scorer, b, mt, min_mean, min_mod):
    """One bin's rows: SweepIndex.candidates of every (k, mod_pos), then the bipartite hits from bipartite_table."""
    rows = []
    own = _own_index(scorer, b, mt)
    canon = CANON[mt]
    for k in range(4, 9):
        for mp in range(k):
            rows += [(b, mt, s, mp, x, y) for s, x, y in own.candidates(k, mp, canon, min_mean, min_mod)]
    code_of = {"A": 0, "T": 1, "G": 2, "C": 3}
    for g in range(4, 9):
        for a, bb in ((3, 3), (3, 4), (4, 3), (4, 4)):
            for o in range(a + bb):
                mp = o if o < a else o + g
                n_mod, n_nomod = (t.cpu().numpy().astype(np.int64) & 0xFFFFFFFF for t in own.bipartite_table(a, g, bb, mp))
                code = np.arange(4 ** (a + bb))
                xbit, ybit = (o, a + o) if o < a else (2 * a + o - a, 2 * a + bb + o - a)
                letter = ((code >> xbit) & 1) << 1 | ((code >> ybit) & 1)
                ok = (letter == code_of[canon]) & (n_mod >= min_mod) & \
                     ((5.0 + n_mod) / (10.0 + n_mod + n_nomod) >= min_mean)
                for c in np.flatnonzero(ok):
                    lt = ["ATGC"[((c >> i) & 1) << 1 | ((c >> (a + i)) & 1)] for i in range(a)]
                    rt = ["ATGC"[((c >> (2 * a + i)) & 1) << 1 | ((c >> (2 * a + bb + i)) & 1)] for i in range(bb)]
                    rows.append((b, mt, "".join(lt) + "N" * g + "".join(rt), mp, int(n_mod[c]), int(n_nomod[c])))
    return rows


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_candidates_equal_per_bin_union(world, sweeps, mt):
    scorer = world[0]
    sw = sweeps[mt]
    df = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD)
    assert list(df.columns) == ["bin", "mod_type", "motif", "mod_position", "n_mod", "n_nomod", "mean"]
    got = list(zip(df["bin"], df["mod_type"], df["motif"], df["mod_position"].tolist(), df["n_mod"].tolist(),
                   df["n_nomod"].tolist()))
    want = [r for b in BINS for r in _expected_frame(scorer, b, mt, MIN_MEAN, MIN_MOD)]
    assert got == want
    assert len(got) > 50
    m, n = df["n_mod"].to_numpy(), df["n_nomod"].to_numpy()
    np.testing.assert_array_equal(df["mean"].to_numpy(), (5.0 + m) / (10.0 + m + n))
    # planted motifs: present in their bin, absent at a higher bar from every bin without them
    strict = sw.candidates(min_mean=0.8, min_mod=MIN_MOD)
    keys = set(zip(df["bin"], df["motif"], df["mod_position"]))
    strict_keys = set(zip(strict["bin"], strict["motif"], strict["mod_position"]))
    checked = 0
    for b, (_, planted) in BINS.items():
        for regex, mp, t in planted:
            if t != mt:
                continue
            motif = _iupac(regex)
            assert (b, motif, mp) in keys, (b, motif, mp)
            others = {ob for ob, (_, pl) in BINS.items() if not any(r == regex and tt == mt for r, _, tt in pl)}
            assert not any((ob, motif, mp) in strict_keys for ob in others), (motif, mp)
            checked += 1
    assert checked >= 1


def test_chunking_and_retry_give_the_same_frame(world, sweeps):
    import pandas as pd

    sw = sweeps["a"]
    ref = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD)
    for kw in ({"scratch_bytes": 1}, {"scratch_bytes": 1 << 50}, {"capacity": 1}, {"scratch_bytes": 1, "capacity": 3}):
        pd.testing.assert_frame_equal(sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, **kw), ref)
    # a subset of k without bipartite is the matching part of the full frame
    part = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, ks=[5, 7], bipartite=False)
    want = ref[ref["motif"].str.len().isin([5, 7])].reset_index(drop=True)  # bipartite motifs have 10..16 letters
    pd.testing.assert_frame_equal(part, want)


def test_argument_errors(world, sweeps):
    from nanomotif_b200.sweep import BinSweep

    sw = sweeps["a"]
    with pytest.raises(ValueError):
        sw.candidates(min_mod=0)
    with pytest.raises(KeyError):
        sw.index("no_such_bin")
    with pytest.raises(KeyError):
        sw.counts("no_such_bin", "GATC", 1)
    with pytest.raises(KeyError):
        BinSweep(world[0], "a", bins=["bin_0", "no_such_bin"])
