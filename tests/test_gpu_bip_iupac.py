"""Degenerate bipartite sweep: X{3,4} N{4..8} Y{3,4} motifs whose halves use the 14 IUPAC letters other than N, per bin
(SweepIndex.bipartite_iupac_table, BinSweep.bipartite_iupac_counts, BinSweep.candidates(bipartite_letters="IUPAC")),
against K2 scans of the same motifs written as regex, the numpy restatement of slice + subset sum, oracle/restate.py
and the ACGT bipartite tables."""
import itertools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O
from test_bip_iupac_host import restate_table

MOD_TYPES = ["a", "m", "21839"]
CANON = {"a": "A", "m": "C", "21839": "C"}
SHAPES = ((3, 3), (3, 4), (4, 3), (4, 4))
PLANTED = (("GAA......[AG]TCG", 2), ("AAC......GT[AG]C", 1), ("TCA.......[AG]TTC", 2))  # EcoR124I, StySPI, EcoDXXI
# bin -> (contig lengths, planted motifs); consecutive bins share tiles, bin_2 has no pileup rows, bin_4 holds contigs
# shorter than the shortest bipartite span (10)
BINS = {
    "bin_0": ((150000, 7), ((PLANTED[0] + ("a",)), ("GATC", 1, "a"), ("CC[AT]GG", 1, "m"))),
    "bin_1": ((120000, 3), ((PLANTED[1] + ("a",)), ("CCGG", 0, "21839"))),
    "bin_2": ((20000, 5), ()),
    "bin_3": ((100000, 2600), ((PLANTED[2] + ("a",)), ("GGCC", 2, "m"))),
    "bin_4": ((2600, 7, 3, 5), (("GAGG", 1, "a"),)),
}
NO_ROWS = "bin_2"
# one occurrence of GAA......[AG]TCG each: non-ACGT letters in the gap (it counts), an R where the half has [AG] and an
# N in the left half (they count for no motif)
EDGE = {"gap_NR": "TTGAAACRTNGATCGTT", "half_R": "TTGAAACGTAGRTCGTT", "half_N": "TTGNAACGTAGATCGTT"}
MIN_MEAN, MIN_MOD = 0.7, 5
_RX = str.maketrans(O.IUPAC_TO_REGEX)


def _regex(iupac):
    return iupac.translate(_RX)


def _iupac(regex):
    sets = {"AG": "R", "CT": "Y", "AT": "W", "CG": "S", "GT": "K", "AC": "M"}
    toks = __import__("re").findall(r"\[[^\]]*\]|.", regex)
    return "".join("N" if t == "." else sets["".join(sorted(t[1:-1]))] if t.startswith("[") else t for t in toks)


@pytest.fixture(scope="module")
def world():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb
    from nanomotif_b200 import synth

    rng = np.random.default_rng(41)
    bins, cols = {}, {k: [] for k in ("contig", "position", "strand", "mod_type", "fraction_mod")}
    n_half = n_gap = 0
    specs = {b: (tuple(synth.random_sequence(rng, L, 0.35 + 0.05 * i, 3e-5) for L in lengths), planted)
             for i, (b, (lengths, planted)) in enumerate(BINS.items())}
    for name, text in EDGE.items():
        specs[name] = ((np.frombuffer(text.encode(), dtype=np.uint8).copy(),), ((PLANTED[0] + ("a",)),))
    for b, (seqs, planted) in specs.items():
        bins[b] = {}
        for j, seq in enumerate(seqs):
            name = f"{b}_c{j}"
            L = len(seq)
            if L > 1000:
                for letter in (b"N", b"R"):  # isolated non-ACGT letters, in halves and in gaps of many windows
                    at = rng.integers(20, L - 20, 15)
                    seq[at] = ord(letter)
                    rows_near = [(seq[p - 2:p + 3] == ord("A")).any() for p in at]  # a row of 'a' within 2 letters
                    n_half += int(np.sum(rows_near))
                    n_gap += int(np.sum([(seq[p + 5:p + 9] == ord("A")).any() for p in at]))
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
    # the cases the file is about
    assert n_half > 20 and n_gap > 20
    for name in EDGE:  # the A of GAA at position 4 carries a '+' row of mod type a
        assert np.any((pile["contig"] == f"{name}_c0") & (pile["position"] == 4) & (pile["strand"] == "+") &
                      (pile["mod_type"] == "a")), name
    assert not np.any(np.isin(pile["contig"], list(bins[NO_ROWS])))
    assert min(len(s) for s in bins["bin_4"].values()) < 10
    spans = [asm.tile_span(*scorer._ranges[b]) for b in bins]
    assert any(t0 + n0 - 1 == t1 for (t0, n0), (t1, _) in zip(spans, spans[1:]))  # neighbouring bins share a tile
    assert spans[0][1] >= 3
    return scorer, bins, pile


@pytest.fixture(scope="module")
def sweeps(world):
    from nanomotif_b200.sweep import BinSweep

    return {mt: BinSweep(world[0], mt) for mt in MOD_TYPES}


def _k2(scorer, bin_names, mt, iupac_motifs, mod_positions):
    """K2 counts [n, 2] in each of `bin_names` of IUPAC motifs written as regex, in batches."""
    import nanomotif_b200 as nmb

    ctxs = [scorer.context(b, mt) for b in bin_names]
    out = [[] for _ in bin_names]
    step = 1 << 17
    for s in range(0, len(iupac_motifs), step):
        motifs = [nmb.Motif(_regex(m), int(p)) for m, p in zip(iupac_motifs[s:s + step], mod_positions[s:s + step])]
        for o, c in zip(out, scorer.score_batch([(ctx, motifs) for ctx in ctxs])):
            o.append(c)
    return [np.concatenate(o).astype(np.int64) for o in out]


def _host(t):
    return t.cpu().numpy().astype(np.int64) & 0xFFFFFFFF


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_whole_tables_equal_k2(world, sweeps, mt):
    from nanomotif_b200.sweep import decode_bipartite_iupac

    scorer = world[0]
    total = 0
    for a, g, b in ((3, 4, 3), (3, 8, 3)):
        for o in range(a + b):
            mp = o if o < a else o + g
            motifs = decode_bipartite_iupac(a, g, b, mp, np.arange(14 ** 5), CANON[mt])
            wants = _k2(scorer, ("bin_0", "bin_3"), mt, motifs, np.full(motifs.size, mp))
            for bin_name, want in zip(("bin_0", "bin_3"), wants):
                n_mod, n_nomod = sweeps[mt].index(bin_name).bipartite_iupac_table(a, g, b, mp, CANON[mt])
                assert n_mod.numel() == 537_824
                np.testing.assert_array_equal(_host(n_mod), want[:, 0], err_msg=str((bin_name, a, g, b, mp)))
                np.testing.assert_array_equal(_host(n_nomod), want[:, 1], err_msg=str((bin_name, a, g, b, mp)))
                total += int(want.sum())
    assert total > 1_000_000


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_sampled_tables(world, sweeps, mt):
    import torch

    from nanomotif_b200.sweep import BIP_LETTERS, SweepIndex

    scorer, bins, pile = world
    sw = sweeps[mt]
    canon = CANON[mt]
    # whole (4, g, 3) and (3, g, 4) tables == the numpy restatement on the device's own finished ACGT histogram
    s = sw.slot["bin_0"]
    for a, g, b, mp in ((4, 5, 3, 1), (3, 7, 4, 3 + 7 + 2)):
        o = mp if mp < a else mp - g
        first, n = SweepIndex.bipartite_block(a, g, b)
        bip = _host(sw.bip[s])
        got = sw.index("bin_0").bipartite_iupac_table(a, g, b, mp, canon)
        for cls in (0, 1):
            block = bip[first + (o * 2 + cls) * n:][:n]
            np.testing.assert_array_equal(_host(got[cls]), restate_table(block, a, b, o, canon), err_msg=str((a, g, b, cls)))
        assert int(got[0].long().sum()) > 0
    # 2000 sampled (4, g, 4) motifs == K2: every letter at every half position, the modified base in both halves
    rng = np.random.default_rng(42 + MOD_TYPES.index(mt))
    letters = list(BIP_LETTERS)
    samples = []
    for _ in range(2000):
        g, o = int(rng.integers(4, 9)), int(rng.integers(0, 8))
        halves = [letters[i] for i in rng.integers(0, 14, 8)]
        halves[o] = canon
        samples.append(("".join(halves[:4]), g, "".join(halves[4:]), o if o < 4 else o + g))
    seen = {(i, ch) for left, _, right, mp in samples for i, ch in enumerate(left + right)}
    assert seen >= {(i, ch) for i in range(8) for ch in BIP_LETTERS}
    assert {mp < 4 for *_, mp in samples} == {True, False}
    motifs = [left + "N" * g + right for left, g, right, _ in samples]
    wants = _k2(scorer, ("bin_0", "bin_1"), mt, motifs, [mp for *_, mp in samples])
    for bin_name, want in zip(("bin_0", "bin_1"), wants):
        index = sw.index(bin_name)
        got = np.zeros_like(want)
        for key in sorted({(g, mp) for _, g, _, mp in samples}):  # one table per (gap, modified position)
            rows = [i for i, (_, g, _, mp) in enumerate(samples) if (g, mp) == key]
            j = torch.tensor([SweepIndex.bipartite_iupac_index(samples[i][0], samples[i][2], key[1] if key[1] < 4 else
                                                               key[1] - key[0]) for i in rows], device=sw.bip.device)
            for cls, t in enumerate(index.bipartite_iupac_table(4, key[0], 4, key[1], canon)):
                got[rows, cls] = _host(t[j])
        np.testing.assert_array_equal(got, want, err_msg=bin_name)
        assert (want.sum(axis=1) > 0).sum() > 500
    # 200 of them through BinSweep.bipartite_iupac_counts == oracle/restate.py
    if mt == "a":
        contigs = bins["bin_1"]
        sel = np.isin(pile["contig"], list(contigs)) & (pile["mod_type"] == mt)
        sub = {k: v[sel] for k, v in pile.items()}
        nonzero = 0
        for left, g, right, mp in samples[:200]:
            ref = _oracle_counts(sub, contigs, left + "N" * g + right, mp)
            assert sw.bipartite_iupac_counts("bin_1", left, g, right, mp) == ref, (left, g, right, mp)
            nonzero += sum(ref) > 0
        assert nonzero > 50


def _oracle_counts(pile, contigs, iupac, mod_pos, low=0.3, high=0.7):
    rx = _regex(iupac)
    rc_rx, rc_pos = O.reverse_complement_motif(rx, mod_pos)
    n_mod = n_nomod = 0
    for name, seq in contigs.items():
        sel = pile["contig"] == name
        pos, strand, frac = pile["position"][sel], pile["strand"][sel], pile["fraction_mod"][sel]
        arr = np.frombuffer(seq.encode(), dtype=np.uint8)
        for st, motif, mp in (("+", rx, mod_pos), ("-", rc_rx, rc_pos)):
            on = strand == st
            a, b = O.methylated_motif_occourances(motif, mp, arr, pos[on & (frac >= high)], pos[on & (frac <= low)], True)
            n_mod += len(a)
            n_nomod += len(b)
    return n_mod, n_nomod


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_acgt_entries_equal_bipartite_table(world, sweeps, mt):
    import torch

    from nanomotif_b200.sweep import SweepIndex

    canon = CANON[mt]
    for bin_name in ("bin_0", "bin_4"):
        index = sweeps[mt].index(bin_name)
        for g in range(4, 9):
            for a, b in SHAPES:
                for o in range(a + b):
                    mp = o if o < a else o + g
                    acgt = index.bipartite_table(a, g, b, mp)
                    iupac = index.bipartite_iupac_table(a, g, b, mp, canon)
                    codes, idx = [], []
                    for c in itertools.product("ATGC", repeat=a + b - 1):
                        full = list(c)
                        full.insert(o, canon)
                        codes.append(SweepIndex.bipartite_index("".join(full[:a]), "".join(full[a:])))
                        idx.append(SweepIndex.bipartite_iupac_index("".join(full[:a]), "".join(full[a:]), o))
                    idx, codes = (torch.tensor(x, device=acgt[0].device) for x in (idx, codes))
                    for cls in (0, 1):
                        assert torch.equal(iupac[cls][idx], acgt[cls][codes]), (bin_name, a, g, b, mp, cls)


def test_non_acgt_contig_letters(world, sweeps):
    """A non-ACGT contig letter inside a half counts for no motif, inside the gap it counts like any letter."""
    scorer = world[0]
    sw = sweeps["a"]
    for name, expect_rows in (("gap_NR", True), ("half_R", False), ("half_N", False)):
        for left, right in (("GAA", "RTCG"), ("GAA", "VTCG"), ("GRA", "DTCG"), ("GAA", "ATCG")):
            got = sw.bipartite_iupac_counts(name, left, 6, right, 2)
            want = _k2(scorer, [name], "a", [left + "N" * 6 + right], [2])[0][0]
            assert got == tuple(want.tolist()), (name, left, right)
            assert (sum(got) > 0) == expect_rows, (name, left, right, got)


def _frame_rows(df):
    return list(zip(df["bin"], df["motif"], df["mod_position"].tolist(), df["n_mod"].tolist(), df["n_nomod"].tolist()))


def _table_rows(sw, mt):
    """Every bin's degenerate bipartite candidates from the full tables, filtered with torch in float64 as
    sweep_pass does, in the frame's order (bin, gap, shape, modified position, index)."""
    import torch

    from nanomotif_b200.sweep import decode_bipartite_iupac

    rows = []
    for b in sw.bins:
        index = sw.index(b)
        for g in range(4, 9):
            for a, bb in SHAPES:
                for o in range(a + bb):
                    mp = o if o < a else o + g
                    m, n = (t.long() & 0xFFFFFFFF for t in index.bipartite_iupac_table(a, g, bb, mp, CANON[mt]))
                    ok = (m >= MIN_MOD) & ((5.0 + m.double()) / (10.0 + m.double() + n.double()) >= MIN_MEAN)
                    idx = torch.nonzero(ok).view(-1)
                    motifs = decode_bipartite_iupac(a, g, bb, mp, idx.cpu().numpy(), CANON[mt])
                    rows += list(zip([b] * motifs.size, motifs.tolist(), [mp] * motifs.size, m[idx].tolist(),
                                     n[idx].tolist()))
    return rows


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_candidate_frame(world, sweeps, mt):
    import pandas as pd

    from nanomotif_b200.sweep import MAX_K, bip_iupac_scratch_bytes

    sw = sweeps[mt]
    default = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD)
    pd.testing.assert_frame_equal(sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite_letters="ACGT"), default)
    df = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite_letters="IUPAC")
    assert list(df.columns) == list(default.columns)
    contiguous = df["motif"].str.len() <= MAX_K
    pd.testing.assert_frame_equal(df[contiguous].reset_index(drop=True),
                                  default[default["motif"].str.len() <= MAX_K].reset_index(drop=True))
    # the degenerate bipartite rows == the full tables filtered, in the same order
    bip_rows = _frame_rows(df[~contiguous])
    assert bip_rows == _table_rows(sw, mt)
    assert len(bip_rows) > 100
    m, n = df["n_mod"].to_numpy(), df["n_nomod"].to_numpy()
    np.testing.assert_array_equal(df["mean"].to_numpy(), (5.0 + m) / (10.0 + m + n))
    # restricted to ACGT halves: the default frame's bipartite rows (as a set: the two index orders differ)
    acgt = [r for r in bip_rows if set(r[1]) <= set("ACGTN")]
    assert sorted(acgt) == sorted(_frame_rows(default[default["motif"].str.len() > MAX_K]))
    assert len(acgt) < len(bip_rows)
    if mt == "a":  # any chunking of the bins and a capacity retry give the same frame
        for kw in ({"scratch_bytes": 1}, {"scratch_bytes": 1 << 50}, {"capacity": 1},
                   {"scratch_bytes": 2 * bip_iupac_scratch_bytes(), "capacity": 3}):
            pd.testing.assert_frame_equal(sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite_letters="IUPAC",
                                                        **kw), df)


def test_planted_motifs(world, sweeps):
    scorer = world[0]
    sw = sweeps["a"]
    df = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite_letters="IUPAC")
    strict = sw.candidates(min_mean=0.8, min_mod=MIN_MOD, bipartite_letters="IUPAC")
    keys = {(b, s, p): (x, y) for b, s, p, x, y in _frame_rows(df)}
    strict_keys = set((b, s, p) for b, s, p, *_ in _frame_rows(strict))
    for regex, mp in PLANTED:
        motif = _iupac(regex)
        planted_in = [b for b, (_, pl) in BINS.items() if any(r == regex for r, *_ in pl)]
        assert len(planted_in) == 1
        for b in planted_in:
            assert (b, motif, mp) in keys, (b, motif, mp)
            want = _k2(scorer, [b], "a", [motif], [mp])[0][0]
            assert keys[(b, motif, mp)] == tuple(want.tolist())
        others = [b for b in sw.bins if b not in planted_in and b not in EDGE]
        assert not any((b, motif, mp) in strict_keys for b in others), motif
    with pytest.raises(ValueError):
        sw.candidates(bipartite_letters="acgt")
    with pytest.raises(ValueError):
        sw.bipartite_iupac_counts("bin_0", "GAN", 6, "RTCG", 2)  # N in a half
    with pytest.raises(ValueError):
        sw.bipartite_iupac_counts("bin_0", "GAA", 6, "RTCG", 4)  # in the gap
    with pytest.raises(ValueError):
        sw.bipartite_iupac_counts("bin_0", "GRA", 6, "RTCG", 1)  # a degenerate modified position
