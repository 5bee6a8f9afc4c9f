"""Candidate pruning of the per-bin sweep (BinSweep.candidates(prune=True), nmb_sweep_*_prune): the pruned rows equal
oracle/sweep_prune.py over the oracle's own tables (k = 4..6) and over the device's finished bipartite
histograms expanded in numpy; for k = 7, 8 and the (4, g, 4) degenerate bipartite tables they equal a torch
restatement of the rule over the device tables that the existing tests pin to the oracle.  The pruned frame is a
subsequence of the full one for any chunking, every planted motif survives, and pruning removes rows in every bin
with planted motifs."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O
from oracle import sweep_prune as P

# the fixture of tests/test_gpu_bin_sweep.py: bins that share tiles, a bin without rows, contigs of 3-7 bp, N and R
# contig letters, three mod types
MOD_TYPES = ["a", "m", "21839"]
CANON = {"a": "A", "m": "C", "21839": "C"}
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
IUPAC = "ATGCRYSWKMBDHVN"
SHAPES = ((3, 3), (3, 4), (4, 3), (4, 4))
MEMBERS = {"A": "A", "T": "T", "G": "G", "C": "C", "R": "AG", "Y": "CT", "S": "GC", "W": "AT", "K": "GT", "M": "AC",
           "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "*": "ACGT"}


def _iupac(regex):
    """The sweep's spelling of a planted regex motif: classes -> IUPAC letters, '.' -> N."""
    sets = {"AG": "R", "CT": "Y", "AT": "W", "CG": "S", "GT": "K", "AC": "M"}
    out = []
    for tok in re.findall(r"\[[^\]]*\]|.", regex):
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

    return {mt: BinSweep(world[0], mt) for mt in MOD_TYPES}


@pytest.fixture(scope="module")
def frames(sweeps):
    """(mod type, bipartite letters, prune) -> candidate frame at MIN_MEAN / MIN_MOD, made once."""
    cache = {}

    def get(mt, letters="ACGT", prune=True):
        key = (mt, letters, prune)
        if key not in cache:
            cache[key] = sweeps[mt].candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite_letters=letters,
                                               prune=prune)
        return cache[key]

    return get


def _rows(df, b=None, sel=None):
    """(motif, mod_position, n_mod, n_nomod) of a frame's rows, optionally of one bin and a boolean selection."""
    keep = np.ones(len(df), dtype=bool) if b is None else (df["bin"] == b).to_numpy()
    if sel is not None:
        keep = keep & sel
    d = df[keep]
    return list(zip(d["motif"], d["mod_position"].tolist(), d["n_mod"].tolist(), d["n_nomod"].tolist()))


def _is_subsequence(short, long):
    it = iter(long)
    return all(any(x == y for y in it) for x in short)


def _contiguous_rows(mask, n_mod, n_nomod, k, mp, canon):
    """Rows of a (k, mp) table mask in index order, canonical form (no flanking N)."""
    from nanomotif_b200.sweep import decode_motifs

    idx = np.flatnonzero(mask)
    motifs = decode_motifs(k, mp, idx, canon)
    return [(s, mp, int(n_mod[i]), int(n_nomod[i])) for s, i in zip(motifs.tolist(), idx.tolist())
            if s[0] != "N" and s[-1] != "N"]


def _frame_group(df, b, k, mp):
    sel = (df["motif"].str.len() == k).to_numpy() & (df["mod_position"] == mp).to_numpy()
    return _rows(df, b, sel)


@pytest.mark.parametrize("mt", ["a", "m"])
def test_kmers_equal_oracle(world, frames, mt):
    """k = 4..6, every modified position, three bins: the pruned rows are P.sweep_prune of O.sweep_table."""
    scorer, bins, pile = world
    df = frames(mt)
    canon = CANON[mt]
    checked = pruned = 0
    for b in ("bin_0", "bin_6", "bin_4"):
        sel = np.isin(pile["contig"], list(bins[b])) & (pile["mod_type"] == mt)
        for k in (4, 5, 6):
            for mp in range(k):
                n_mod, n_nomod = O.sweep_table(bins[b], pile["contig"][sel], pile["position"][sel],
                                               pile["strand"][sel], pile["fraction_mod"][sel], k, mp, canon)
                keep = P.sweep_prune(n_mod, n_nomod, P.SWEEP_LATTICE, MIN_MEAN, MIN_MOD)
                passes = (n_mod >= MIN_MOD) & ((5.0 + n_mod) / (10.0 + n_mod + n_nomod) >= MIN_MEAN)
                want = _contiguous_rows(keep, n_mod, n_nomod, k, mp, canon)
                assert _frame_group(df, b, k, mp) == want, (b, k, mp)
                checked += len(want)
                pruned += len(_contiguous_rows(passes, n_mod, n_nomod, k, mp, canon)) - len(want)
    assert checked >= 2 and pruned > 10  # 'm': CCWGG@1 in bin_0 and GGCC@2 in bin_4 are the only k <= 6 rows


def _torch_prune(n_mod, n_nomod, n_letters, lattice, min_mean, min_mod):
    """The rule restated in torch over a whole device table (flat, n_letters^n entries, first axis most significant):
    True where the entry passes and is not pruned.  Covers from the oracle's lattice."""
    import math

    widen, narrow = P.lattice_covers(lattice)
    n_axes = int(round(math.log(n_mod.numel()) / math.log(n_letters)))
    assert n_letters ** n_axes == n_mod.numel()
    m = (n_mod.long() & 0xFFFFFFFF).view((n_letters,) * n_axes)
    u = (n_nomod.long() & 0xFFFFFFFF).view((n_letters,) * n_axes)

    def mean(a, b):
        return (5.0 + a.double()) / (10.0 + a.double() + b.double())

    passes = (m >= min_mod) & (mean(m, u) >= min_mean)
    pruned = passes.new_zeros(passes.shape)
    for ax in range(n_axes):
        mv, uv, pv, out = (x.movedim(ax, 0) for x in (m, u, passes, pruned))
        for i in range(n_letters):
            if not (widen[i] or narrow[i]):
                continue
            hit = pv.new_zeros(pv.shape[1:])
            for j in widen[i]:
                hit |= pv[j] & (mean(mv[j] - mv[i], uv[j] - uv[i]) >= min_mean)
            for j in narrow[i]:
                hit |= pv[j] & (mean(mv[i] - mv[j], uv[i] - uv[j]) < min_mean)
            out[i] |= hit
    return (passes & ~pruned).reshape(-1)


def test_long_kmers_equal_torch_restatement(sweeps, frames):
    """k = 7 and 8, every modified position: the pruned rows are the rule restated in torch over
    BinSweep.index(b).table(k, mp, canonical), which tests/test_gpu_bin_sweep.py pins to the oracle."""
    sw, df = sweeps["a"], frames("a")
    checked = 0
    for b in ("bin_4", "bin_0"):
        index = sw.index(b)
        for k in (7, 8):
            for mp in range(k):
                n_mod, n_nomod = index.table(k, mp, "A")
                keep = _torch_prune(n_mod, n_nomod, 15, P.SWEEP_LATTICE, MIN_MEAN, MIN_MOD).cpu().numpy()
                a = n_mod.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
                u = n_nomod.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
                want = _contiguous_rows(keep, a, u, k, mp, "A")
                assert _frame_group(df, b, k, mp) == want, (b, k, mp)
                checked += len(want)
                del n_mod, n_nomod
    assert checked > 0
    # GRNGAAGY@5, planted in bin_4, is an 8-mer row
    assert ("GRNGAAGY", 5) in {(s, p) for s, p, _, _ in _rows(df, "bin_4")}


def _bip_tables(bip_slot, a, g, b, o, canon, letters):
    """n_mod / n_nomod of one (shape, gap, offset) of a finished ACGT bipartite histogram, the a + b - 1 free half
    letters as axes (first most significant), each expanded in numpy from the 4 states to `letters` (MEMBERS)."""
    from nanomotif_b200.sweep import SweepIndex

    first, n = SweepIndex.bipartite_block(a, g, b)
    free = a + b - 1
    w = np.arange(4 ** free)
    code = np.zeros(w.size, dtype=np.int64)
    rest = w.copy()
    for p in reversed(range(a + b)):
        if p == o:
            dig = np.full(w.size, "ATGC".index(canon))
        else:
            dig, rest = rest % 4, rest // 4
        xbit, ybit = (p, a + p) if p < a else (2 * a + p - a, 2 * a + b + p - a)
        code |= (dig >> 1) << xbit | (dig & 1) << ybit
    expand = np.array([[int(s in MEMBERS[ch]) for s in "ATGC"] for ch in letters])
    out = []
    for cls in (0, 1):
        base = first + (o * 2 + cls) * n
        t = bip_slot[base:base + n][code]
        t = t.reshape((4,) * free)
        for ax in range(free):
            t = np.moveaxis(np.tensordot(expand, t, axes=([1], [ax])), 0, ax)
        out.append(t.reshape(-1))
    return out


def _bip_rows(mask, n_mod, n_nomod, a, g, b, o, canon, letters):
    """Rows of an expanded bipartite table mask without the pseudo-letter * (the last letter)."""
    n_l, free = len(letters), a + b - 1
    idx = np.flatnonzero(mask)
    rows = []
    for i in idx.tolist():
        digs = [(i // n_l ** (free - 1 - p)) % n_l for p in range(free)]
        if max(digs) == n_l - 1:
            continue
        halves = [letters[d] for d in digs]
        halves.insert(o, canon)
        motif = "".join(halves[:a]) + "N" * g + "".join(halves[a:])
        rows.append((motif, o if o < a else o + g, int(n_mod[i]), int(n_nomod[i])))
    return rows


def test_bipartite_acgt_equals_oracle(sweeps, frames):
    """Every bin, gap, shape and offset: the pruned ACGT bipartite rows are P.sweep_prune over the finished
    histogram expanded to A T G C *."""
    sw, df = sweeps["a"], frames("a")
    bip = sw.bip.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    is_bip = (df["motif"].str.len() > 8).to_numpy()
    total = pruned = 0
    for s, b in enumerate(sw.bins):
        want = []
        for g in range(4, 9):
            for a, bb in SHAPES:
                for o in range(a + bb):
                    n_mod, n_nomod = _bip_tables(bip[s], a, g, bb, o, "A", "ATGC*")
                    keep = P.sweep_prune(n_mod, n_nomod, P.BIP_ACGT_LATTICE, MIN_MEAN, MIN_MOD)
                    passes = (n_mod >= MIN_MOD) & ((5.0 + n_mod) / (10.0 + n_mod + n_nomod) >= MIN_MEAN)
                    want += _bip_rows(keep, n_mod, n_nomod, a, g, bb, o, "A", "ATGC*")
                    pruned += len(_bip_rows(passes, n_mod, n_nomod, a, g, bb, o, "A", "ATGC*"))
        got = _rows(df, b, is_bip)
        assert sorted(got) == sorted(want), b
        total += len(want)
        pruned -= len(want)
    assert total > 0 and pruned > 0


def test_bipartite_iupac_equals_oracle(sweeps, frames):
    """Halves over the 14 letters other than N: P.sweep_prune over the histogram expanded to those letters and * for
    every (3, g, 3) group and the (4, 6, 3) / (3, 6, 4) groups of the bins with planted bipartite motifs; the (4, 6, 4)
    groups against the torch restatement over the device's bipartite_iupac_table with * appended per axis."""
    import torch

    sw, df = sweeps["a"], frames("a", "IUPAC")
    letters = IUPAC[:-1] + "*"
    bip = sw.bip.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    checked = 0
    for b in ("bin_1", "bin_5"):
        s = sw.bins.index(b)
        groups = [(3, g, 3) for g in range(4, 9)] + ([(4, 6, 3), (3, 6, 4)] if b == "bin_1" else [])
        for a, g, bb in groups:
            for o in range(a + bb):
                mp = o if o < a else o + g
                n_mod, n_nomod = _bip_tables(bip[s], a, g, bb, o, "A", letters)
                keep = P.sweep_prune(n_mod, n_nomod, P.BIP_IUPAC_LATTICE, MIN_MEAN, MIN_MOD)
                want = _bip_rows(keep, n_mod, n_nomod, a, g, bb, o, "A", letters)
                shape = re.compile(f"[^N]{{{a}}}N{{{g}}}[^N]{{{bb}}}")
                sel = (df["motif"].str.fullmatch(shape) & (df["mod_position"] == mp)).to_numpy()
                assert _rows(df, b, sel) == want, (b, a, g, bb, o)
                checked += len(want)
    # (4, 6, 4): the 14^7 device table, * appended on every axis in torch, then the torch restatement
    index = sw.index("bin_1")
    for o in range(8):
        mp = o if o < 4 else o + 6
        tabs = []
        for t in index.bipartite_iupac_table(4, 6, 4, mp, "A"):
            t = (t.long() & 0xFFFFFFFF).view((14,) * 7)
            for ax in range(7):
                t = t.movedim(ax, 0)
                t = torch.cat([t, t[:4].sum(0, keepdim=True)]).movedim(0, ax)
            tabs.append(t.reshape(-1))
        keep = _torch_prune(tabs[0], tabs[1], 15, P.BIP_IUPAC_LATTICE, MIN_MEAN, MIN_MOD)
        star = torch.zeros((15,) * 7, dtype=torch.bool, device=keep.device)
        for ax in range(7):
            star.movedim(ax, 0)[14] = True
        keep = keep & ~star.reshape(-1)
        idx = torch.nonzero(keep).flatten()
        # index over 15 letters -> index over the 14 of the frame
        digits = [(idx // 15 ** (6 - p)) % 15 for p in range(7)]
        idx14 = sum(d * 14 ** (6 - p) for p, d in enumerate(digits)).cpu().numpy()
        from nanomotif_b200.sweep import decode_bipartite_iupac

        motifs = decode_bipartite_iupac(4, 6, 4, mp, idx14, "A")
        m, u = (t[idx].cpu().numpy() for t in tabs)
        want = sorted(zip(motifs.tolist(), [mp] * len(motifs), m.tolist(), u.tolist()))
        sel = (df["motif"].str.fullmatch("[^N]{4}N{6}[^N]{4}") & (df["mod_position"] == mp)).to_numpy()
        assert sorted(_rows(df, "bin_1", sel)) == want, o
        checked += len(want)
    assert checked > 0


def test_pruned_is_subsequence_for_any_chunking(sweeps, frames):
    import pandas as pd

    sw = sweeps["a"]
    full, ref = frames("a", prune=False), frames("a")
    assert list(ref.columns) == list(full.columns)
    assert _is_subsequence(_rows(ref), _rows(full))
    assert len(ref) < len(full)
    np.testing.assert_array_equal(ref["mean"].to_numpy(),
                                  (5.0 + ref["n_mod"].to_numpy()) / (10.0 + ref["n_mod"].to_numpy() + ref["n_nomod"].to_numpy()))
    for kw in ({"scratch_bytes": 1}, {"scratch_bytes": 1 << 50}, {"capacity": 1}, {"scratch_bytes": 1, "capacity": 3}):
        pd.testing.assert_frame_equal(sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, prune=True, **kw), ref)
    # the full frame itself is unchanged by the new argument
    pd.testing.assert_frame_equal(sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD), full)
    iupac_full, iupac = frames("a", "IUPAC", False), frames("a", "IUPAC")
    assert _is_subsequence(_rows(iupac), _rows(iupac_full)) and len(iupac) < len(iupac_full)
    pd.testing.assert_frame_equal(sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, bipartite_letters="IUPAC",
                                                prune=True, scratch_bytes=1, capacity=1), iupac)
    part = sw.candidates(min_mean=MIN_MEAN, min_mod=MIN_MOD, ks=[5, 7], bipartite=False, prune=True)
    pd.testing.assert_frame_equal(part, ref[ref["motif"].str.len().isin([5, 7])].reset_index(drop=True))


def _witness(sw, b, motif, mp):
    """Why a motif is pruned: every widening / narrowing neighbour that prunes it, with P or C and Q's counts."""
    widen = {"A": "RWM", "T": "YWK", "G": "RSK", "C": "YSM", "R": "DV", "Y": "BH", "S": "BV", "W": "DH", "K": "BD",
             "M": "HV", "B": "N", "D": "N", "H": "N", "V": "N", "N": ""}
    narrow = {x: "".join(y for y, up in widen.items() if x in up) for x in widen}
    mean = lambda q: (5.0 + q[0]) / (10.0 + q[0] + q[1])
    passes = lambda c: c[0] >= MIN_MOD and mean(c) >= MIN_MEAN
    m = sw.counts(b, motif, mp)
    out = []
    bipartite = len(motif) > 8
    for i, ch in enumerate(motif):
        if i == mp or (bipartite and ch == "N"):
            continue
        ups = "*" if bipartite else widen[ch]
        for up in ups:
            if up == "*":
                parts = [sw.counts(b, motif[:i] + x + motif[i + 1:], mp) for x in "ACGT"]
                p = tuple(sum(c[j] for c in parts) for j in (0, 1))
            else:
                p = sw.counts(b, motif[:i] + up + motif[i + 1:], mp)
            q = (p[0] - m[0], p[1] - m[1])
            if passes(p) and mean(q) >= MIN_MEAN:
                out.append(f"(a) P={motif[:i] + up + motif[i + 1:]} {p} Q={q}")
        for down in ("" if bipartite else narrow[ch]):
            c = sw.counts(b, motif[:i] + down + motif[i + 1:], mp)
            q = (m[0] - c[0], m[1] - c[1])
            if passes(c) and mean(q) < MIN_MEAN:
                out.append(f"(b) C={motif[:i] + down + motif[i + 1:]} {c} Q={q}")
    return f"{b} {motif}@{mp} {m}: " + "; ".join(out)


@pytest.mark.parametrize("mt", MOD_TYPES)
def test_planted_motifs_survive_and_rows_shrink(sweeps, frames, mt):
    sw = sweeps[mt]
    full = frames(mt, prune=False)
    for letters in ("ACGT", "IUPAC"):
        df = frames(mt, letters)
        keys = set(zip(df["bin"], df["motif"], df["mod_position"]))
        checked = 0
        for b, (_, planted) in BINS.items():
            for regex, mp, t in planted:
                if t != mt:
                    continue
                motif = _iupac(regex)
                assert (b, motif, mp) in keys, _witness(sw, b, motif, mp)
                checked += 1
        assert checked >= 1
    counts, full_counts = frames(mt)["bin"].value_counts(), full["bin"].value_counts()
    for b, (_, planted) in BINS.items():
        if any(t == mt for _, _, t in planted):
            assert counts.get(b, 0) < full_counts[b], b
    assert NO_ROWS not in set(frames(mt)["bin"])
