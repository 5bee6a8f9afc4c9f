"""K2's sibling runs (one parent chain pair + a four-base split per run of search-expansion children) against the
general path and the oracle, bit for bit, in dynamic and static item scheduling and for several motif block sizes:
runs in contig-edge warps (contigs shorter than a warp and shorter than the motif), the split position first and
last, the modified base alone as the parent, bracket sets and '.' at the split position, two-word halos, non-ACGT
warps, adjacent runs with different split positions, duplicates and search-shaped work lists."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import restate as O  # the checker, never the thing under test


@pytest.fixture(scope="module")
def nmb():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200 as nmb

    return nmb


HAND = [
    [("GA", 1), ("CA", 1), ("TA", 1), ("AA", 1)],                          # parent = the modified base alone, j first
    [("AG", 0), ("AC", 0), ("AT", 0)],                                     # j last
    [("GA.C", 1), ("GA[CT]C", 1), ("GA[AG]C", 1), ("GA[ACG]C", 1)],       # '.' and bracket sets at j
    [("GATC", 1), ("GATG", 1), ("GAAG", 1), ("GACG", 1)],                 # adjacent runs, different j
    [("GATC", 1), ("GATC", 1), ("GATG", 1), ("GATC", 1), ("GATC", 1)],    # duplicates inside a run
    [("GATC", 1), ("GATC", 1)],                                            # duplicates alone
    [("GATC", 1), ("GATG", 1), ("CATC", 1), ("GAT.C", 1)],                # mixed: runs break and restart
    [("A" + "." * 30 + "C", 0), ("A" + "." * 30 + "G", 0)],                # split 31 right of the modified base
    [("C" + "." * 30 + "A", 31), ("T" + "." * 30 + "A", 31)],              # ... 31 left
    [("A" + "." * 40 + "C", 0), ("A" + "." * 40 + "G", 0), ("A" + "." * 40 + "T", 0)],   # two-word halo, 41 right
    [("C" + "." * 40 + "GA", 42), ("T" + "." * 40 + "GA", 42)],            # ... 42 left
    [("G" + "." * 20 + "A" + "." * 30 + "CT", 21), ("G" + "." * 20 + "A" + "." * 30 + "GT", 21)],
    [("CAT", 1), ("CAG", 1), ("CA[CG]", 1), ("CA.", 1)],                   # last member: shorter once stripped
]


def _pileup(rng, lengths, synth, n_rate):
    contigs, cols = {}, {k: [] for k in ("contig", "position", "strand", "fraction_mod")}
    for i, L in enumerate(lengths):
        seq = synth.random_sequence(rng, int(L), 0.45, n_rate if L > 1000 else 0.0)
        contigs[f"c{i}"] = seq.tobytes().decode()
        p = synth.synth_pileup(seq, rng, depth=15, mod_types=("a",))
        cols["contig"].append(np.full(len(p["position"]), f"c{i}", dtype=object))
        cols["position"].append(p["position"])
        cols["strand"].append(np.where(np.asarray(p["strand"]) == 0, "+", "-"))
        cols["fraction_mod"].append(p["fraction_mod"])
    return contigs, {k: np.concatenate(v) for k, v in cols.items()}


def _check(nmb, contigs, pile, flat, mpis, per_contig=False):
    from nanomotif_b200 import device as D

    scorer = nmb.BinScorer(pile, contigs, 0.3, 0.7)
    want = np.array([O.motif_model_bin(pile["contig"], pile["position"], pile["strand"], pile["fraction_mod"], contigs,
                                       m.string, m.mod_position, fast=True) for m in flat])
    old = D.FAMILIES, D.BALANCED
    try:
        D.FAMILIES, D.BALANCED = False, True
        general = scorer.counts_by_strand(flat, motifs_per_item=4).cpu().numpy()
        general_pc = scorer.counts_by_strand(flat, per_contig=True).cpu().numpy() if per_contig else None
        np.testing.assert_array_equal(np.stack([general[:, 0] + general[:, 2], general[:, 1] + general[:, 3]], 1), want)
        for balanced in (True, False):
            D.FAMILIES, D.BALANCED = True, balanced
            for mpi in mpis:
                got = scorer.counts_by_strand(flat, motifs_per_item=mpi).cpu().numpy()
                np.testing.assert_array_equal(got, general, err_msg=f"balanced={balanced} mpi={mpi}")
            if per_contig:  # every contig its own output row: edge warps count per contig
                got = scorer.counts_by_strand(flat, per_contig=True).cpu().numpy()
                np.testing.assert_array_equal(got, general_pc, err_msg=f"per contig, balanced={balanced}")
    finally:
        D.FAMILIES, D.BALANCED = old
    return want


def test_sibling_links_written_by_the_compiler(nmb):
    import torch

    from nanomotif_b200.device import MotifPrograms
    from nanomotif_b200.motif import pack_motifs, sibling_links

    packed = pack_motifs([nmb.Motif(m, p) for kids in HAND for m, p in kids])
    progs = MotifPrograms(packed, torch.device("cuda", 0))
    dev = progs.siblings[:4 * len(packed)].view(torch.int32).cpu().numpy().view(np.uint32)
    np.testing.assert_array_equal(dev, sibling_links(packed))


def test_hand_made_runs_at_contig_edges_and_non_acgt(nmb):
    from nanomotif_b200 import synth

    rng = np.random.default_rng(41)
    # many contigs shorter than a warp's 16 384 positions, some shorter than the motifs, N letters in the long ones
    lengths = np.concatenate([[150000, 66000, 131072 - 64], rng.integers(1, 40, 12), rng.integers(40, 3000, 30)])
    rng.shuffle(lengths)
    contigs, pile = _pileup(rng, lengths, synth, 3e-5)
    flat = [nmb.Motif(m, p) for kids in HAND for m, p in kids]
    short = [m for m in flat if len(m.string) <= 32]  # one-word halos; with the longer ones the launch takes two
    for motifs in (short, flat):
        want = _check(nmb, contigs, pile, motifs, (None, 2, 3, 4, 32), per_contig=True)
        assert int(want.sum()) > 10000


def test_frontier_worklists(nmb):
    """Search-shaped work lists of several (bin, mod type) pairs over bins laid out like cfg3's."""
    from nanomotif_b200 import synth

    rng = np.random.default_rng(7)
    contigs, pile = _pileup(rng, np.maximum(2500, rng.lognormal(0.0, 1.0, 40) / 40 * 1_500_000).astype(int), synth, 1e-5)
    flat = [nmb.Motif(m, p) for seed in range(4) for kids in synth.frontier_worklist(seed, "A", rounds=64)
            for m, p in kids]
    want = _check(nmb, contigs, pile, flat, (None, 3, 4, 32))
    assert int(want.sum()) > 100000
