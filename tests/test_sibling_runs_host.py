"""The sibling-run predicate of K2 (host mirror nanomotif_b200.motif.sibling_links / sibling_runs): every round of a
search-shaped work list is exactly one run, and runs break where the motifs stop differing at one common position."""
import numpy as np

from nanomotif_b200 import synth
from nanomotif_b200.motif import Motif, pack_motifs, sibling_links, sibling_runs


def _runs(specs, begin=0, count=None):
    packed = pack_motifs([Motif(m, p) for m, p in specs])
    return sibling_runs(sibling_links(packed), begin, len(specs) - begin if count is None else count)


def test_every_frontier_round_is_one_run():
    for seed in range(12):
        rounds = synth.frontier_worklist(seed, "ACG"[seed % 3], rounds=64, width=4)
        for kids in rounds:
            assert len(_runs(kids)) == 1 and _runs(kids)[0][:2] == (0, len(kids)), kids
        # a block of several rounds (the batched schedules) is cut into exactly those rounds
        flat = [k for kids in rounds for k in kids]
        starts = np.concatenate([[0], np.cumsum([len(k) for k in rounds])[:-1]]).tolist()
        assert [(a, n) for a, n, _ in _runs(flat)] == list(zip(starts, [len(k) for k in rounds]))


def test_mixed_rounds_break_runs():
    assert _runs([("GATC", 1), ("GATG", 1), ("CATC", 1), ("GAT.C", 1)]) == [(0, 2, 3)]
    # adjacent runs with different split positions
    assert _runs([("GATC", 1), ("GATG", 1), ("GAAG", 1), ("GACG", 1)]) == [(0, 2, 3), (2, 2, 2)]
    # identical motifs alone form no run; next to a differing sibling they join it
    assert _runs([("GATC", 1), ("GATC", 1)]) == []
    assert _runs([("GATC", 1), ("GATC", 1), ("GATG", 1), ("GATG", 1)]) == [(0, 4, 3)]
    # different mod_pos or length: no link
    assert _runs([("GATC", 1), ("GATG", 2)]) == []
    assert _runs([("GATC", 1), ("GATCA", 1)]) == []
    # a bracket set or a wildcard at j, a parent that is the modified base alone
    assert _runs([("GA.C", 1), ("GA[CT]C", 1), ("GA[AG]C", 1)]) == [(0, 3, 2)]
    assert _runs([("GA", 1), ("CA", 1), ("TA", 1), ("AA", 1)]) == [(0, 4, 0)]


def test_runs_are_cut_at_block_boundaries():
    specs = [("GATC", 1), ("GATG", 1), ("GATA", 1), ("GATT", 1)]
    assert _runs(specs, 0, 2) == [(0, 2, 3)]
    assert _runs(specs, 1, 3) == [(1, 3, 3)]
    assert _runs(specs, 3, 1) == []
    # a block that starts inside a run of identical motifs still finds the split position further right
    assert _runs([("GATC", 1), ("GATC", 1), ("GATC", 1), ("GATG", 1)], 1, 3) == [(1, 3, 3)]


def test_link_word_layout():
    packed = pack_motifs([Motif("GATC", 1), Motif("GATG", 1), Motif("GATG", 1), Motif("AATG", 2)])
    w = sibling_links(packed)
    assert w[0] == 0
    assert w[1] == 3 | 2 << 6 | 0b0100 << 8 | 0b1000 << 12  # j = 3, differ: own G, previous C
    assert w[2] == 1 << 6
    assert w[3] == 0
