"""Host side of the per-bin sweep (sweep.BinSweep): the vectorised decoders of candidate records against the scalar
SweepIndex helpers they replace, and the argument checks of the histogram entry points (no GPU needed)."""
import ctypes as C

import numpy as np

from nanomotif_b200 import _lib
from nanomotif_b200.sweep import IUPAC_ORDER, SweepIndex, decode_bipartite, decode_motifs, table_scratch_bytes


def test_decode_motifs_equals_index_motif():
    for mp in range(4):
        idx = np.arange(15 ** 3)
        got = decode_motifs(4, mp, idx, "A")
        assert got.tolist() == [SweepIndex.index_motif(i, 4, mp, "A") for i in range(15 ** 3)]
    rng = np.random.default_rng(7)
    for mp in range(8):
        idx = rng.integers(0, 15 ** 7, 2000)
        got = decode_motifs(8, mp, idx, "C")
        assert got.tolist() == [SweepIndex.index_motif(int(i), 8, mp, "C") for i in idx]
        assert [SweepIndex.motif_index(s, mp) for s in got] == idx.tolist()
    assert set("".join(decode_motifs(5, 2, np.arange(15 ** 4), "A"))) == set(IUPAC_ORDER)


def test_decode_bipartite_inverts_bipartite_index():
    rng = np.random.default_rng(8)
    counters, want = [], []
    for _ in range(3000):
        a, g, b = int(rng.integers(3, 5)), int(rng.integers(4, 9)), int(rng.integers(3, 5))
        left, right = "".join(rng.choice(list("ACGT"), a)), "".join(rng.choice(list("ACGT"), b))
        o = int(rng.integers(0, a + b))
        first, n = SweepIndex.bipartite_block(a, g, b)
        counters.append(first + o * 2 * n + SweepIndex.bipartite_index(left, right))
        want.append((left + "N" * g + right, o if o < a else o + g))
    motifs, mod_pos = decode_bipartite(np.array(counters))
    assert list(zip(motifs.tolist(), mod_pos.tolist())) == want
    assert decode_bipartite(np.zeros(0, np.int64))[0].size == 0


def test_scratch_per_bin():
    # k = 8: the 25 x 15^5 input and the 5 x 15^6 output of the last written expansion step, two classes of uint32
    assert table_scratch_bytes(8) == 2 * 4 * (25 * 15 ** 5 + 5 * 15 ** 6) == 607_500_000
    assert all(table_scratch_bytes(k) < table_scratch_bytes(k + 1) for k in range(4, 8))


def test_histogram_entry_points_refuse_bad_slot_maps():
    lib = _lib.lib
    asm = _lib.NmbAssembly()  # no tiles: an accepted call launches nothing
    p = np.zeros(16, dtype=np.uint32).ctypes.data
    slot_map = np.zeros(4, dtype=np.int32).ctypes.data
    for fn in (lib.nmb_sweep_hist, lib.nmb_sweep_bipartite):
        # a null map counts the contig range into one histogram; a map routes contigs into n_slots > 0 histograms
        assert fn(C.byref(asm), p, 0, 0, 0, 0, None, 1, p, None) == 0
        assert fn(C.byref(asm), p, 0, 0, 0, 0, slot_map, 3, p, None) == 0
        for contig_slot, n_slots in ((None, 0), (None, 2), (slot_map, 0), (slot_map, -1)):
            assert fn(C.byref(asm), p, 0, 0, 0, 0, contig_slot, n_slots, p, None) == -1
            assert b"bad slot map" in lib.nmb_last_error() and fn.__name__.encode() in lib.nmb_last_error()
        assert fn(C.byref(asm), p, 0, 1, 0, 0, None, 1, p, None) == -1  # tiles outside the assembly
    assert lib.nmb_sweep_finalize(p, 0, None) == -1 and lib.nmb_sweep_bipartite_finalize(p, 0, None) == -1
    assert lib.nmb_sweep_slice(p, 0, 0, p, 1, 1, 0, None) == -1
