"""Host side of the per-bin sweep (sweep.BinSweep): the vectorised decoders of candidate records against the scalar
SweepIndex helpers they replace (no GPU needed)."""
import numpy as np

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
