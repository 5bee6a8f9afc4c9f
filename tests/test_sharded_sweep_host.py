"""Host logic of the sharded per-bin sweep (sharding.ShardedBinSweep), no device: the designated rank of every bin, the
row order of the split-bin all-reduce, and the merge of per-rank hit records into the single-GPU frame order."""
import numpy as np
import pytest

from nanomotif_b200 import _lib, sharding
from nanomotif_b200.sweep import BIP_SIZE, _candidate_groups, _frame

LAYOUTS = {
    "bins": {"bin_big": (90000, 70000, 60000, 40000), "bin_s1": (30000, 8000), "bin_s2": (25000,),
             "bin_s3": (9000, 7000, 3000)},
    "mono": {"mono": (200000, 9000), "bin_s1": (12000, 8000)},
    "many": {f"bin_{i}": tuple(1000 + 700 * ((i * 7 + j) % 11) for j in range(1 + i % 4)) for i in range(23)},
    "empty": {"bin_a": (5000, 3), "no_contigs": (), "bin_b": (40000,)},
}


def _bins(layout):
    return {b: {f"{b}_c{i}": n for i, n in enumerate(lens)} for b, lens in LAYOUTS[layout].items()}


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_designated_rank_and_split_order_follow_from_the_plan(layout, world):
    bins = _bins(layout)
    _, per_rank, split_bins, bin_ranks = sharding.ShardedMultiBinScorer.plan(bins, world)
    rng = np.random.default_rng(world)
    for order in (list(bins), list(rng.permutation(list(bins)))):
        layouts = [sharding.sweep_layout(order, bin_ranks, split_bins, set(per_rank[r])) for r in range(world)]
        designated, split = layouts[0][0], layouts[0][1]
        for r, (des, spl, local, slot) in enumerate(layouts):
            assert des == designated and spl == split  # every rank derives the same
            assert local == [b for b in order if b in per_rank[r]]
            assert [order[s] for s in slot] == local and slot.dtype == np.int32
        assert split == [b for b in order if len(bin_ranks[b]) > 1]
        for b in order:
            holders = [r for r in range(world) if b in per_rank[r]]
            assert designated[b] == (holders[0] if holders else 0)
            if holders:
                assert b in layouts[designated[b]][2]  # the designated rank holds the bin
    if layout == "bins" and world == 2:
        assert split_bins == {"bin_big"}
    if layout == "mono" and world == 2:
        assert split_bins == {"mono"} and bin_ranks["mono"] == [0, 1]
    if layout == "empty":
        assert bin_ranks["no_contigs"] == [] and all("no_contigs" not in p for p in per_rank)


def _records(rng, n, n_slots, groups, bip_groups):
    """n synthetic hit records of distinct (slot, group, index): index within each group's table."""
    n_groups = len(groups) + (1 if bip_groups is None else len(bip_groups))
    seen, out = set(), []
    while len(out) < n:
        slot, g = int(rng.integers(n_slots)), int(rng.integers(n_groups))
        if g < len(groups):
            size = 15 ** (groups[g][0] - 1)
        elif bip_groups is None:
            size = BIP_SIZE
        else:
            a, _, b, _ = bip_groups[g - len(groups)]
            size = 14 ** (a + b - 1)
        idx = int(rng.integers(size))
        if bip_groups is None and g == len(groups):
            idx = _n_mod_counter(idx)
        if (slot, g, idx) in seen:
            continue
        seen.add((slot, g, idx))
        out.append((slot, g, idx, int(rng.integers(1, 1000)), int(rng.integers(0, 1000))))
    return out


def _n_mod_counter(i):
    """An n_mod counter of the bipartite histogram near counter i (the decoder reads n_mod positions)."""
    from nanomotif_b200.sweep import _BIP_SHAPES, SweepIndex

    per_gap = SweepIndex.bipartite_block(3, 5, 3)[0]
    g, rem = i // per_gap + 4, i % per_gap
    for a, b in _BIP_SHAPES:
        first, n = SweepIndex.bipartite_block(a, 4, b)
        if first <= rem < first + (a + b) * 2 * n:
            r = rem - first
            return (g - 4) * per_gap + first + (r // (2 * n)) * 2 * n + r % n
    raise AssertionError(i)


@pytest.mark.parametrize("letters", ["ACGT", "IUPAC"])
@pytest.mark.parametrize("world", [2, 3, 5])
def test_merged_records_give_the_single_gpu_order(letters, world):
    """Records of every rank, local slots mapped to global ones, in any part order -> the frame of the same records
    with global slots in one part; its rows are the brute-force sort by (slot, group, index)."""
    import pandas as pd

    rng = np.random.default_rng(7 + world)
    bins = [f"bin_{i}" for i in rng.permutation(9)]
    _, groups, bip_groups = _candidate_groups(1, [4, 6, 8], True, letters, True)
    recs = _records(rng, 3000, len(bins), groups, bip_groups)
    # each bin on one designated rank; the last rank holds no bin (it still takes part with no records)
    rank_of = {b: int(rng.integers(world - 1)) for b in bins}
    parts = []
    for r in range(world):
        des, _, local, slot = sharding.sweep_layout(bins, {b: [rank_of[b]] for b in bins}, set(),
                                                    {b for b in bins if rank_of[b] == r})
        local_slot = {b: i for i, b in enumerate(local)}
        mine = [x for x in recs if rank_of[bins[x[0]]] == r]
        by_group = {}
        for s, g, idx, m, n in mine:
            by_group.setdefault(g, []).append((local_slot[bins[s]], idx, m, n))
        rank_parts = []
        for g, rows in by_group.items():
            rows = [rows[i] for i in rng.permutation(len(rows))]
            for chunk in np.array_split(np.arange(len(rows)), 1 + int(rng.integers(3))):
                h = np.array([rows[i] for i in chunk], dtype=_lib.SWEEP_HIT_DTYPE)
                rank_parts.append((g, h))
        if r == world - 1:
            assert not local and not rank_parts and not len(slot)
        parts.append(sharding.global_parts(rank_parts, slot))
    merged = [p for r in rng.permutation(world) for p in parts[r]]
    got = _frame(merged, groups, bip_groups, bins, "a", "A")
    one = [(g, np.array([(s, i, m, n) for s, gg, i, m, n in recs if gg == g], dtype=_lib.SWEEP_HIT_DTYPE))
           for g in sorted({x[1] for x in recs})]
    pd.testing.assert_frame_equal(got, _frame(one, groups, bip_groups, bins, "a", "A"))
    want = sorted(recs, key=lambda x: (x[0], x[1], x[2]))
    assert list(got["bin"]) == [bins[s] for s, _, _, _, _ in want]
    assert got["n_mod"].tolist() == [m for _, _, _, m, _ in want]
    assert got["n_nomod"].tolist() == [n for _, _, _, _, n in want]
    assert len(got) == len(recs)


def test_no_records_on_any_rank():
    _, groups, bip_groups = _candidate_groups(5, range(4, 9), True, "ACGT", True)
    df = _frame([p for _ in range(3) for p in sharding.global_parts([], np.zeros(0, np.int32))], groups, bip_groups,
                ["bin_0", "bin_1"], "m", "C")
    assert len(df) == 0
    assert list(df.columns) == ["bin", "mod_type", "motif", "mod_position", "n_mod", "n_nomod", "mean"]


def test_argument_checks_need_no_device():
    with pytest.raises(ValueError):
        _candidate_groups(0, range(4, 9), True, "ACGT", True)
    with pytest.raises(ValueError):
        _candidate_groups(5, [3, 4], True, "ACGT", True)
    with pytest.raises(ValueError):
        _candidate_groups(5, [4], True, "N", True)
    with pytest.raises(ValueError):
        _candidate_groups(5, [4], True, "ACGT", False)
    ks, groups, bip = _candidate_groups(5, [5, 4, 5], False, "IUPAC", False)
    assert ks == [4, 5] and groups == [(4, 0), (4, 1), (4, 2), (4, 3)] + [(5, i) for i in range(5)] and bip is None
