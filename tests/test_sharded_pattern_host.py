"""Host logic of the sharded methylation-pattern table (sharding.ShardedPatternTable), no device: each rank's contig
columns placed into global contig order, the exact gather of the table over gloo on CPU tensors (world sizes 1-4,
ranks without contigs included), and the agreement of every rank on the mismatch flag and on the motif list."""
import os
import socket
import traceback

import numpy as np
import pytest
import torch

from nanomotif_b200 import sharding

LAYOUTS = {
    "mixed": (90000, 7, 3000, 40000, 5, 25000, 12000, 3, 60000, 800, 4),
    "mono": (500000, 9000, 300, 7),
    "solo": (30000,),  # one contig: every rank but rank 0 is empty
    "pair": (5000, 5000),
}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _table(n_motifs, n_contigs, seed=3):
    """A whole table as pattern_table returns it: n_motif_obs 0 in some cells, value NaN exactly there."""
    rng = np.random.default_rng(seed)
    stats = rng.integers(0, 1 << 40, size=(n_motifs, n_contigs, 3), dtype=np.int64)
    stats[:, :, 0] = np.where(rng.random((n_motifs, n_contigs)) < 0.3, 0, stats[:, :, 0] % 1000)
    value = rng.random((n_motifs, n_contigs))
    value[rng.random((n_motifs, n_contigs)) < 0.05] = 0.0
    value[stats[:, :, 0] == 0] = np.nan
    return stats, value


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_rank_columns_land_at_their_global_contig(layout, world):
    lengths = LAYOUTS[layout]
    owner = sharding.plan_shards(lengths, world)
    stats, value = _table(5, len(lengths))
    total_s = np.zeros_like(stats)
    total_v = np.zeros_like(value)
    for r in range(world):
        cols = np.flatnonzero(owner == r)
        got_s, got_v = sharding.place_columns(torch.from_numpy(stats[:, cols].copy()), torch.from_numpy(value[:, cols].copy()),
                                              cols, len(lengths))
        want_s, want_v = np.zeros_like(stats), np.zeros_like(value)
        for c in cols:  # brute force, one cell at a time
            for m in range(stats.shape[0]):
                want_s[m, c] = stats[m, c]
                want_v[m, c] = value[m, c] if stats[m, c, 0] > 0 else 0.0
        np.testing.assert_array_equal(got_s.numpy(), want_s)
        np.testing.assert_array_equal(got_v.numpy(), want_v)  # no NaN: the ranks' tensors can be added
        total_s += got_s.numpy()
        total_v += got_v.numpy()
        s_only, v_none = sharding.place_columns(torch.from_numpy(stats[:, cols].copy()), None, cols, len(lengths))
        assert v_none is None and torch.equal(s_only, got_s)
    np.testing.assert_array_equal(total_s, stats)  # every contig has exactly one owner
    np.testing.assert_array_equal(np.where(stats[:, :, 0] > 0, total_v, np.nan), value)


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    fails = []
    try:
        for layout, lengths in sorted(LAYOUTS.items()):
            owner = sharding.plan_shards(lengths, world)
            cols = np.flatnonzero(owner == rank)
            stats, value = _table(7, len(lengths), seed=len(lengths))
            for median in (True, False):
                v = torch.from_numpy(value[:, cols].copy()) if median else None
                got_s, got_v = sharding.gather_columns(torch.from_numpy(stats[:, cols].copy()), v, cols, len(lengths), world)
                if not np.array_equal(got_s.numpy(), stats):
                    fails.append(f"{layout}: stats")
                if median and not np.array_equal(got_v.numpy(), value, equal_nan=True):
                    fails.append(f"{layout}: value")
                if not median and got_v is not None:
                    fails.append(f"{layout}: value without median")
        # the mismatch flag: set on one rank only, seen by every rank
        for setter in range(world):
            hi, lo = sharding.rank_extremes([int(rank == setter), 5], "cpu", world)
            if hi.tolist() != [1, 5] or lo.tolist() != [int(world == 1), 5]:
                fails.append(f"flag of rank {setter}: {hi.tolist()} {lo.tolist()}")
        motifs = ["GATC_a_1", "CCWGG_m_1", "CCGG_21839_0"]
        sharding.check_same_motifs(motifs, "cpu", world)
        for other in (motifs[::-1], motifs[:2], motifs + ["GATC_a_1"], ["GATC_a_1", "CCWGG_m_1", "CCGG_21839_1"]):
            mine = other if rank == world - 1 else motifs
            try:
                sharding.check_same_motifs(mine, "cpu", world)
                raised = False
            except ValueError:
                raised = True
            if raised != (world > 1):
                fails.append(f"motif list {other}: raised={raised}")
        q.put((rank, fails))
    except Exception:  # noqa: BLE001 -- reported to the test process
        q.put((rank, [traceback.format_exc()]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_gather_flag_and_motif_check_over_gloo(world):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = sorted(q.get(timeout=300) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    for rank, fails in results:
        assert not fails, f"rank {rank}:\n" + "\n".join(fails)


def test_motif_list_key_is_stable_and_order_sensitive():
    key = sharding.motif_list_key(["GATC_a_1", "CCWGG_m_1"])
    assert key == sharding.motif_list_key(("GATC_a_1", "CCWGG_m_1"))
    assert key[0] == 2 and 0 <= key[1] < 1 << 62
    assert key != sharding.motif_list_key(["CCWGG_m_1", "GATC_a_1"])
