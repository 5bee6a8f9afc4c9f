"""Host logic of the sharded motif discovery (sharding.discover), no device: the whole-bin plan derived from lengths
alone, the gather of every rank's candidate rows into the order of one GPU over gloo on CPU tensors (world sizes 1-4,
ranks without bins included), and the agreement of every rank on an error raised on one of them."""
import os
import socket
import traceback

import numpy as np
import pandas as pd
import pytest

from nanomotif_b200 import search, sharding

MOD_TYPES = ("a", "m", "21839")
LAYOUTS = {
    # {bin: contig lengths}
    "mixed": {"b0": (90000, 7, 3000), "b1": (40000,), "b2": (5, 25000, 12000, 3), "b3": (60000, 800), "b4": (4,)},
    "giant": {"big": (500000, 400000), "s0": (9000,), "s1": (300, 7), "s2": (20000,)},  # one bin >> 1.25 / world
    "solo": {"only": (30000, 2000)},  # one bin: every rank but one is empty
    "pair": {"x": (5000,), "y": (5000,)},
}


def _bins(layout, as_sequences=False):
    return {b: {f"{b}_c{i}": ("A" * n if as_sequences else n) for i, n in enumerate(lens)}
            for b, lens in LAYOUTS[layout].items()}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_every_bin_lands_whole_on_one_rank(layout, world):
    bins = _bins(layout)
    plan = sharding.discovery_plan(bins, world)
    assert list(plan) == list(bins)
    assert all(0 <= r < world for r in plan.values())
    assert plan == sharding.discovery_plan(_bins(layout, as_sequences=True), world)  # lengths are all it needs
    # the greedy packing of plan_shards over one unit per bin: the longest bin goes to rank 0, and with at least as
    # many ranks as bins every bin has a rank of its own
    totals = {b: sum(lens) for b, lens in LAYOUTS[layout].items()}
    assert plan[max(totals, key=totals.get)] == 0
    if world >= len(bins):
        assert len(set(plan.values())) == len(bins)
    if layout == "giant" and world > 1:  # the contig plan of the scorer spreads this bin; the discovery plan does not
        _, _, split, _ = sharding.ShardedMultiBinScorer.plan(bins, world)
        assert "big" in split
        assert plan["big"] == 0 and all(plan[b] != 0 for b in ("s0", "s1", "s2"))


def test_plan_ignores_sequence_content_and_contig_split():
    bins = {"p": {"c0": 1000, "c1": 1000}, "q": {"d0": 1500}, "r": {"e0": 400}}
    same = {"p": {"c0": 2000}, "q": {"d0": "ACGT" * 375}, "r": {"e0": 100, "e1": 300}}
    for world in (1, 2, 3):
        assert sharding.discovery_plan(bins, world) == sharding.discovery_plan(same, world)


def _rows(layout, seed=11):
    """Candidate rows of every (bin, mod type) pair in the order of one GPU; some pairs have none."""
    rng = np.random.default_rng(seed)
    rows = []
    for b in LAYOUTS[layout]:
        for mt in MOD_TYPES:
            for k in range(int(rng.integers(0, 4))):
                rows.append(dict(bin=b, mod_type=mt, motif="".join(rng.choice(list("ACGT."), size=int(rng.integers(2, 9)))),
                                 mod_position=int(rng.integers(0, 8)), n_mod=int(rng.integers(0, 1 << 40)),
                                 n_nomod=int(rng.integers(0, 1000)), score=float(rng.normal()) if k else -1.0))
    return rows


def test_merge_restores_bin_then_mod_type_order():
    rows = _rows("mixed")
    for seed in range(5):
        rng = np.random.default_rng(seed)
        # each rank's rows are in its own order; ranks come in any order, pairs stay contiguous within a rank
        by_rank = {}
        for r in rows:
            by_rank.setdefault(hash(r["bin"]) % 3, []).append(r)
        parts = [by_rank[k] for k in rng.permutation(sorted(by_rank))]
        got = sharding.merge_discovery_rows([r for p in parts for r in p], list(LAYOUTS["mixed"]), MOD_TYPES)
        assert got == rows


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    fails = []
    try:
        for layout in sorted(LAYOUTS):
            bins = _bins(layout)
            plan = sharding.discovery_plan(bins, world)
            rows = _rows(layout)
            mine = [r for r in rows if plan[r["bin"]] == rank]
            got = sharding.gather_discovery(mine, None, bins, MOD_TYPES, rank, world, "cpu")
            try:
                pd.testing.assert_frame_equal(got, search.discovery_frame(rows), check_exact=True)
            except AssertionError as exc:
                fails.append(f"{layout}: {exc}")
            if list(got.columns) != list(search.DISCOVERY_COLUMNS):
                fails.append(f"{layout}: columns {list(got.columns)}")
        empty = sharding.gather_discovery([], None, _bins("pair"), MOD_TYPES, rank, world, "cpu")
        if len(empty) or list(empty.dtypes) != list(search.discovery_frame(_rows("pair")).dtypes):
            fails.append("empty frame")
        # an error on one rank (or several: the lowest rank's wins) raises on every rank
        cases = [({s: ValueError(f"short contig on rank {s}")}, f"short contig on rank {s}") for s in range(world)]
        cases.append(({r: KeyError(f"rank {r}") for r in range(world)}, None))
        for errors, message in cases:
            try:
                sharding.gather_discovery([], errors.get(rank), _bins("pair"), MOD_TYPES, rank, world, "cpu")
                fails.append(f"{errors}: no exception")
            except ValueError as exc:
                if str(exc) != message:
                    fails.append(f"{errors}: {exc}")
            except KeyError as exc:
                if message is not None or exc.args != ("rank 0",):
                    fails.append(f"{errors}: {exc!r}")

        class Unpicklable(Exception):
            def __reduce__(self):
                raise TypeError("no pickling")

        try:
            sharding.agree_on_error(Unpicklable("x") if rank == world - 1 else None, "cpu", world, rank)
            fails.append("unpicklable: no exception")
        except RuntimeError as exc:
            if not str(exc).startswith(f"rank {world - 1}: "):
                fails.append(f"unpicklable: {exc}")
        except Unpicklable:
            if world > 1 and rank != world - 1:
                fails.append("unpicklable: raised the original on another rank")
        sharding.agree_on_error(None, "cpu", world, rank)  # nobody failed: returns on every rank
        q.put((rank, fails))
    except Exception:  # noqa: BLE001 -- reported to the test process
        q.put((rank, [traceback.format_exc()]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_gather_order_and_error_agreement_over_gloo(world):
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


def test_candidate_rows_from_a_search_result():
    from nanomotif_b200.model import BetaBernoulliModel
    from nanomotif_b200.motif import Motif

    graph = search.MotifGraph()
    found, missed = Motif("...GATC..", 4), Motif("..C.A....", 4)
    for m, counts, score in ((found, (90, 3), 2.5), (missed, (40, 7), 1.75)):
        model = BetaBernoulliModel()
        model.update(*counts)
        graph.add_node(m, model=model, score=np.float64(score))
    rows = search.candidate_rows("b7", "a", (graph, [found, missed]))
    assert rows == [dict(bin="b7", mod_type="a", motif="GATC", mod_position=1, n_mod=90, n_nomod=3, score=2.5),
                    dict(bin="b7", mod_type="a", motif="C.A", mod_position=2, n_mod=40, n_nomod=7, score=1.75)]
    assert search.candidate_rows("b7", "a", None) == []
    df = search.discovery_frame(rows)
    assert df["n_mod"].dtype == np.int64 and df["score"].dtype == np.float64 and df["mod_position"].dtype == np.int64
