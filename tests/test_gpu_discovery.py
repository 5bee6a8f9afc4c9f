"""search.discover and sharding.discover on CUDA devices.  One GPU: the frame reproduces the recorded reference search
traces (synthetic bin and the cfg1 plasmid bin), equals sequential search.run on a GpuBinBackend per (bin, mod type)
pair, scores every round of all pairs with one launch, does not depend on the bin order or a bin subset, and leaves the
caller's `random` state alone.  World size 2 (NCCL on two GPUs, gloo over CUDA tensors when the box has one): every
rank returns the one-GPU frame, from a table, the partitioned dict or local scorers, and errors raise on both ranks."""
import os
import random
import socket
import traceback

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from search_common import build_inputs, check_against_trace, load_trace

MOD_TYPES = ["a", "m"]
PAD, LOW, HIGH, MIN_KL, MIN_SCORE = 20, 0.3, 0.7, 0.05, 1.5
PLANTED = {"bin0": [("GATC", 1, "a"), ("CCTGG", 1, "m")], "bin1": [("GAATTC", 2, "a"), ("GCAC......GTT", 2, "a")],
           "bin2": [("CTGCAG", 4, "a"), ("CCTGG", 1, "m")], "bin3": [("TTAA", 3, "a"), ("GCGC", 1, "m")]}


@pytest.fixture(scope="module")
def nmb():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import nanomotif_b200

    return nanomotif_b200


def _metagenome():
    """({bin: {contig: sequence}}, pandas pileup) of four bins and two mod types.  The 'm' rows of bin2 are all below
    the high threshold: that pair has no methylation windows."""
    import pandas as pd

    from nanomotif_b200 import synth

    rng = np.random.default_rng(23)
    bins, parts = {}, []
    for b, planted in PLANTED.items():
        bins[b] = {}
        for i in range(int(rng.integers(1, 4))):
            name = f"{b}_contig_{i}"
            seq = synth.random_sequence(rng, int(rng.integers(20000, 60000)), float(rng.uniform(0.4, 0.6)), 2e-5)
            bins[b][name] = seq.tobytes().decode()
            p = synth.synth_pileup(seq, rng, depth=20, mod_types=tuple(MOD_TYPES), planted=planted)
            frac = p["fraction_mod"]
            if b == "bin2":
                frac = np.where(p["mod_type"] == 1, np.minimum(frac, 0.5), frac)
            n = len(p["position"])
            parts.append(pd.DataFrame({"contig": np.full(n, name, dtype=object), "position": p["position"],
                                       "strand": np.where(p["strand"] == 0, "+", "-").astype(object),
                                       "mod_type": np.array(MOD_TYPES, dtype=object)[p["mod_type"]],
                                       "fraction_mod": frac}))
    return bins, pd.concat(parts, ignore_index=True)


def _sequential(nmb, bins, table, seed):
    """The frame from one search.run per (bin, mod type) pair on its own BinScorer and DeviceDNAarray."""
    from nanomotif_b200 import growth, search

    rows = []
    for b, contigs in bins.items():
        for mt in MOD_TYPES:
            sub = table[table["contig"].isin(list(contigs)) & (table["mod_type"] == mt)]
            pile = {k: sub[k].to_numpy() for k in ("contig", "position", "strand", "fraction_mod")}
            scorer = nmb.BinScorer(pile, contigs, LOW, HIGH)
            asm = scorer.assembly
            cid = np.array([asm.index[c] for c in pile["contig"]], dtype=np.int64)
            windows = growth.methylation_windows(asm, cid, pile["position"], (pile["strand"] == "-").astype(np.uint8),
                                                 pile["fraction_mod"], HIGH, PAD)
            if windows is None:
                continue
            random.seed(seed)
            bg = growth.background_pssm(asm, contigs, search.CANONICAL[mt], PAD)
            co = search.find_candidates(mt, PAD, bg, windows.shape[0], min_kl=MIN_KL, score_threshold=MIN_SCORE)
            rows += search.candidate_rows(b, mt, search.run(co, search.GpuBinBackend(scorer, windows)))
    return search.discovery_frame(rows)


@pytest.mark.parametrize("trace_file", ["search_trace.json", "search_trace_cfg1.json"])
def test_discover_reproduces_reference_trace(nmb, trace_file, monkeypatch):
    from nanomotif_b200 import growth, search
    from nanomotif_b200.motif import Motif

    trace = load_trace(trace_file)
    spec = trace["spec"]
    contigs, pile = build_inputs(spec)
    pile["mod_type"] = np.full(len(pile["position"]), spec["mod_type"], dtype=object)
    multi = nmb.MultiBinScorer(pile, {"bin": contigs}, [spec["mod_type"]], spec["low"], spec["high"])
    setups, results = [], []
    prepare, rows_of = growth.prepare_searches, search.candidate_rows
    monkeypatch.setattr(growth, "prepare_searches", lambda *a, **k: setups.append(prepare(*a, **k)) or setups[-1])
    monkeypatch.setattr(search, "candidate_rows", lambda b, mt, res: results.append(res) or rows_of(b, mt, res))
    df = search.discover(multi, padding=spec["padding"], min_kl=spec["min_kl"], min_motif_score=spec["score_threshold"],
                         seed=spec["random_seed"])
    (_, pssms, totals), = setups
    assert totals == [trace["total_windows"]]
    np.testing.assert_array_equal(pssms[0], np.array(trace["bin_pssm"]))
    # best candidates, every node's alpha / beta / score / priority / depth and the edges (the outer rounds are not
    # recorded through discover: the trace's own rounds stand in for them)
    check_against_trace(trace, results[0], [r for r in trace["rounds"] if "score" in r])
    nodes = {n["motif"]: n for n in trace["nodes"]}
    want = []
    for s in trace["best_candidates"] + trace["missed"]:
        m = Motif(s, spec["padding"]).new_stripped_motif()
        prior = nmb.BetaBernoulliModel()
        want.append(dict(bin="bin", mod_type=spec["mod_type"], motif=m.string, mod_position=m.mod_position,
                         n_mod=nodes[s]["alpha"] - prior._alpha_prior, n_nomod=nodes[s]["beta"] - prior._beta_prior))
    assert df.drop(columns="score").to_dict("records") == want
    np.testing.assert_allclose(df["score"], [nodes[s]["score"] for s in trace["best_candidates"] + trace["missed"]],
                               rtol=1e-6)
    if trace_file == "search_trace_cfg1.json":
        assert df["motif"].tolist()[:3] == ["GATC", "ACCCA", "CCAAAT"]


@pytest.fixture(scope="module")
def meta(nmb):
    bins, table = _metagenome()
    multi = nmb.MultiBinScorer(table, bins, MOD_TYPES, LOW, HIGH)
    return bins, table, multi


def test_discover_equals_sequential_runs_per_pair(nmb, meta, monkeypatch):
    import pandas as pd

    from nanomotif_b200 import search

    bins, table, multi = meta
    launches, kinds = [], []
    real_score, real_find = multi.score_batch, search.find_candidates
    monkeypatch.setattr(multi, "score_batch", lambda reqs: launches.append(len(reqs)) or real_score(reqs))

    def recording(*args, **kw):  # the request kinds of every search, in order: request k is answered in round k
        log = []
        kinds.append(log)
        co = real_find(*args, **kw)
        try:
            request = next(co)
            while True:
                log.append(request[0])
                request = co.send((yield request))
        except StopIteration as stop:
            return stop.value

    monkeypatch.setattr(search, "find_candidates", recording)
    random.seed(4321)
    state = random.getstate()
    df = search.discover(multi, seed=7)
    assert random.getstate() == state
    monkeypatch.undo()
    want = _sequential(nmb, bins, table, 7)
    pd.testing.assert_frame_equal(df, want, check_exact=True)
    assert len(df) >= 4 and set(df["mod_type"]) == set(MOD_TYPES)
    assert not ((df["bin"] == "bin2") & (df["mod_type"] == "m")).any()  # no confident rows: no search, no rows
    assert len(kinds) == len(bins) * len(MOD_TYPES) - 1
    rounds = sorted({k for log in kinds for k, kind in enumerate(log) if kind == "score"})
    assert launches == [sum(len(log) > k and log[k] == "score" for log in kinds) for k in rounds]
    assert launches[0] == len(kinds)  # every pair's root in the first launch


def test_bin_subset_and_order(nmb, meta):
    import pandas as pd

    from nanomotif_b200 import search

    bins, table, multi = meta
    full = search.discover(multi, seed=3)
    for order in (["bin3", "bin1", "bin0", "bin2"], ["bin2", "bin0"], ["bin1"]):
        want = pd.concat([full[full["bin"] == b] for b in order], ignore_index=True)
        pd.testing.assert_frame_equal(search.discover(multi, bins=order, seed=3), want, check_exact=True)
        permuted = nmb.MultiBinScorer(table, {b: bins[b] for b in order}, MOD_TYPES, LOW, HIGH)
        pd.testing.assert_frame_equal(search.discover(permuted, seed=3), want, check_exact=True)
    only_m = search.discover(multi, mod_types=["m"], seed=3)
    pd.testing.assert_frame_equal(only_m, full[full["mod_type"] == "m"].reset_index(drop=True), check_exact=True)
    assert search.discover(multi, bins=[], seed=3).empty
    with pytest.raises(KeyError):
        search.discover(multi, bins=["bin9"])
    with pytest.raises(ValueError):
        search.discover(multi, mod_types=["21839"])


def test_prepare_errors_pass_through(nmb, meta):
    from nanomotif_b200 import search

    bins, table, _ = meta
    short = nmb.MultiBinScorer(table, {"tiny": {"t0": "ACGT" * 15}}, MOD_TYPES, LOW, HIGH)  # 60 bp: 20 window starts
    with pytest.raises(ValueError, match="Too many samples requested for unique subsequences"):
        search.discover(short)
    no_rows = nmb.MultiBinScorer(table, bins, MOD_TYPES, LOW, HIGH, keep_rows=False)
    with pytest.raises(ValueError, match="keeps no pileup rows"):
        search.discover(no_rows)


# ---------------------------------------------------------------------------------------------
# world size 2
# ---------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _checks(rank, world, dev):
    import pandas as pd

    import nanomotif_b200 as nmb
    from nanomotif_b200 import search, sharding

    fails = []

    def same(got, want, what):
        try:
            pd.testing.assert_frame_equal(got, want, check_exact=True)
        except AssertionError as exc:
            fails.append(f"{what}: {exc}")

    def raises(fn, message, what):
        try:
            fn()
            fails.append(f"{what}: no ValueError")
        except ValueError as exc:
            if message not in str(exc):
                fails.append(f"{what}: {exc}")
        except Exception as other:  # noqa: BLE001
            fails.append(f"{what}: {other!r} instead of ValueError")

    bins, table = _metagenome()
    want = search.discover(nmb.MultiBinScorer(table, bins, MOD_TYPES, LOW, HIGH, dev), seed=5)
    plan = sharding.discovery_plan(bins, world)
    held = [b for b in bins if plan[b] == rank]
    if not held:
        fails.append(f"rank {rank} holds no bin of four")
    args = (bins, MOD_TYPES, LOW, HIGH, rank, world)
    same(sharding.discover(table, *args, seed=5, device=dev), want, "table")
    parts = {(b, mt): table[table["contig"].isin(list(cs)) & (table["mod_type"] == mt)]
             for b, cs in bins.items() for mt in MOD_TYPES}
    same(sharding.discover(parts, *args, seed=5, device=dev), want, "partitioned")
    lengths = {b: {c: (s if b in held else len(s)) for c, s in cs.items()} for b, cs in bins.items()}
    local = nmb.MultiBinScorer(table, {b: bins[b] for b in held}, MOD_TYPES, LOW, HIGH, dev)
    same(sharding.discover_local(local, lengths, MOD_TYPES, rank, world, seed=5), want, "local scorer")
    same(sharding.discover(table, lengths, MOD_TYPES, LOW, HIGH, rank, world, seed=5, device=dev), want,
         "other ranks' contigs by length")

    # a rank without bins takes part
    one = {"bin1": bins["bin1"]}
    want_one = search.discover(nmb.MultiBinScorer(table, one, MOD_TYPES, LOW, HIGH, dev), seed=5)
    same(sharding.discover(table, one, MOD_TYPES, LOW, HIGH, rank, world, seed=5, device=dev), want_one, "one bin")
    mine = nmb.MultiBinScorer(table, one, MOD_TYPES, LOW, HIGH, dev) if rank == 0 else None
    same(sharding.discover_local(mine, one, MOD_TYPES, rank, world, seed=5, device=dev), want_one, "one bin, local")

    # errors on one rank raise on both: a contig too short for its background samples, a local scorer off the plan
    short = {"bin0": bins["bin0"], "tiny": {"t0": "ACGT" * 15}}
    if sharding.discovery_plan(short, world) != {"bin0": 0, "tiny": 1}:
        fails.append("short-contig layout")
    raises(lambda: sharding.discover(table, short, MOD_TYPES, LOW, HIGH, rank, world, device=dev),
           "Too many samples requested for unique subsequences", "short contig")
    wrong = local if rank == 0 else None
    raises(lambda: sharding.discover_local(wrong, lengths, MOD_TYPES, rank, world, device=dev),
           "rank 1: the local scorer's bins are not those the discovery plan gives this rank", "local scorer off plan")
    raises(lambda: sharding.discover(table, {b: {c: len(s) for c, s in cs.items()} for b, cs in bins.items()},
                                     MOD_TYPES, LOW, HIGH, rank, world, device=dev),
           "which was given by length only", "own contig by length")
    same(sharding.discover(table, *args, seed=5, device=dev), want, "after the errors")
    return fails, len(want)


def _worker(rank, world, port, backend, q):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        q.put((rank,) + _checks(rank, world, dev))
    except Exception:  # noqa: BLE001 -- reported to the test process
        q.put((rank, [traceback.format_exc()], 0))
    finally:
        dist.destroy_process_group()


def test_two_ranks_return_the_one_gpu_frame():
    import torch
    import torch.multiprocessing as mp

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    world = 2
    backend = "nccl" if torch.cuda.device_count() >= world else "gloo"
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, backend, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = sorted(q.get(timeout=900) for _ in range(world))
        for p in procs:
            p.join(timeout=120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    for rank, fails, _ in results:
        assert not fails, f"rank {rank}:\n" + "\n".join(fails[:20])
    assert results[0][2] == results[1][2] > 0
