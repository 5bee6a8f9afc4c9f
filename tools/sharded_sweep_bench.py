#!/usr/bin/env python
"""The sharded per-bin sweep (sharding.ShardedBinSweep) at the cfg3 scale (development tool): the 400 bins bench.py
keeps resident (synth.cfg3_plan, 2.0 Gbp), mod type 'a', shard plan of ShardedMultiBinScorer.plan; every rank builds
its own bins on its own GPU (bench.Resident + MultiBinScorer.from_device + ShardedMultiBinScorer.from_local).

  * histogram launches (CUDA events around every nmb_sweep_hist / nmb_sweep_bipartite launch) and the split-bin
    all-reduce (CUDA events around every all-reduce the sweep issues), maximum over ranks;
  * candidates(prune=True) over all bins and candidates(prune=True, bipartite_letters="IUPAC") over the first
    --iupac-bins bins: wall time with a device synchronise, maximum over ranks, --reps repetitions;
  * peak device memory of every rank, and the SHA-256 of each frame's CSV bytes (checked equal on every rank);
  * with one process, also the frames of BinSweep over the same scorer, as tools/sweep_prune_bench.py computes them.

    python -m torch.distributed.run --nproc-per-node N tools/sharded_sweep_bench.py [--bins 400] [--iupac-bins 100]
        [--reps 2] [--json out.json]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (Resident: the resident bins of the benchmark)
from nanomotif_b200 import synth  # noqa: E402
from nanomotif_b200._lib import lib  # noqa: E402
from nanomotif_b200.api import MultiBinScorer  # noqa: E402
from nanomotif_b200.sharding import ShardedBinSweep, ShardedMultiBinScorer  # noqa: E402
from nanomotif_b200.sweep import BinSweep  # noqa: E402


def gpu_info(n: int) -> list:
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[:n] if out else [torch.cuda.get_device_name(0)]


class EventTimer:
    """Wraps callables of a module with CUDA events on the current stream; ms() sums the device time of the calls
    since the last reset (read after a synchronise)."""

    def __init__(self, module, names):
        self.events = []
        for name in names:
            setattr(module, name, self._wrap(getattr(module, name)))

    def _wrap(self, fn):
        def call(*args, **kw):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            rc = fn(*args, **kw)
            ev[1].record()
            self.events.append(ev)
            return rc

        call.__name__ = fn.__name__
        return call

    def reset(self):
        self.events = []

    def ms(self):
        return sum(a.elapsed_time(b) for a, b in self.events)


def gather(x, world):
    if world == 1:
        return [x]
    out = [None] * world
    dist.all_gather_object(out, x)
    return out


def barrier(world):
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()


def frame_sha(df) -> str:
    return hashlib.sha256(df.to_csv(index=False).encode()).hexdigest()


def timed_candidates(sw, world, reps, **kw):
    walls = []
    for _ in range(reps):
        barrier(world)
        t0 = time.perf_counter()
        df = sw.candidates(**kw)
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    walls = np.max(np.array(gather(walls, world)), axis=0)  # per repetition: the slowest rank
    shas = gather(frame_sha(df), world)
    assert len(set(shas)) == 1, shas
    return {"wall_s": [round(float(w), 3) for w in walls], "rows": len(df), "sha256": shas[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bins", type=int, default=400)
    ap.add_argument("--iupac-bins", type=int, default=100)
    ap.add_argument("--bin-bp", type=int, default=5_000_000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--min-mean", type=float, default=0.7)
    ap.add_argument("--min-mod", type=int, default=50)
    ap.add_argument("--json", default=None, help="rank 0 also writes the result here")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    result = {"gpus": gpu_info(world), "world_size": world, "bins": args.bins, "iupac_bins": args.iupac_bins,
              "bin_bp": args.bin_bp, "mod_type": "a", "min_mean": args.min_mean, "min_mod": args.min_mod}

    t0 = time.perf_counter()
    plan = synth.cfg3_plan(args.bins, args.bin_bp)
    names = [f"bin_{b}" for b in range(args.bins)]
    bins = {f"bin_{b}": {f"contig_{i}": int(plan["lengths"][i]) for i in range(*plan["ranges"][b])}
            for b in range(args.bins)}
    _, per_rank, split, _ = ShardedMultiBinScorer.plan(bins, world)
    if split:  # bench.Resident builds whole bins; pieces of a split bin would need their own text and rows
        raise SystemExit(f"bins split over ranks: {sorted(split)}")
    mine = [int(b[4:]) for b in per_rank[rank]]
    local = None
    if mine:
        res = bench.Resident(synth, plan, mine, dev)
        local = MultiBinScorer.from_device(res.asm, res.pile, {f"bin_{b}": res.ranges[b] for b in res.bins},
                                           bench.MOD_TYPES)
    scorer = ShardedMultiBinScorer.from_local(local, bins, bench.MOD_TYPES, rank, world, dev)
    barrier(world)
    result["setup_s"] = round(max(gather(time.perf_counter() - t0, world)), 1)
    result["bins_per_rank"] = gather(len(mine), world)
    result["bp_per_rank"] = gather(int(local.assembly.total_bp) if local else 0, world)
    result["split_bins"] = len(split)

    hist_timer = EventTimer(lib, ("nmb_sweep_hist", "nmb_sweep_bipartite"))
    reduce_timer = EventTimer(dist, ("all_reduce",))
    ssw = ShardedBinSweep(scorer, "a")
    if ssw.local is not None:
        ssw.local.hist, ssw.local.bip  # finish the histograms outside the timed calls
    barrier(world)
    result["hist_ms"] = round(max(gather(hist_timer.ms(), world)), 2)
    result["split_allreduce_ms"] = round(max(gather(reduce_timer.ms(), world)), 3)
    result["split_allreduces"] = len(reduce_timer.events)
    kw = dict(min_mean=args.min_mean, min_mod=args.min_mod, prune=True)
    result["acgt_pruned"] = timed_candidates(ssw, world, args.reps, **kw)
    if rank == 0:
        print(json.dumps(result), flush=True)
    del ssw
    torch.cuda.empty_cache()

    sub = ShardedBinSweep(scorer, "a", bins=names[:args.iupac_bins])
    if sub.local is not None:
        sub.local.hist, sub.local.bip
    result["iupac_pruned"] = timed_candidates(sub, world, args.reps, bipartite_letters="IUPAC", **kw)
    result["max_memory_allocated_gb"] = [round(x / 1e9, 2) for x in gather(torch.cuda.max_memory_allocated(dev), world)]
    del sub
    torch.cuda.empty_cache()

    if world == 1:  # the frames of one BinSweep over the same bins, as tools/sweep_prune_bench.py computes them
        sw = BinSweep(local, "a")
        result["binsweep_acgt_pruned_sha256"] = frame_sha(sw.candidates(**kw))
        del sw
        torch.cuda.empty_cache()
        sw = BinSweep(local, "a", bins=names[:args.iupac_bins])
        result["binsweep_iupac_pruned_sha256"] = frame_sha(sw.candidates(bipartite_letters="IUPAC", **kw))
    if rank == 0:
        print(json.dumps(result, indent=1), flush=True)
        if args.json:
            os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
            with open(args.json, "w") as f:
                f.write(json.dumps(result) + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
