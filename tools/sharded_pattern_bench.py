#!/usr/bin/env python
"""The sharded contig x motif methylation-pattern table (sharding.ShardedPatternTable) at the cfg4 shape (development
tool): 50 000 lognormal contigs over 1.5 Gbp and 500 bin-motifs.tsv-style motifs (tools/pattern_bench.py bin_motifs),
mod type 'a'.  Every rank derives the shard plan from the contig lengths and generates only its own contigs and rows on
its own GPU (synth.device_pattern_workload with keep=, from a fixed seed: the same data at every world size), then
ShardedPatternTable.from_local.

Reported as the maximum over ranks: index build time; table time (median and weighted mean, wall time with a device
synchronise, the gather included) and, inside it, the gather time (place + all-reduce + NaN restore); motif*bp/s of the
table.  Also the SHA-256 of the finished arrays (equal at every world size) and the card name and power limit.

    python -m torch.distributed.run --nproc-per-node N tools/sharded_pattern_bench.py [--contigs 50000]
        [--bp 1500000000] [--motifs 500] [--reps 3] [--json out.json]
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
sys.path.insert(0, os.path.join(ROOT, "tools"))
from nanomotif_b200 import sharding, synth  # noqa: E402
from pattern_bench import bin_motifs  # noqa: E402


def gpu_info(n: int) -> list:
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[:n] if out else [torch.cuda.get_device_name(0)]


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


class GatherTimer:
    """Wall time of every sharding.gather_columns call, between device synchronises."""

    def __init__(self):
        self.s = 0.0
        inner = sharding.gather_columns

        def timed(*args, **kw):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = inner(*args, **kw)
            torch.cuda.synchronize()
            self.s += time.perf_counter() - t0
            return out

        sharding.gather_columns = timed


def digest(stats, value) -> str:
    h = hashlib.sha256(stats.cpu().numpy().tobytes())
    if value is not None:
        h.update(value.cpu().numpy().tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=50_000)
    ap.add_argument("--bp", type=int, default=1_500_000_000)
    ap.add_argument("--motifs", type=int, default=500)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None, help="rank 0 also writes the result here")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    result = {"gpus": gpu_info(world), "world_size": world, "contigs": args.contigs, "bp": args.bp, "motifs": args.motifs}

    lengths = synth.pattern_workload_lengths(args.bp, args.contigs)
    contigs = {f"c{i}": int(n) for i, n in enumerate(lengths)}
    keep = np.flatnonzero(sharding.plan_shards(lengths, world) == rank)
    asm, rows = synth.device_pattern_workload(dev, args.bp, args.contigs, keep=keep) if len(keep) else (None, None)
    n_rows = int(rows["position"].numel()) if rows is not None else 0
    result["contigs_per_rank"] = gather(len(keep), world)
    result["bp_per_rank"] = gather(int(lengths[keep].sum()), world)
    result["rows_per_rank"] = gather(n_rows, world)
    motifs = [f"{m.iupac()}_a_{m.mod_position}" for m in bin_motifs(np.random.default_rng(2), args.motifs)]

    barrier(world)
    t0 = time.perf_counter()
    tab = sharding.ShardedPatternTable.from_local(asm, rows, contigs, ["a"], rank, world, dev)
    torch.cuda.synchronize()
    result["index_s"] = round(max(gather(time.perf_counter() - t0, world)), 4)
    del rows

    timer = GatherTimer()
    units = len(motifs) * int(lengths.sum())
    for median in (True, False):
        tab.table(motifs[:64], median, on_device=True)  # warm-up: modules, allocator, communicator
        walls, gathers = [], []
        for _ in range(args.reps):
            barrier(world)
            timer.s = 0.0
            t0 = time.perf_counter()
            stats, value = tab.table(motifs, median, on_device=True)
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
            gathers.append(timer.s)
        wall = np.max(np.array(gather(walls, world)), axis=0)  # per repetition: the slowest rank
        gat = np.max(np.array(gather(gathers, world)), axis=0)
        shas = gather(digest(stats, value), world)
        assert len(set(shas)) == 1, shas
        key = "median" if median else "weighted_mean"
        result[key] = {"table_s": [round(float(w), 4) for w in wall], "gather_s": [round(float(g), 4) for g in gat],
                       "motif_bp_per_s": float(units / wall.min()), "cells_observed": int((stats[:, :, 0] > 0).sum()),
                       "sha256": shas[0]}
        del stats, value
    result["peak_mem_gb"] = gather(round(torch.cuda.max_memory_allocated(dev) / 1e9, 1), world)
    if rank == 0:
        line = json.dumps(result)
        print(line, flush=True)
        if args.json:
            os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
            with open(args.json, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
