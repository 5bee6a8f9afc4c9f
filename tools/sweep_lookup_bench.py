#!/usr/bin/env python
"""Sweep lookup at the cfg3 scale (development tool): BinSweep.count_matrix over the bins bench.py keeps resident
(synth.cfg3_plan, built by bench.Resident, as tools/bin_sweep_bench.py builds them), mod type 'a'.

  * nmb_sweep_lookup kernel time (CUDA events, after a warm-up launch) and count_matrix wall time for three motif sets:
    (a) the union of every bin's candidates(prune=True) motifs, (b) random covered motifs of every shape, (c) N-heavy
    8-mers, the worst case (up to 5^7 cells per class);
  * cells and 32-byte sectors the launch reads, from the records (a slot starts every HIST_SIZE / BIP_SIZE counters;
    HIST_SIZE * 4 bytes is 16 mod 32, so odd IUPAC slots are shifted by half a sector);
  * BinSweep.counts per call on a small sample, the one-motif route the lookup replaces;
  * MultiBinScorer.score_batch (K2, one scan launch) on the same matrix for set (a), and whether it agrees;
  * sha256 of every matrix, so that runs can be compared.

The histograms (400 bins: 24.6 GB finished) are far larger than L2, but a set that touches few cells per bin is
partly served from L2 across the timed repetitions; the sector counts say how much each launch has to read.

    python tools/sweep_lookup_bench.py [--bins 400] [--bin-bp 5000000] [--random 100000] [--reps 5] [--json out.json]
"""
import argparse
import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (Resident: the resident bins of the benchmark)
from nanomotif_b200 import _lib, synth  # noqa: E402
from nanomotif_b200.api import MultiBinScorer  # noqa: E402
from nanomotif_b200.motif import Motif  # noqa: E402
from nanomotif_b200.sweep import (BIP_LETTERS, BIP_SIZE, HIST_SIZE, IUPAC_ORDER, BinSweep,  # noqa: E402
                                  _lookup_records)
from tools.bin_sweep_bench import gpu_info  # noqa: E402


def random_motifs(rng, n, canon="A"):
    """n covered motifs: 60 % IUPAC 4..8-mers, 20 % ACGT bipartite, 20 % bipartite with IUPAC halves."""
    motifs, mps = [], []
    for _ in range(n):
        r = rng.random()
        if r < 0.6:
            s = list(rng.choice(list(IUPAC_ORDER), int(rng.integers(4, 9))))
            o = int(rng.integers(len(s)))
            s[o] = canon
            motifs.append("".join(s))
            mps.append(o)
        else:
            a, b = (int(x) for x in rng.choice([3, 4], 2))
            g = int(rng.integers(4, 9))
            h = list(rng.choice(list("ACGT" if r < 0.8 else BIP_LETTERS), a + b))
            o = int(rng.integers(a + b))
            h[o] = canon
            motifs.append("".join(h[:a]) + "N" * g + "".join(h[a:]))
            mps.append(o if o < a else o + g)
    return motifs, mps


def n_heavy(rng, n, canon="A"):
    """8-mers whose every letter but the modified one is N with probability 0.9, else a random IUPAC letter."""
    motifs, mps = [], []
    for _ in range(n):
        o = int(rng.integers(8))
        s = ["N" if rng.random() < 0.9 else IUPAC_ORDER[int(rng.integers(15))] for _ in range(8)]
        s[o] = canon
        motifs.append("".join(s))
        mps.append(o)
    return motifs, mps


def cells_and_sectors(records, n_bins) -> dict:
    """Counters and 32-byte sectors one launch over n_bins slots reads, from the records."""
    off, owner = records["base"].astype(np.int64), np.arange(len(records))
    for p in range(7):
        ns = np.where(p < records["n_pos"][owner], records["n_states"][owner, p], 1).astype(np.int64)
        rep = np.repeat(np.arange(len(off)), ns)
        digit = np.arange(len(rep)) - np.repeat(np.cumsum(ns) - ns, ns)
        off = off[rep] + np.where(p < records["n_pos"][owner[rep]], records["offset"][owner[rep], p, digit], 0)
        owner = owner[rep]
    step = records["class_step"][owner].astype(np.int64)
    kind = records["kind"][owner]
    counters = np.concatenate([off, off + step])
    key_owner, key_kind = np.concatenate([owner, owner]), np.concatenate([kind, kind])
    sectors = 0
    for k, size in ((0, HIST_SIZE), (1, BIP_SIZE)):
        sel = key_kind == k
        for shift, slots in ((0, (n_bins + 1) // 2), ((size % 8), n_bins // 2)):  # even / odd slots
            keys = key_owner[sel] * (1 << 24) + (counters[sel] + shift) // 8
            sectors += len(np.unique(keys)) * slots
    return {"queries": len(records), "cells_per_class": int(len(off)), "max_cells": int(np.bincount(owner).max()),
            "counters_read": int(2 * len(off)) * n_bins, "sectors_read": int(sectors),
            "bytes_read_sectors": int(sectors) * 32}


def digest(*arrays) -> str:
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bins", type=int, default=400)
    ap.add_argument("--bin-bp", type=int, default=5_000_000)
    ap.add_argument("--random", type=int, default=100_000)
    ap.add_argument("--heavy", type=int, default=500)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--counts-sample", type=int, default=20)
    ap.add_argument("--min-mean", type=float, default=0.7)
    ap.add_argument("--min-mod", type=int, default=50)
    ap.add_argument("--json", default=None, help="also write the result here")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = {**gpu_info(), "bins": args.bins, "bin_bp": args.bin_bp, "mod_type": "a"}
    print(json.dumps(result), flush=True)

    t0 = time.perf_counter()
    plan = synth.cfg3_plan(args.bins, args.bin_bp)
    res = bench.Resident(synth, plan, range(args.bins), dev)
    scorer = MultiBinScorer.from_device(res.asm, res.pile, {f"bin_{b}": res.ranges[b] for b in res.bins},
                                        bench.MOD_TYPES)
    sw = BinSweep(scorer, "a")
    sw.hist, sw.bip
    torch.cuda.synchronize()
    result["assembly_bp"] = int(res.asm.total_bp)
    result["setup_s"] = round(time.perf_counter() - t0, 1)
    t0 = time.perf_counter()
    df = sw.candidates(min_mean=args.min_mean, min_mod=args.min_mod, prune=True)
    result["candidates_prune_s"] = round(time.perf_counter() - t0, 2)
    pairs = sorted(set(zip(df["motif"], df["mod_position"].tolist())))
    rng = np.random.default_rng(2026)
    sets = {"candidates_union": ([m for m, _ in pairs], [p for _, p in pairs]),
            "random": random_motifs(rng, args.random), "n_heavy_8mers": n_heavy(rng, args.heavy)}
    n_bins = len(sw.bins)
    slots = torch.arange(n_bins, dtype=torch.int32, device=dev)
    matrices = {}
    for name, (motifs, mps) in sets.items():
        records = _lookup_records(motifs, mps, True, "")
        q = torch.from_numpy(records.view(np.uint8)).to(dev)
        out = torch.empty((n_bins, len(records), 2), dtype=torch.int64, device=dev)

        def launch():
            _lib.check(_lib.lib.nmb_sweep_lookup(_lib.ptr(sw.hist), _lib.ptr(sw.bip), _lib.ptr(slots), n_bins,
                                                 _lib.ptr(q), len(records), _lib.ptr(out), None), "nmb_sweep_lookup")

        launch()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            launch()
            ev[1].record()
            torch.cuda.synchronize()
            times.append(ev[0].elapsed_time(ev[1]))
        t0 = time.perf_counter()
        n_mod, n_nomod = sw.count_matrix(motifs, mps)
        wall = time.perf_counter() - t0
        assert np.array_equal(out[..., 0].cpu().numpy(), n_mod)
        matrices[name] = (motifs, mps, n_mod, n_nomod)
        shape = cells_and_sectors(records, n_bins)
        ms = sorted(times)[len(times) // 2]
        result[name] = {**shape, "kernel_ms": sorted(round(t, 3) for t in times), "count_matrix_wall_s": round(wall, 3),
                        "sector_GB_per_s": round(shape["bytes_read_sectors"] / (ms * 1e-3) / 1e9, 1),
                        "nonzero_entries": int((n_mod > 0).sum()), "hash": digest(n_mod, n_nomod)}
        print(json.dumps({name: result[name]}), flush=True)
        del q, out

    # the one-motif route: BinSweep.counts per (bin, motif)
    motifs, mps, n_mod, n_nomod = matrices["random"]
    per_call, agree = [], True
    for i in range(args.counts_sample):
        b, j = int(rng.integers(n_bins)), int(rng.integers(len(motifs)))
        if len(motifs[j]) > 8 and not set(motifs[j]) <= set("ACGTN"):
            continue
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = sw.counts(sw.bins[b], motifs[j], mps[j])
        per_call.append((time.perf_counter() - t0) * 1e3)
        agree &= got == (int(n_mod[b, j]) & 0xFFFFFFFF, int(n_nomod[b, j]) & 0xFFFFFFFF)
    result["counts_per_call_ms"] = {"n": len(per_call), "median": round(float(np.median(per_call)), 3),
                                    "max": round(float(max(per_call)), 3), "agrees_with_count_matrix": bool(agree)}

    # K2 on the candidate-union matrix
    motifs, mps, n_mod, n_nomod = matrices["candidates_union"]
    objs = [Motif(m, p).from_iupac() for m, p in zip(motifs, mps)]
    requests = [(scorer.context(b, "a"), objs) for b in sw.bins]
    scorer.score_batch(requests)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    k2 = scorer.score_batch(requests)
    result["k2_score_batch_s"] = round(time.perf_counter() - t0, 3)
    k2 = np.stack(k2)  # [bin][motif][2]
    result["k2_motifs"] = len(objs)
    result["k2_equal"] = bool(np.array_equal(k2[..., 0], n_mod) and np.array_equal(k2[..., 1], n_nomod))
    result["k2_hash"] = digest(k2[..., 0], k2[..., 1])
    print(json.dumps(result, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(json.dumps(result) + "\n")


if __name__ == "__main__":
    main()
