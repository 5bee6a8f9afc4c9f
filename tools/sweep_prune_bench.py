#!/usr/bin/env python
"""Candidate pruning of the per-bin sweep at the cfg3 scale (development tool): the bins bench.py keeps resident
(synth.cfg3_plan, built by bench.Resident), mod type 'a'.

  * BinSweep.candidates() against candidates(prune=True), alternating: wall time (host frame included), device time
    of the filter passes (CUDA events around every nmb_sweep_*filter launch), and rows in total, per-bin median and
    per-bin maximum; the same for bipartite_letters="IUPAC" on the first --iupac-bins bins;
  * planted recovery: how many planted 'a' motifs of sweep shape appear verbatim in their bin's frame, and in how
    many bins where they were not planted;
  * residual noise: the pruned rows that are not a planted motif of their bin, per bin.

    python tools/sweep_prune_bench.py [--bins 400] [--iupac-bins 100] [--reps 2] [--json out.json]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (Resident: the resident bins of the benchmark)
from nanomotif_b200 import synth  # noqa: E402
from nanomotif_b200._lib import lib  # noqa: E402
from nanomotif_b200.api import MultiBinScorer  # noqa: E402
from nanomotif_b200.sweep import MAX_K, BinSweep  # noqa: E402

SETS = {"AG": "R", "CT": "Y", "AT": "W", "CG": "S", "GT": "K", "AC": "M"}
FILTERS = ("nmb_sweep_expand_filter", "nmb_sweep_bipartite_filter", "nmb_sweep_bip_iupac_expand_filter")


def iupac(regex: str) -> str:
    toks = re.findall(r"\[[^\]]*\]|.", regex)
    return "".join("N" if t == "." else SETS["".join(sorted(t[1:-1]))] if t.startswith("[") else t for t in toks)


def sweep_shape(motif: str) -> bool:
    return len(motif) <= MAX_K or re.fullmatch(r"[ACGT]{3,4}N{4,8}[ACGT]{3,4}", motif) is not None


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, power = (out[0].split(", ") + ["?"])[:2] if out else (torch.cuda.get_device_name(0), "?")
    return {"gpu": name, "power_limit": power}


class FilterTimer:
    """Wraps the three filter entry points of the bound library with CUDA events on the current stream; `ms()` is the
    summed device time of the launches since the last reset (call after a synchronize)."""

    def __init__(self):
        self.events = []
        for name in FILTERS:
            setattr(lib, name, self._wrap(getattr(lib, name)))

    def _wrap(self, fn):
        def call(*args):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            rc = fn(*args)
            ev[1].record()
            self.events.append(ev)
            return rc

        call.__name__ = fn.__name__
        return call

    def reset(self):
        self.events = []

    def ms(self):
        return sum(a.elapsed_time(b) for a, b in self.events)


def run(sw, timer, **kw):
    torch.cuda.synchronize()
    timer.reset()
    t0 = time.perf_counter()
    df = sw.candidates(**kw)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return df, wall, timer.ms(), len(timer.events)


def per_bin(df, names):
    counts = df["bin"].value_counts().reindex(names, fill_value=0).to_numpy()
    return {"rows": int(counts.sum()), "per_bin_median": float(np.median(counts)), "per_bin_max": int(counts.max()),
            "rows_bipartite": int((df["motif"].str.len() > MAX_K).sum())}


def planted_sets(plan, bins, names):
    """bin name -> {(motif, mod_position)} of its planted 'a' motifs of sweep shape."""
    own = {}
    for b, name in zip(bins, names):
        own[name] = {(iupac(regex), mp) for regex, mp, mt in plan["planted"][b]
                     if mt == "a" and sweep_shape(iupac(regex))}
    return own


def planted_recovery(df, own, names):
    """Planted 'a' motifs of sweep shape: found verbatim in their bin, and bins without them that list them."""
    pool = {(iupac(regex), mp) for regex, mp in synth.PLANT_POOL["a"] if sweep_shape(iupac(regex))}
    sel = df[df["motif"].isin({m for m, _ in pool})]  # the few rows that spell a planted motif
    keys = set(zip(sel["bin"], sel["motif"], sel["mod_position"]))
    found = sum((name, m, p) in keys for name in names for m, p in own[name])
    total = sum(len(own[name]) for name in names)
    elsewhere = {f"{m}@{p}": sum((name, m, p) in keys and (m, p) not in own[name] for name in names)
                 for m, p in sorted(pool)}
    return {"found": found, "planted": total, "bins_listing_it_where_not_planted": elsewhere}


def residual(df, own, names):
    """Rows that are not a planted motif of their bin, per bin, and the most frequent such rows over all bins."""
    is_own = np.array([(m, p) in own[b] for b, m, p in zip(df["bin"], df["motif"], df["mod_position"])], dtype=bool)
    rest = df[~is_own]
    counts = rest["bin"].value_counts().reindex(names, fill_value=0).to_numpy()
    top = rest.groupby(["motif", "mod_position"]).size().sort_values(ascending=False).head(15)
    return {"rows": int(counts.sum()), "per_bin_median": float(np.median(counts)), "per_bin_max": int(counts.max()),
            "bins_without_residual": int((counts == 0).sum()),
            "most_frequent": [[m, int(p), int(n)] for (m, p), n in top.items()]}


def compare(sw, timer, names, reps, plan, bins, letters, args):
    kw = dict(min_mean=args.min_mean, min_mod=args.min_mod, bipartite_letters=letters)
    times = {"full": [], "pruned": []}
    frames = {}
    for r in range(reps):  # alternating, the order swapped every repetition
        for name in (("full", "pruned") if r % 2 == 0 else ("pruned", "full")):
            df, wall, dev, launches = run(sw, timer, prune=name == "pruned", **kw)
            times[name].append({"wall_s": round(wall, 3), "filter_device_ms": round(dev, 2), "filter_launches": launches})
            frames[name] = df
            del df
    out = {"times": times}
    own = planted_sets(plan, bins, names)
    for name, df in frames.items():
        out[name] = per_bin(df, names)
        out[name]["planted"] = planted_recovery(df, own, names)
    out["pruned"]["residual"] = residual(frames["pruned"], own, names)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bins", type=int, default=400)
    ap.add_argument("--iupac-bins", type=int, default=100)
    ap.add_argument("--bin-bp", type=int, default=5_000_000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--min-mean", type=float, default=0.7)
    ap.add_argument("--min-mod", type=int, default=50)
    ap.add_argument("--json", default=None, help="also write the result here")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = {**gpu_info(), "bins": args.bins, "iupac_bins": args.iupac_bins, "bin_bp": args.bin_bp, "mod_type": "a",
              "min_mean": args.min_mean, "min_mod": args.min_mod}
    print(json.dumps(result), flush=True)

    t0 = time.perf_counter()
    plan = synth.cfg3_plan(args.bins, args.bin_bp)
    res = bench.Resident(synth, plan, range(args.bins), dev)
    names = [f"bin_{b}" for b in res.bins]
    scorer = MultiBinScorer.from_device(res.asm, res.pile, {f"bin_{b}": res.ranges[b] for b in res.bins},
                                        bench.MOD_TYPES)
    result["assembly_bp"] = int(res.asm.total_bp)
    result["setup_s"] = round(time.perf_counter() - t0, 1)
    timer = FilterTimer()

    sw = BinSweep(scorer, "a")
    sw.hist, sw.bip  # finish the histograms outside the timed calls
    result["acgt"] = compare(sw, timer, names, args.reps, plan, res.bins, "ACGT", args)
    print(json.dumps({"setup_s": result["setup_s"], "acgt": result["acgt"]}), flush=True)
    del sw
    torch.cuda.empty_cache()

    sub = names[:args.iupac_bins]
    sw = BinSweep(scorer, "a", bins=sub)
    sw.hist, sw.bip
    result["iupac"] = compare(sw, timer, sub, args.reps, plan, res.bins[:args.iupac_bins], "IUPAC", args)
    text = json.dumps(result)
    print(json.dumps(result, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
