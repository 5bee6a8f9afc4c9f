#!/usr/bin/env python
"""Per-bin sweep at the cfg3 scale (development tool): the bins bench.py keeps resident (synth.cfg3_plan, built by
bench.Resident), mod type 'a'.

  * the per-bin histograms (IUPAC, bipartite) of all bins from one launch each (sweep.BinSweep) against one
    SweepIndex(...).add(begin, end) per bin, alternating, timed with CUDA events; every bin's raw and finished
    histograms must be bit-identical between the two;
  * BinSweep.candidates() for all bins: time and rows;
  * device bytes of each phase, from shapes;
  * per bin, whether its planted 'a' motifs of sweep shape are among its candidates, and in which other bins they
    show up.

    python tools/bin_sweep_bench.py [--bins 400] [--bin-bp 5000000] [--reps 3] [--json out.json]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (Resident: the resident bins of the benchmark)
from nanomotif_b200 import synth  # noqa: E402
from nanomotif_b200.api import MultiBinScorer  # noqa: E402
from nanomotif_b200.sweep import BIP_SIZE, HIST_SIZE, MAX_K, BinSweep, SweepIndex, table_scratch_bytes  # noqa: E402

SETS = {"AG": "R", "CT": "Y", "AT": "W", "CG": "S", "GT": "K", "AC": "M"}


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bins", type=int, default=400)
    ap.add_argument("--bin-bp", type=int, default=5_000_000)
    ap.add_argument("--reps", type=int, default=3)
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
    names = [f"bin_{b}" for b in res.bins]
    scorer = MultiBinScorer.from_device(res.asm, res.pile, {f"bin_{b}": res.ranges[b] for b in res.bins},
                                        bench.MOD_TYPES)
    result["assembly_bp"] = int(res.asm.total_bp)
    result["setup_s"] = round(time.perf_counter() - t0, 1)

    sw = BinSweep(scorer, "a")
    loop = [SweepIndex(res.asm, res.pile, 0).add_bipartite(*res.ranges[b]) for b in res.bins]  # warm + allocate
    torch.cuda.synchronize()

    def one_launch():
        sw.raw.zero_()
        sw.bip_raw.zero_()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        sw.add()
        ev[1].record()
        sw.add_bipartite()
        ev[2].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])

    def per_bin_loop():
        for idx in loop:
            idx.raw.zero_()
            idx.bip_raw.zero_()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        for idx, b in zip(loop, res.bins):
            idx.add(*res.ranges[b])
        ev[1].record()
        for idx, b in zip(loop, res.bins):
            idx.add_bipartite(*res.ranges[b])
        ev[2].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])

    one_launch(), per_bin_loop()  # warm-up
    times = {"one_launch": [], "per_bin_loop": []}
    for r in range(args.reps):  # alternating, the order swapped every repetition
        for name in (("one_launch", "per_bin_loop") if r % 2 == 0 else ("per_bin_loop", "one_launch")):
            times[name].append((one_launch if name == "one_launch" else per_bin_loop)())
    result["hist_ms"] = {k: sorted(t[0] for t in v) for k, v in times.items()}
    result["bipartite_ms"] = {k: sorted(t[1] for t in v) for k, v in times.items()}

    # bit-identity of every bin's histograms (both sides hold exactly one pass now)
    raw, bip_raw = sw.raw.view(-1, HIST_SIZE), sw.bip_raw.view(-1, BIP_SIZE)
    mismatched = []
    for s, idx in enumerate(loop):
        same = torch.equal(raw[s], idx.raw) and torch.equal(bip_raw[s], idx.bip_raw) and \
            torch.equal(sw.hist[s], idx.hist) and torch.equal(sw.bip[s], idx.bip)
        idx._hist = idx._bip = None
        if not same:
            mismatched.append(names[s])
    result["bins_bit_identical"] = len(loop) - len(mismatched)
    result["bins_mismatched"] = mismatched
    result["increments"] = int(sw.raw.long().sum()) + int(sw.bip_raw.long().sum())
    del loop
    torch.cuda.empty_cache()

    # candidates of all bins
    sw._hist = sw._bip = None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sw.hist, sw.bip
    torch.cuda.synchronize()
    result["finalize_ms"] = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    df = sw.candidates(min_mean=args.min_mean, min_mod=args.min_mod)
    result["candidates_s"] = time.perf_counter() - t0
    result["candidate_rows"] = len(df)
    result["candidate_rows_bipartite"] = int((df["motif"].str.len() > MAX_K).sum())
    scratch = 8 << 30
    chunk = max(1, scratch // table_scratch_bytes(MAX_K))
    n = len(names)
    result["bytes"] = {
        "raw_iupac": n * HIST_SIZE * 4, "raw_bipartite": n * BIP_SIZE * 4,
        "finished_iupac": n * HIST_SIZE * 4, "finished_bipartite": n * BIP_SIZE * 4,
        "candidate_scratch": chunk * table_scratch_bytes(MAX_K), "candidate_records": len(df) * 16,
        "per_bin_k8_table_unfused": 15 ** 7 * 2 * 4,
    }

    # planted-motif recovery
    keys = set(zip(df["bin"], df["motif"], df["mod_position"]))
    per_bin, found, total, elsewhere = {}, 0, 0, {}
    for b, name in zip(res.bins, names):
        rows = []
        for regex, mp, mt in plan["planted"][b]:
            motif = iupac(regex)
            if mt != "a" or not sweep_shape(motif):
                continue
            hit = (name, motif, mp) in keys
            rows.append([motif, mp, hit])
            found += hit
            total += 1
        per_bin[name] = rows
    for regex, mp in synth.PLANT_POOL["a"]:
        motif = iupac(regex)
        planted_in = {f"bin_{b}" for b in res.bins if any(r == regex and t == "a" for r, _, t in plan["planted"][b])}
        elsewhere[f"{motif}@{mp}"] = {"planted_bins": len(planted_in),
                                      "found_in_planted": sum((x, motif, mp) in keys for x in planted_in),
                                      "found_elsewhere": sorted(x for x in names
                                                                if x not in planted_in and (x, motif, mp) in keys)}
    result["planted_found"] = f"{found}/{total}"
    result["planted_by_motif"] = elsewhere
    result["planted_per_bin"] = per_bin
    text = json.dumps(result)
    print(json.dumps({k: v for k, v in result.items() if k != "planted_per_bin"}, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
