#!/usr/bin/env python
"""Degenerate bipartite sweep at the cfg3 shape (development tool): bins of the cfg3 generator (synth.cfg3_plan,
built on the device by bench.Resident), mod type 'a', with this script's own plan that plants the Type I motifs
GAA......[AG]TCG (EcoR124I), AAC......GT[AG]C (StySPI) and TCA.......[AG]TTC (EcoDXXI) into three of every four bins
(synth.PLANT_POOL, which bench.py's workload comes from, is left alone).

  * device time and bytes of each phase: the bipartite histogram pass, its finalisation, and the slice / 4 -> 14
    expansion / fused filter passes of one chunk of bins over all 140 (gap, shape, modified position) groups;
  * BinSweep.candidates(bipartite_letters="IUPAC") and the default ACGT run: wall time (device + host frame) and rows;
  * per planted degenerate motif: the bins it was planted in where it is a candidate, and the bins where it was not
    planted but is a candidate.

    python tools/bip_iupac_bench.py [--bins 100] [--bin-bp 5000000] [--json out.json]
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
import bench  # noqa: E402  (Resident: bins of the cfg3 generator on the device)
from nanomotif_b200 import synth  # noqa: E402
from nanomotif_b200._lib import check, lib, ptr  # noqa: E402
from nanomotif_b200.api import MultiBinScorer  # noqa: E402
from nanomotif_b200.sweep import BIP_SIZE, MAX_K, BinSweep, bip_iupac_scratch_bytes  # noqa: E402

PLANTED = (("GAA......[AG]TCG", 2), ("AAC......GT[AG]C", 1), ("TCA.......[AG]TTC", 2))
SETS = {"AG": "R", "CT": "Y", "AT": "W", "CG": "S", "GT": "K", "AC": "M"}
SHAPES = ((3, 3), (3, 4), (4, 3), (4, 4))


def iupac(regex: str) -> str:
    toks = re.findall(r"\[[^\]]*\]|.", regex)
    return "".join("N" if t == "." else SETS["".join(sorted(t[1:-1]))] if t.startswith("[") else t for t in toks)


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, power = (out[0].split(", ") + ["?"])[:2] if out else (torch.cuda.get_device_name(0), "?")
    return {"gpu": name, "power_limit": power}


def timed(fn):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1])


def phase_passes(sw, ns, min_mean, min_mod):
    """Device time (ms) and bytes of the slice, expansion and fused filter passes of the first `ns` bins over every
    (gap, shape, modified position) group, each kind summed over the groups; the same launches candidates() makes.
    The buffers are allocated outside the timed windows, so the passes are launched here rather than through
    sweep._expand."""
    d = sw.asm.device
    canon = {"A": 0, "T": 1, "G": 2, "C": 3}[sw.canonical]
    ms = {"slice": 0.0, "expand": 0.0, "filter": 0.0}
    nbytes = {"slice": 0, "expand": 0, "filter": 0}
    n_out = torch.zeros(1, dtype=torch.int64, device=d)
    hits = 0
    for g in range(4, 9):
        for a, b in SHAPES:
            n = a + b - 1
            for o in range(a + b):
                mp = o if o < a else o + g
                tab = [torch.empty(ns * 4 ** n, dtype=torch.int32, device=d) for _ in (0, 1)]

                def run_slice():
                    for cls, t in enumerate(tab):
                        check(lib.nmb_sweep_bip_iupac_slice(ptr(sw.bip), ns, a, g, b, mp, cls, canon, ptr(t), None))

                ms["slice"] += timed(run_slice)
                nbytes["slice"] += 2 * ns * 4 ** n * 4 * 2  # gathered read + write, two classes
                for step in range(n - 1):
                    outer, inner = ns * 4 ** (n - 1 - step), 14 ** step
                    nxt = [torch.empty(outer * 14 * inner, dtype=torch.int32, device=d) for _ in (0, 1)]

                    def run_expand():
                        for t, e in zip(tab, nxt):
                            check(lib.nmb_sweep_bip_iupac_expand(ptr(t), ptr(e), outer, inner, None))

                    ms["expand"] += timed(run_expand)
                    nbytes["expand"] += 2 * outer * (4 + 14) * inner * 4
                    tab = nxt

                def run_filter():
                    check(lib.nmb_sweep_bip_iupac_expand_filter(ptr(tab[0]), ptr(tab[1]), ns, 14 ** (n - 1), min_mean,
                                                                min_mod, 0, None, 0, ptr(n_out), None))

                ms["filter"] += timed(run_filter)
                nbytes["filter"] += 2 * ns * 4 * 14 ** (n - 1) * 4  # records not counted (count-only run)
                hits += int(n_out.item())
                del tab
    return ms, nbytes, hits


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bins", type=int, default=100)
    ap.add_argument("--bin-bp", type=int, default=5_000_000)
    ap.add_argument("--min-mean", type=float, default=0.7)
    ap.add_argument("--min-mod", type=int, default=50)
    ap.add_argument("--json", default=None, help="also write the result here")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    result = {**gpu_info(), "bins": args.bins, "bin_bp": args.bin_bp, "mod_type": "a", "min_mean": args.min_mean,
              "min_mod": args.min_mod}
    print(json.dumps(result), flush=True)

    t0 = time.perf_counter()
    plan = synth.cfg3_plan(args.bins, args.bin_bp)
    plan["planted"] = [tuple(p) + (((PLANTED[b % 4] + ("a",)),) if b % 4 < 3 else ()) for b, p in enumerate(plan["planted"])]
    res = bench.Resident(synth, plan, range(args.bins), dev)
    names = [f"bin_{b}" for b in res.bins]
    scorer = MultiBinScorer.from_device(res.asm, res.pile, {f"bin_{b}": res.ranges[b] for b in res.bins},
                                        bench.MOD_TYPES)
    result["assembly_bp"] = int(res.asm.total_bp)
    result["setup_s"] = round(time.perf_counter() - t0, 1)

    sw = BinSweep(scorer, "a")
    sw.bip_raw.zero_()
    timed(sw.add_bipartite)  # warm-up
    sw.bip_raw.zero_()
    result["bipartite_hist_ms"] = timed(sw.add_bipartite)
    result["finalize_ms"] = timed(lambda: sw.bip)
    n = len(names)
    chunk = min(n, max(1, (8 << 30) // bip_iupac_scratch_bytes()))  # candidates()' default scratch_bytes
    phase_passes(sw, 1, args.min_mean, args.min_mod)  # warm-up
    ms, nbytes, hits = phase_passes(sw, chunk, args.min_mean, args.min_mod)
    result["chunk_bins"] = chunk
    result["chunk_phase_ms"] = ms
    result["chunk_phase_bytes"] = nbytes
    result["chunk_phase_GBps"] = {k: nbytes[k] / ms[k] / 1e6 for k in ms}
    result["chunk_hits"] = hits
    result["bytes"] = {"raw_bipartite": n * BIP_SIZE * 4, "finished_bipartite": n * BIP_SIZE * 4,
                       "iupac_scratch_per_bin": bip_iupac_scratch_bytes(),
                       "iupac_scratch_chunk": chunk * bip_iupac_scratch_bytes()}

    for letters in ("ACGT", "IUPAC"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        df = sw.candidates(min_mean=args.min_mean, min_mod=args.min_mod, bipartite_letters=letters)
        result[f"candidates_{letters}_s"] = time.perf_counter() - t0
        result[f"candidate_rows_{letters}"] = len(df)
        result[f"candidate_rows_{letters}_bipartite"] = int((df["motif"].str.len() > MAX_K).sum())
        if letters == "ACGT":
            del df
    result["bytes"]["candidate_records_IUPAC"] = len(df) * 16

    keys = set(zip(df["bin"], df["motif"], df["mod_position"]))
    found = {}
    for j, (regex, mp) in enumerate(PLANTED):
        motif = iupac(regex)
        planted_in = {f"bin_{b}" for b in res.bins if b % 4 == j}
        found[f"{motif}@{mp}"] = {"planted_bins": len(planted_in),
                                  "found_in_planted": sum((x, motif, mp) in keys for x in planted_in),
                                  "found_elsewhere": sorted(x for x in names if x not in planted_in and (x, motif, mp) in keys)}
    result["planted"] = found
    text = json.dumps(result)
    print(json.dumps(result, indent=1))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
