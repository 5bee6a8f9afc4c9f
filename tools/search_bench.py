#!/usr/bin/env python
"""Lock-step motif search over many bins (scaled-down BASELINE cfg 3) through search.discover: every (bin, mod type)
search advances together, one K2 launch per score round and one K4 launch per expand / remove round (development tool).

    python tools/search_bench.py [--bins 16] [--bin-bp 1000000] [--cpu-bins 1]
    python tools/search_bench.py --cfg3 [--bins 300]
    python -m torch.distributed.run --nproc-per-node N tools/search_bench.py --cfg3 [--json out.json]

--cfg3 runs sharding.discover_local: every rank generates only the cfg3 bins the discovery plan gives it, on its own
GPU, and searches them; one gather joins the rows.  Reported as the maximum over ranks: ingest, setup
(growth.prepare_searches), search (search.run_lockstep) and gather time, the rounds of each kind; the motifs scored per
rank; the SHA-256 of the frame (the same at every GPU count); the card name and power limit.
"""
import argparse
import hashlib
import json
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import nanomotif_b200 as nmb  # noqa: E402
from nanomotif_b200 import growth, search, sharding, synth  # noqa: E402

PLANTED = [("GATC", 1), ("CTGCAG", 4), ("GA[AG]TC", 1), ("GCAC......GTT", 2), ("CAA..[AT]TG", 2), ("TTAA", 3), ("ACC.GT", 0),
           ("GAAG[CT]", 2)]


class Probe:
    """Counts and times the parts of a discover call by wrapping the module functions it calls: the hook calls of
    search.run_lockstep (one per round of a kind that more than one search has pending), the motifs of the score
    rounds, and the wall time (between device synchronises) of run_lockstep, growth.prepare_searches and
    sharding.gather_rows."""

    def __init__(self):
        self.counts = {"score": 0, "expand": 0, "remove": 0, "motifs": 0}
        self.seconds = {"setup": 0.0, "search": 0.0, "gather": 0.0}
        self.windows = 0
        run, prepare, gather = search.run_lockstep, growth.prepare_searches, sharding.gather_rows

        def counting(kind, fn):
            def hook(reqs):
                self.counts[kind] += 1
                if kind == "score":
                    self.counts["motifs"] += sum(len(m) for _, m in reqs)
                return fn(reqs)
            return hook

        def run_counted(searches, batch_score=None, batch_expand=None, batch_remove=None):
            return self._timed("search", run, searches, counting("score", batch_score), counting("expand", batch_expand),
                               counting("remove", batch_remove))

        def prepare_timed(*args, **kw):
            out = self._timed("setup", prepare, *args, **kw)
            self.windows += int(out[0].n_total)
            return out

        search.run_lockstep = run_counted
        growth.prepare_searches = prepare_timed
        sharding.gather_rows = lambda *args, **kw: self._timed("gather", gather, *args, **kw)

    def _timed(self, key, fn, *args, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn(*args, **kw)
        torch.cuda.synchronize()
        self.seconds[key] += time.perf_counter() - t0
        return out


def expansions(m):
    """Concrete strings of a planted motif: the search reports bracket classes as separate motifs."""
    out = [""]
    for t in nmb.motif.tokenize(m):
        out = [o + c for o in out for c in (t[1:-1] if t.startswith("[") else t)]
    return out


def found_by_pair(df) -> dict:
    """{(bin, mod type): set of motif strings} of a discover frame."""
    best = {}
    for b, mt, motif in zip(df["bin"], df["mod_type"], df["motif"]):
        best.setdefault((b, mt), set()).add(motif)
    return best


def build_bin(b, rng, bin_bp, depth):
    contigs, cols = {}, {k: [] for k in ("contig", "position", "strand", "fraction_mod")}
    n = int(rng.integers(2, 6))
    lens = np.maximum(20000, (rng.dirichlet(np.ones(n)) * bin_bp).astype(int))
    planted = [(PLANTED[i][0], PLANTED[i][1], "a") for i in rng.choice(len(PLANTED), size=int(rng.integers(1, 4)), replace=False)]
    for i, L in enumerate(lens):
        seq = synth.random_sequence(rng, int(L), float(rng.uniform(0.35, 0.65)), 2e-5)
        name = f"bin{b}_contig_{i}"
        contigs[name] = seq.tobytes().decode()
        p = synth.synth_pileup(seq, rng, depth=depth, mod_types=("a",), planted=planted)
        cols["contig"].append(np.full(len(p["position"]), name, dtype=object))
        cols["position"].append(p["position"])
        cols["strand"].append(np.where(p["strand"] == 0, "+", "-").astype(object))
        cols["fraction_mod"].append(p["fraction_mod"])
    return contigs, {k: np.concatenate(v) for k, v in cols.items()}, planted


def windows_for(asm, contigs, pile, pad, high):
    strand = (pile["strand"] == "-").astype(np.uint8)
    conf = pile["fraction_mod"] >= high
    ci, pos, st = [], [], []
    for name, seq in contigs.items():
        in_contig = conf & (pile["contig"] == name)
        for s in (0, 1):
            p = pile["position"][in_contig & (strand == s)]
            p = p[(p > pad) & (p < len(seq) - pad)]
            ci.append(np.full(len(p), asm.index[name]))
            pos.append(p)
            st.append(np.full(len(p), s, dtype=np.uint8))
    return growth.DeviceDNAarray.from_positions(asm, np.concatenate(ci), np.concatenate(pos), np.concatenate(st), pad)


def gpu_info(n: int) -> list:
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[:n] if out else [torch.cuda.get_device_name(0)]


def cfg3_scorer(synth_m, plan, bins, dev, mod_types):
    """MultiBinScorer.from_device over cfg3 bins `bins` (generated on `dev`), with the rows the window step needs."""
    from nanomotif_b200.dataload import DeviceRows
    from nanomotif_b200.device import DeviceAssembly, DevicePileup

    low, high = 0.3, 0.7
    names, lens, ranges, parts = [], [], {}, []
    for b in bins:
        d = synth_m.cfg3_bin_device(plan, b, dev, ascii_only=True)
        lo, hi = plan["ranges"][b]
        ranges[f"bin_{b}"] = (len(names), len(names) + hi - lo)
        names += [f"contig_{i}" for i in range(lo, hi)]
        lens.append(d["lengths"])
        parts.append(d["ascii"])
    lens = np.concatenate(lens)
    off = np.zeros(len(lens), dtype=np.int64)
    off[1:] = np.cumsum(lens)[:-1]
    asm = DeviceAssembly(names, lens, torch.cat(parts), off, dev)
    del parts
    pile = DevicePileup(asm, len(mod_types), low, high).clear()
    rows = []
    for b in bins:
        d = synth_m.cfg3_bin_device(plan, b, dev)
        cid = (d["contig"] + ranges[f"bin_{b}"][0]).to(torch.int32)
        pile.add_columns(cid, d["position"], d["strand"], d["fraction_mod"], d["mod_type"], sync=False)
        rows.append(DeviceRows(names, mod_types, dev, contig_id=cid, position=d["position"], strand=d["strand"],
                               mod_type=d["mod_type"], fraction_mod=d["fraction_mod"]))
    torch.cuda.synchronize()
    return nmb.MultiBinScorer.from_device(asm, pile, ranges, mod_types, rows), sum(len(r) for r in rows)


def cfg3_main(args):
    """--cfg3: the lock-step search of EVERY (bin, mod type) of the cfg3 metagenome (bench.py's generator: 300 bins x
    5 Mbp, three mod types, planted motifs per bin), one GPU per rank."""
    import torch.distributed as dist

    import bench

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def gather(x):
        if world == 1:
            return [x]
        out = [None] * world
        dist.all_gather_object(out, x)
        return out

    synth_m = bench.load_synth()
    plan = synth_m.cfg3_plan(bench.N_BINS + bench.SWEEP_EXTRA_BINS, bench.BIN_BP)
    pad, min_kl, thr = 20, 0.05, 1.5
    bins = {f"bin_{b}": {f"contig_{i}": int(plan["lengths"][i]) for i in range(*plan["ranges"][b])} for b in range(args.bins)}
    owner = sharding.discovery_plan(bins, world)
    mine = [b for b in range(args.bins) if owner[f"bin_{b}"] == rank]
    t0 = time.perf_counter()
    local, n_rows = cfg3_scorer(synth_m, plan, mine, dev, bench.MOD_TYPES) if mine else (None, 0)
    t_gen = time.perf_counter() - t0
    asm_bp = local.assembly.total_bp if local is not None else 0
    n_contigs = local.assembly.n_contigs if local is not None else 0
    probe = Probe()
    df = sharding.discover_local(local, bins, bench.MOD_TYPES, rank, world, padding=pad, min_kl=min_kl,
                                 min_motif_score=thr, seed={f"bin_{b}": 1 + b for b in range(args.bins)}, device=dev)
    found = total = 0
    best = found_by_pair(df)
    for b in range(args.bins):
        for motif, _, mt in plan["planted"][b]:
            got = best.get((f"bin_{b}", mt), set())
            total += 1
            found += motif in got or all(e in got for e in expansions(motif))
    per_rank = gather({"bins": len(mine), "bp": int(asm_bp), "contigs": int(n_contigs), "rows": int(n_rows),
                       "ingest_s": t_gen, "windows": probe.windows, "counts": probe.counts, **probe.seconds})
    sha = hashlib.sha256(df.to_csv(index=False).encode()).hexdigest()
    shas = gather(sha)
    assert len(set(shas)) == 1, shas
    if rank == 0:
        top = lambda k: max(r[k] for r in per_rank)
        rounds = {k: max(r["counts"][k] for r in per_rank) for k in ("score", "expand", "remove")}
        motifs = [r["counts"]["motifs"] for r in per_rank]
        n_pairs = args.bins * len(bench.MOD_TYPES)
        print(f"cfg3: {args.bins} bins, {sum(r['bp'] for r in per_rank) / 1e9:.2f} Gbp, "
              f"{sum(r['contigs'] for r in per_rank)} contigs, {sum(r['rows'] for r in per_rank) / 1e9:.2f} G pileup rows "
              f"(device generation + packing + class planes {top('ingest_s'):.1f} s)")
        print(f"windows + background PSSMs of all {n_pairs} searches (growth.prepare_searches, host random.sample stream "
              f"kept) {top('setup'):.1f} s; windows: {sum(r['windows'] for r in per_rank)}")
        print(f"lock-step search of {n_pairs} (bin, mod type) pairs: {top('search'):.1f} s; rounds: score {rounds['score']} "
              f"({sum(motifs)} motifs), expand {rounds['expand']}, remove {rounds['remove']}")
        print(f"planted motifs recovered: {found} / {total}")
        result = {"gpus": gpu_info(world), "world_size": world, "bins": args.bins, "pairs": n_pairs,
                  "bins_per_rank": [r["bins"] for r in per_rank], "bp_per_rank": [r["bp"] for r in per_rank],
                  "ingest_s": round(top("ingest_s"), 3), "setup_s": round(top("setup"), 3),
                  "search_s": round(top("search"), 3), "gather_s": round(top("gather"), 4), "rounds": rounds,
                  "motifs_per_rank": motifs, "frame_rows": len(df), "planted_recovered": [found, total],
                  "frame_sha256": sha}
        print(json.dumps(result), flush=True)
        if args.json:
            os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
            with open(args.json, "w") as f:
                f.write(json.dumps(result) + "\n")
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg3", action="store_true", help="the whole cfg3 metagenome (device-generated), all mod types")
    ap.add_argument("--bins", type=int, default=16)
    ap.add_argument("--bin-bp", type=int, default=1_000_000)
    ap.add_argument("--depth", type=int, default=20)
    ap.add_argument("--cpu-bins", type=int, default=1, help="bins also searched with the CPU oracle backend (slow)")
    ap.add_argument("--check-setup", action="store_true", help="compare the batched setup with the per-bin host-driven one")
    ap.add_argument("--json", default=None, help="--cfg3: rank 0 also writes the result line here")
    args = ap.parse_args()
    if args.cfg3:
        if args.bins == 16:
            args.bins = 300
        return cfg3_main(args)
    pad, low, high, min_kl, thr = 20, 0.3, 0.7, 0.05, 1.5
    rng = np.random.default_rng(5)
    t0 = time.perf_counter()
    bins, piles, truth = {}, [], {}
    for b in range(args.bins):
        contigs, pile, planted = build_bin(b, rng, args.bin_bp, args.depth)
        pile["mod_type"] = np.full(len(pile["position"]), "a", dtype=object)
        bins[f"bin{b}"], truth[f"bin{b}"] = contigs, planted
        piles.append(pile)
    pile = {k: np.concatenate([p[k] for p in piles]) for k in piles[0]}
    import pyarrow as pa

    # the input a polars frame would hold: Arrow columns (built here, outside the timed setup: it is the INPUT)
    table = pa.table({"contig": pa.array(pile["contig"], type=pa.large_string()), "position": pa.array(pile["position"]),
                      "strand": pa.array(pile["strand"], type=pa.large_string()),
                      "mod_type": pa.array(pile["mod_type"], type=pa.large_string()),
                      "fraction_mod": pa.array(pile["fraction_mod"])})
    t_gen = time.perf_counter() - t0
    nmb.MultiBinScorer(table.slice(0, 1000), {"w": {"w": "ACGT" * 100}}, ["a"], low, high)  # CUDA context, caches
    from nanomotif_b200 import device as _D

    _D._stager(torch.device("cuda", torch.cuda.current_device()))  # the pinned staging slots exist once per process
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    multi = nmb.MultiBinScorer(table, bins, ["a"], low, high)
    torch.cuda.synchronize()
    t_ingest = time.perf_counter() - t0
    seeds = {f"bin{b}": 1 + b for b in range(args.bins)}
    if args.check_setup:  # the old per-bin host-driven setup must give the same windows and backgrounds
        pool, pssms, _ = growth.prepare_searches(multi, "a", pad, high, seeds=list(seeds.values()))
        asm = multi.assembly
        for b in range(args.bins):
            random.seed(1 + b)
            w = windows_for(asm, bins[f"bin{b}"], piles[b], pad, high)
            bg = growth.background_pssm(asm, bins[f"bin{b}"], "A", pad)
            assert torch.equal(pool.windows[pool.begin[b]:pool.end[b]], w.windows) and np.array_equal(bg, pssms[b])
    probe = Probe()
    # windows of every bin + every bin's background PSSM, batched on the device (growth.prepare_searches), then the
    # lock-step search of all bins
    df = search.discover(multi, ["a"], padding=pad, min_kl=min_kl, min_motif_score=thr, seed=seeds)
    t_setup = t_ingest + probe.seconds["setup"]
    t_search = probe.seconds["search"]
    counts = probe.counts
    best = found_by_pair(df)
    found = 0
    for b in range(args.bins):
        got = best.get((f"bin{b}", "a"), set())
        found += all(p[0] in got or all(e in got for e in expansions(p[0])) for p in truth[f"bin{b}"])
    total_bp = sum(len(s) for cs in bins.values() for s in cs.values())
    print(f"{args.bins} bins, {total_bp / 1e6:.1f} Mbp, {len(pile['position']) / 1e6:.1f} M pileup rows (host generation {t_gen:.1f} s)")
    print(f"device setup from the Arrow table (ingest {t_ingest:.3f} s + windows / backgrounds of all bins) {t_setup:7.3f} s")
    print(f"lock-step search of {args.bins} (bin, mod type) pairs          {t_search:7.2f} s   rounds: score {counts['score']} "
          f"({counts['motifs']} motifs), expand {counts['expand']}, remove {counts['remove']}")
    print(f"bins whose planted motifs were all recovered: {found} / {args.bins}")
    if args.cpu_bins:
        from search_common import OracleBackend

        t0 = time.perf_counter()
        for b in range(args.cpu_bins):
            spec = dict(padding=pad, high=high, low=low, mod_type="a", random_seed=1 + b)
            be = OracleBackend(bins[f"bin{b}"], piles[b], spec)
            co = search.find_candidates("a", pad, be.bin_pssm, be.arr.shape[0], min_kl=min_kl, score_threshold=thr)
            search.run(co, be)
        t_cpu = (time.perf_counter() - t0) / args.cpu_bins
        print(f"same search with the CPU oracle backend (regex + np.isin, one core): {t_cpu:7.2f} s per bin "
              f"-> {t_cpu * args.bins:.0f} s for {args.bins} bins sequentially; lock-step GPU speed-up {t_cpu * args.bins / t_search:.0f}x")


if __name__ == "__main__":
    main()
