#!/usr/bin/env python
"""bench.py -- motif x contig-bp scored / second on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

The inputs are seeded: two runs with the same arguments score the same data, so the counts that --dump-outputs
writes can be compared output for output between two builds.

Workload (config.workload = "cfg3"): BASELINE.json configs[2], the synthetic metagenome of SURVEY.md 8d --
300 bins x 5 Mbp = 1.5 Gbp in ~23 k contigs, per-bin GC in U(0.3, 0.7), 1-5 planted motifs per bin, a depth-30
modkit-style pileup for 6mA / 5mC / 4mC (2.35e9 rows).  It is the largest single-GPU configuration (2.6 GB of
packed sequence + class planes); cfg2 (one 4.6 Mbp contig), the M = 1 streaming pass and the cfg5 sweep are
sub-objects of the same line.

One job per (bin, mod type) = 900 jobs, each with a SEARCH-SHAPED motif list: 64 expansion rounds of the <= 4
children of one parent (find_motifs_bin.py:1116-1145), ~225 motifs per job.  One STEP scores every job's whole list
over the bin's contigs, both strands, in the schedule a lock-step search driver produces -- 64 frontier rounds,
one scan launch per round with 3-4 motifs per job.  `regimes` reports the same work list scheduled as 64 x 4, 8 x 32
and 1 x 256 motifs per job and launch.

  value   device-timed throughput, inputs resident in HBM (packed contigs, class planes, motif records, job tables)
  e2e     the same metric through the drop-in boundary from HOST data, nothing hoisted: a reference-shaped pileup
          table (Arrow columns contig: str, position: i64, strand: str, mod_type: str, fraction_mod: f64 -- what
          find_motifs_bin.py:399-427 hands to workers) and {bin: {contig: str}} go into nmb.MultiBinScorer /
          sharding.ShardedMultiBinScorer, then the 64 frontier rounds run through score_batch with the counts read
          back to the host every round.  Timed region = table -> device, name resolution, packing, class planes,
          scans, D2H.  Run on a bounded sample of the bins (host memory); the sample is stated.
  roofline  the scan kernel against the measured HBM copy bandwidth, ALGORITHMIC bytes = 0.75 B per motif*bp
          (SURVEY 8d).  With M motifs per tile visit the tile is re-used from shared memory, so DRAM traffic is far
          below the algorithmic bytes and `frac` can exceed 1 (the kernel is then bound by the integer pipes);
          `stream` is the M = 1 pass where the same kernel is genuinely HBM-bound.
  cpu_baseline  the reference's own regex + np.isin path (oracle/cpu_baseline.py) on the host cores on a bounded
          sample of the SAME (bin, motif) list; its counts are also compared with the GPU's (parity inside the bench).

N > 1 (torchrun): STRONG scaling of the same 300 bins through the product sharding path: sharding.plan_shards keeps
bins whole, every rank packs and scores only its own bins, and the per-round count tensor is summed with one NCCL
all-reduce (the only data-path collective, SURVEY 8e) that overlaps the next round's scan.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True  # the tree may be read-only: the bench leaves no bytecode cache in it
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "motif x contig-bp scored/sec"
UNIT = "motif*bp/s"
ALG_BYTES_PER_UNIT = 0.75  # SURVEY.md 8d: 2-bit sequence L/4 B + four 1-bit class planes L/2 B
MOD_TYPES = ("a", "m", "21839")
N_BINS, BIN_BP, SWEEP_EXTRA_BINS = 300, 5_000_000, 100
ROUNDS, WIDTH = 64, 4
LOW, HIGH = 0.3, 0.7


_JSON_FD = None


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def load_synth():
    """nanomotif_b200/synth.py loaded BY PATH: the generators are plain numpy / torch, and the reference arm must
    not import the package (which dlopens libnmb200.so)."""
    spec = importlib.util.spec_from_file_location("_nmb_synth", os.path.join(ROOT, "nanomotif_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def recorded_traffic(kernel: str):
    """Per-launch dram bytes of a kernel from the committed ncu --set full summaries (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def config_dict(plan, n_jobs, motifs_per_job, e2e_bins):
    return {"workload": "cfg3: synthetic metagenome (BASELINE.json configs[2], SURVEY 8d)",
            "bins": N_BINS, "assembly_bp": int(plan["lengths"][plan["bin_of"] < N_BINS].sum()),
            "contigs": int((plan["bin_of"] < N_BINS).sum()), "mod_types": list(MOD_TYPES), "pileup_depth": plan["depth"],
            "jobs": n_jobs, "motifs_per_job": motifs_per_job,
            "motif_list": f"search-shaped: {ROUNDS} expansion rounds of the <= {WIDTH} children of one parent per "
                          "(bin, mod type), seeded (nanomotif_b200.synth.frontier_worklist)",
            "schedule": f"{ROUNDS} frontier rounds per step, one scan launch per round",
            "thresholds": [LOW, HIGH], "e2e_sample_bins": e2e_bins,
            "l2": "inputs larger than L2: every launch streams its bins' tile records (2.6 GB per pass over all jobs)"}


def job_worklists(synth, bins):
    """{(bin, mod type index): [[(motif, mod_pos)] per round]} for the given bins."""
    return {(b, mt): synth.frontier_worklist(b * len(MOD_TYPES) + mt, synth.CANONICAL[name], ROUNDS, WIDTH)
            for b in bins for mt, name in enumerate(MOD_TYPES)}


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampling during the timed region (rank 0 samples every GPU of the job)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, indices):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                 ",".join(str(i) for i in indices)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons, loaded = {}, [], set(), 0
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in out.strip().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.setdefault(int(parts[0]), []).append(float(parts[1]))
                mx.append(float(parts[2]))
                loaded += float(parts[4]) >= 50.0
            except ValueError:
                continue
            for name, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        per_gpu = {g: float(np.median(v)) for g, v in sorted(sm.items())}
        out = {"sm_mhz": min(per_gpu.values()) if per_gpu else None, "sm_max_mhz": float(max(mx)) if mx else None,
               "samples": sum(len(v) for v in sm.values()), "samples_under_load": int(loaded), "reasons": sorted(reasons)}
        if len(per_gpu) > 1:
            out["per_gpu_sm_mhz"] = per_gpu  # the step time is the max over ranks: the slowest GPU sets it
        return out


# ---------------------------------------------------------------------------------------------
# host-generated sample bins (shared by the e2e leg and the CPU legs)
# ---------------------------------------------------------------------------------------------
_POOL_G = {}


def _gen_bin(b):
    return b, _POOL_G["synth"].cfg3_bin_host(_POOL_G["plan"], b)


def host_bins(synth, plan, bins, workers=None):
    """{b: cfg3_bin_host(plan, b)} for the given bins, generated in a fork pool (numpy, ~3 s per bin and core).
    Must run before CUDA is initialised in this process."""
    bins = list(bins)
    if not bins:
        return {}
    import multiprocessing as mp

    _POOL_G.update(synth=synth, plan=plan)
    workers = min(len(bins), workers or os.cpu_count() or 1)
    if workers <= 1:
        return dict(_gen_bin(b) for b in bins)
    with mp.get_context("fork").Pool(workers) as pool:
        return dict(pool.map(_gen_bin, bins, chunksize=1))


def arrow_table(plan, hb: dict):
    """The reference-shaped pileup table of some host-generated bins: Arrow columns as a polars frame holds them
    (String -> large_utf8 buffers).  Built outside the timed region: it is the INPUT of the e2e leg."""
    import pyarrow as pa

    names, contig, cols = [], [], {k: [] for k in ("position", "strand", "mod_type", "fraction_mod", "Nvalid_cov")}
    base = 0
    for b, d in hb.items():
        lo, hi = plan["ranges"][b]
        names += [f"contig_{i}" for i in range(lo, hi)]
        contig.append(d["contig"].astype(np.int32) + base)
        base += hi - lo
        for k in cols:
            cols[k].append(d[k])
    cat = {k: np.concatenate(v) for k, v in cols.items()}
    dict_col = lambda codes, values: pa.DictionaryArray.from_arrays(pa.array(codes), pa.array(values)).cast(pa.large_string())
    return pa.table({
        "contig": dict_col(np.concatenate(contig), names),
        "position": pa.array(cat["position"], type=pa.int64()),
        "mod_type": dict_col(cat["mod_type"].astype(np.int8), list(MOD_TYPES)),
        "strand": dict_col(cat["strand"].astype(np.int8), ["+", "-"]),
        "fraction_mod": pa.array(cat["fraction_mod"], type=pa.float64()),
        "Nvalid_cov": pa.array(cat["Nvalid_cov"], type=pa.int64()),
    })


def table_bytes(table, columns=("contig", "position", "mod_type", "strand", "fraction_mod")) -> int:
    return int(sum(table.column(c).nbytes for c in columns))


def contig_strings(plan, b, d) -> dict:
    lo, hi = plan["ranges"][b]
    starts = np.concatenate([[0], np.cumsum(d["lengths"])[:-1]])
    return {f"contig_{lo + i}": d["ascii"][s:s + n].tobytes().decode("ascii")
            for i, (s, n) in enumerate(zip(starts.tolist(), d["lengths"].tolist()))}


# ---------------------------------------------------------------------------------------------
# CPU legs
# ---------------------------------------------------------------------------------------------
def cpu_work(worklists, bins, plan):
    """The (bin, motif, mod_pos, mod type) tasks of the sample bins in a seeded random order, and bp per bin."""
    tasks = [(b, m, p, mt) for (b, mt), rounds in sorted(worklists.items()) if b in bins for kids in rounds for m, p in kids]
    order = np.random.default_rng(7).permutation(len(tasks))
    bp = {b: int(plan["lengths"][plan["ranges"][b][0]:plan["ranges"][b][1]].sum()) for b in bins}
    return [tasks[i] for i in order], bp


def make_cpu_pool(hb, workers=None):
    from oracle.cpu_baseline import CpuPool, best_kind, presplit_bin

    bins = {b: presplit_bin(d["ascii"], d["lengths"], d["contig"], d["position"], d["strand"], d["mod_type"],
                            d["fraction_mod"], len(MOD_TYPES), LOW, HIGH) for b, d in hb.items()}
    return CpuPool(bins=bins, workers=workers, kind=best_kind())


def cpu_leg(hb, worklists, plan, target_s: float, gpu_counts=None):
    pool = make_cpu_pool(hb)
    try:
        tasks, bp = cpu_work(worklists, set(hb), plan)
        _, t_probe = pool.run(tasks[:pool.workers])
        n = int(max(pool.workers, min(len(tasks), pool.workers * max(1.0, target_s / max(t_probe, 1e-3)))))
        res, secs = pool.run(tasks[:n])
    finally:
        pool.close()
    units = sum(bp[t[0]] for t in tasks[:n])
    out = {"value": units / secs, "unit": UNIT, "cores": pool.workers, "kind": pool.kind,
           "sample": f"{n} of {len(tasks)} (bin, motif, mod type) tasks of the e2e sample bins {sorted(hb)} "
                     f"(each = one motif over the ~{BIN_BP // 1000000} Mbp of a bin, both strands), {secs:.1f} s; "
                     "regex.finditer(overlapped) + np.isin exactly as nanomotif/utils.py:44-67 and "
                     "find_motifs_bin.py:1234-1331, pileup pre-split once (favours the CPU)",
           "seconds": secs}
    if gpu_counts is not None:  # parity inside the bench: the CPU counts of the sample against the GPU's
        bad = [(t, r, gpu_counts[t]) for t, r in zip(tasks[:n], res) if tuple(gpu_counts[t]) != tuple(r)]
        out["parity_checked"] = n
        out["parity_mismatches"] = len(bad)
        if bad:
            raise AssertionError(f"GPU counts differ from the CPU path: {bad[:3]}")
    return out


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores; no repo kernel, no package import."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    synth = load_synth()
    plan = synth.cfg3_plan(N_BINS + SWEEP_EXTRA_BINS, BIN_BP)
    bins = list(range(args.ref_bins))
    hb = host_bins(synth, plan, bins)
    worklists = job_worklists(synth, bins)
    pool = make_cpu_pool(hb)
    tasks, bp = cpu_work(worklists, set(bins), plan)
    per_step = args.ref_tasks_per_core * pool.workers  # bounded sample per step
    try:
        k, total, units = 0, 0.0, 0
        for i in range(args.warmup + args.steps):
            chunk = tasks[k:k + per_step]
            _, s = pool.run(chunk)
            if i >= args.warmup:
                total += s
                units += sum(bp[t[0]] for t in chunk)
            k = (k + per_step) % max(1, len(tasks) - per_step)
    finally:
        pool.close()
    value = units / total
    n_jobs = N_BINS * len(MOD_TYPES)
    mpj = float(np.mean([sum(len(k) for k in r) for r in worklists.values()]))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "python str + regex matches / int64 positions", "data": "synthetic",
            "config": config_dict(plan, n_jobs, mpj, list(range(args.e2e_bins))),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": pool.workers, "kind": pool.kind,
                             "sample": f"{per_step} (bin, motif, mod type) tasks per step from bins {bins} of the cfg3 "
                                       "work list, each one motif over a ~5 Mbp bin, both strands"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------------------------
# resident state of the value leg
# ---------------------------------------------------------------------------------------------
class Resident:
    """The rank's bins on the device: packed contigs, class planes of the three mod types, and the work list as
    resident motif records + job tables for the three schedules."""

    def __init__(self, synth, plan, my_bins, device):
        import torch

        from nanomotif_b200.device import DeviceAssembly, DevicePileup

        self.device, self.plan = device, plan
        self.bins = list(my_bins)
        lens, names, self.ranges = [], [], {}
        ascii_parts = []
        for b in self.bins:
            d = synth.cfg3_bin_device(plan, b, device, ascii_only=True)
            lo, hi = plan["ranges"][b]
            self.ranges[b] = (len(names), len(names) + hi - lo)
            names += [f"contig_{i}" for i in range(lo, hi)]
            lens.append(d["lengths"])
            ascii_parts.append(d["ascii"])
        lens = np.concatenate(lens) if lens else np.zeros(0, np.int64)
        off = np.zeros(len(lens), dtype=np.int64)
        off[1:] = np.cumsum(lens)[:-1]
        ascii_d = torch.cat(ascii_parts) if ascii_parts else torch.zeros(1, dtype=torch.uint8, device=device)
        del ascii_parts
        self.asm = DeviceAssembly(names, lens, ascii_d, off, device)
        del ascii_d
        self.pile = DevicePileup(self.asm, len(MOD_TYPES), LOW, HIGH).clear()
        self.n_rows = 0
        for b in self.bins:
            d = synth.cfg3_bin_device(plan, b, device)
            self.pile.add_columns(d["contig"] + self.ranges[b][0], d["position"], d["strand"], d["fraction_mod"],
                                  d["mod_type"], sync=False)
            self.n_rows += int(d["position"].numel())
            del d
        torch.cuda.synchronize(device)
        assert self.pile.duplicate_rows == 0
        self.bin_bp = {b: int(lens[self.ranges[b][0]:self.ranges[b][1]].sum()) for b in self.bins}

    def schedules(self, worklists, job_bins, all_jobs):
        """Resident launches for the schedules 64 x <=4, 8 x <=32 and 1 x all motifs per job.  `all_jobs` is the
        GLOBAL ordered job list (every rank uses the same output row layout, so one all-reduce merges the ranks);
        this rank scans the jobs of `job_bins`."""
        from nanomotif_b200.device import MotifPrograms, PreparedJobs, make_jobs
        from nanomotif_b200.motif import Motif, pack_motifs

        packed = {}  # job -> (packed motif records in round order, round boundaries)
        for key in all_jobs:
            rounds = worklists[key]
            bounds = np.concatenate([[0], np.cumsum([len(k) for k in rounds])])
            if key[0] in job_bins:
                packed[key] = (pack_motifs([Motif(m, p) for kids in rounds for m, p in kids]), bounds)
            else:
                packed[key] = (None, bounds)
        out = {}
        for name, group in (("frontier4", 1), ("batch32", 8), ("batch256", ROUNDS)):
            launches = []
            for r0 in range(0, ROUNDS, group):
                recs, rows, row, m_at = [], [], 0, 0
                for key in all_jobs:
                    p, bounds = packed[key]
                    a, z = int(bounds[r0]), int(bounds[min(ROUNDS, r0 + group)])
                    if p is not None and z > a:
                        rows.append((key, row, m_at, z - a))
                        recs.append(p[a:z])
                        m_at += z - a
                    row += z - a
                jobs = make_jobs(len(rows))
                units = 0
                for j, (key, row0, m0, cnt) in enumerate(rows):
                    b, mt = key
                    cb, ce = self.ranges[b]
                    jobs[j]["motif_begin"], jobs[j]["motif_count"], jobs[j]["modtype"] = m0, cnt, mt
                    jobs[j]["tile_begin"], jobs[j]["tile_count"] = self.asm.tile_span(cb, ce)
                    jobs[j]["contig_begin"], jobs[j]["contig_end"] = cb, ce
                    jobs[j]["group_mode"], jobs[j]["n_groups"], jobs[j]["out_base"] = 0, 1, row0
                    units += cnt * self.bin_bp[b]
                progs = MotifPrograms(np.concatenate(recs), self.device) if recs else None
                launches.append({"progs": progs, "jobs": PreparedJobs(jobs, self.device) if len(rows) else None,
                                 "rows": row, "units": units, "n_motifs": m_at, "n_jobs": len(rows)})
            out[name] = launches
        return out


def run_schedule(res: Resident, launches, outs, world, scan_events=None, pending=None, keep=None):
    """One pass over a schedule: per launch compile the motif records, zero the count tensor, scan, and (N > 1)
    start the all-reduce of the counts, which overlaps the next launch's scan (two count tensors alternate).
    `keep`, one [rows, 4] tensor per launch, replaces the alternating tensors so that every launch's counts remain."""
    import torch.distributed as dist

    from nanomotif_b200.device import scan_count

    pending = pending if pending is not None else [None, None]
    for i, L in enumerate(launches):
        slot = i & 1
        if pending[slot] is not None:
            pending[slot].wait()  # the collective that last used this count tensor
            pending[slot] = None
        out = outs[slot][:L["rows"]] if keep is None else keep[i]
        out.zero_()
        if L["progs"] is not None:
            L["progs"].compile()  # motif records -> scan programs (device kernel)
            if scan_events is not None:
                ev = scan_events.pop()
                ev[0].record()
            scan_count(res.asm, res.pile, L["progs"], L["jobs"], L["rows"], out=out)
            if scan_events is not None:
                ev[1].record()
        if world > 1:
            pending[slot] = dist.all_reduce(out, async_op=True)  # bin-level counts over the ranks (NCCL, int64 sum)
    return pending


def drain(pending):
    for i, w in enumerate(pending):
        if w is not None:
            w.wait()
            pending[i] = None


# ---------------------------------------------------------------------------------------------
# sub-objects
# ---------------------------------------------------------------------------------------------
def stream_leg(res: Resident, reps: int = 5):
    """M = 1: one motif over every contig of the rank's cfg3 bins, one mod type -- the HBM-bound regime."""
    import torch

    import nanomotif_b200 as nmb
    from nanomotif_b200 import _lib
    from nanomotif_b200.device import MotifPrograms, make_jobs, scan_count

    asm, device = res.asm, res.device
    cfg3 = [b for b in res.bins if b < N_BINS]
    cb, ce = res.ranges[cfg3[0]][0], res.ranges[cfg3[-1]][1]
    t0, tn = asm.tile_span(cb, ce)
    bp = int(asm.lengths[cb:ce].sum())
    out = {}
    for name, motif in (("GATC", nmb.Motif("GATC", 1)), ("GRNGAAGY", nmb.Motif("G[AG].GAAG[CT]", 5))):
        progs = MotifPrograms([motif], device)
        jobs = make_jobs(1)
        jobs["motif_count"], jobs["tile_begin"], jobs["tile_count"] = 1, t0, tn
        jobs["contig_begin"], jobs["contig_end"], jobs["n_groups"] = cb, ce, 1
        r = torch.zeros((1, 4), dtype=torch.int64, device=device)
        for _ in range(2):
            scan_count(asm, res.pile, progs, jobs, 1, out=r)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:
            a.record()
            scan_count(asm, res.pile, progs, jobs, 1, out=r)
            b.record()
        torch.cuda.synchronize()
        ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
        out[name] = {"ms": ms, "motif_bp_per_s": bp / (ms * 1e-3), "alg_gbs": ALG_BYTES_PER_UNIT * bp / (ms * 1e-3) / 1e9,
                     "record_gbs": tn * (_lib.SEQ_REC_WORDS + _lib.CLS_REC_WORDS) * 4 / (ms * 1e-3) / 1e9}
    out["assembly_bp"], out["contigs"], out["tiles"] = bp, ce - cb, tn
    return out


def sweep_leg(res: Resident, world, reps: int = 2):
    """cfg5 (BASELINE.json configs[4]): every IUPAC 4-8-mer + the bipartite shapes over the rank's share of the 2 Gbp
    assembly (all 400 bins), mod type 'a': one histogram pass each + one all-reduce of the histograms."""
    import torch
    import torch.distributed as dist

    from nanomotif_b200.sweep import SweepIndex

    ms = {"hist": [], "bipartite": [], "allreduce": []}
    for _ in range(reps):
        index = SweepIndex(res.asm, res.pile, 0)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        index.add()
        ev[1].record()
        index.add_bipartite()
        ev[2].record()
        if world > 1:
            index.all_reduce()
        ev[3].record()
        torch.cuda.synchronize()
        for k, a, b in (("hist", 0, 1), ("bipartite", 1, 2), ("allreduce", 2, 3)):
            ms[k].append(ev[a].elapsed_time(ev[b]))
        n_inc = int(index.raw.long().sum().item())
        del index
    t = torch.tensor([min(ms["hist"]), min(ms["bipartite"]), min(ms["allreduce"])], dtype=torch.float64, device=res.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()], n_inc


def _one_job(make_jobs, asm, modtype, n_motifs):
    j = make_jobs(1)
    j["motif_count"], j["modtype"], j["tile_count"], j["contig_end"], j["n_groups"] = n_motifs, modtype, asm.n_tiles, 1, 1
    return j


def cfg2_leg(synth, device, steps: int = 10):
    """Round-1 headline kept for continuity: one 4.6 Mbp contig (BASELINE.json configs[1]), 3 x 1000 random motifs
    in one launch, inputs resident, 256 MiB L2 flush between steps."""
    import torch

    import nanomotif_b200 as nmb
    from nanomotif_b200.device import DeviceAssembly, DevicePileup, MotifPrograms, PreparedJobs, make_jobs, scan_count
    from nanomotif_b200.motif import pack_motifs

    rng = np.random.default_rng(1)
    seq = synth.random_sequence(rng, 4_600_000, 0.508, 1e-6)
    pile = synth.synth_pileup(seq, rng, depth=100, mod_types=MOD_TYPES)
    mrng = np.random.default_rng(1001)
    work = [(s, p, mt) for mt, name in enumerate(MOD_TYPES) for s, p in synth.random_motifs(mrng, 1000, synth.CANONICAL[name])]
    asm = DeviceAssembly(["contig_0"], [len(seq)], seq, [0], device)
    dp = DevicePileup.from_columns(asm, np.zeros(len(pile["position"]), np.int32), pile["position"], pile["strand"],
                                   pile["fraction_mod"], LOW, HIGH, pile["mod_type"], n_modtypes=len(MOD_TYPES))
    progs = MotifPrograms(pack_motifs([nmb.Motif(s, p) for s, p, _ in work]), device)
    jobs = make_jobs(len(MOD_TYPES))
    for mt in range(len(MOD_TYPES)):
        j = jobs[mt]
        j["motif_begin"], j["motif_count"], j["modtype"] = 1000 * mt, 1000, mt
        j["tile_begin"], j["tile_count"], j["contig_begin"], j["contig_end"] = 0, asm.n_tiles, 0, 1
        j["group_mode"], j["n_groups"], j["out_base"] = 0, 1, 1000 * mt
    prepared = PreparedJobs(jobs, device)
    out = torch.zeros((len(work), 4), dtype=torch.int64, device=device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(3 + steps):
        flush.zero_()
        progs.compile()
        out.zero_()
        if i >= 3:
            evs[i - 3][0].record()
        scan_count(asm, dp, progs, prepared, len(work), out=out)
        if i >= 3:
            evs[i - 3][1].record()
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    units = len(work) * len(seq)
    res = {"workload": "cfg2: one 4.6 Mbp contig, 3 x 1000 random motifs in one launch (round-1 headline)",
           "scan_ms": ms, "value": units / (ms * 1e-3), "alg_frac": ALG_BYTES_PER_UNIT * units / (ms * 1e-3) / 1e9}
    # the motifs the REFERENCE search visited (tests/golden/search_trace*.json, recorded from the real MotifSearcher):
    # every expansion = the children of one parent (graph edges), scored expansion by expansion as the search does
    # (SURVEY 8d cfg 2: "the actual motif sequence visited by the reference search")
    try:
        rounds_t = []
        for name in ("search_trace.json", "search_trace_cfg1.json"):
            with open(os.path.join(ROOT, "tests", "golden", name)) as f:
                tr = json.load(f)
            pad = tr["spec"]["padding"]
            kids = {}
            for parent, child in tr["edges"]:
                kids.setdefault(parent, []).append(child)
            rounds_t += [[nmb.Motif(c, pad) for c in cs] for cs in kids.values()]
        n_visited = sum(len(r) for r in rounds_t)
        one = PreparedJobs(_one_job(make_jobs, asm, 0, n_visited), device)
        all_progs = MotifPrograms(pack_motifs([m for r in rounds_t for m in r]), device)
        per_round = [(MotifPrograms(pack_motifs(r), device), PreparedJobs(_one_job(make_jobs, asm, 0, len(r)), device), len(r))
                     for r in rounds_t]
        out_t = torch.zeros((n_visited, 4), dtype=torch.int64, device=device)

        def timed(fn, reps=5):
            fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        def as_rounds():
            for pr, jb, n in per_round:
                scan_count(asm, dp, pr, jb, n, out=out_t[:n])

        ms_rounds = timed(as_rounds)
        ms_one = timed(lambda: scan_count(asm, dp, all_progs, one, n_visited, out=out_t))
        res["reference_search_trace"] = {
            "motifs": n_visited, "expansions": len(rounds_t),
            "ms_expansion_by_expansion": ms_rounds, "value_expansion_by_expansion": n_visited * len(seq) / (ms_rounds * 1e-3),
            "ms_one_launch": ms_one, "value_one_launch": n_visited * len(seq) / (ms_one * 1e-3),
            "note": "mod type 'a' over the 4.6 Mbp contig; one launch per expansion is launch-latency bound on ONE small bin "
                    "(~70 tiles): the lock-step driver batches the expansions of all bins instead (headline schedule)"}
    except (OSError, KeyError, ValueError) as exc:  # the golden traces are test fixtures; the bench does not depend on them
        res["reference_search_trace"] = {"unavailable": repr(exc)}
    # round-1's end-to-end leg, kept for continuity: the repo's own pre-compacted 7-byte rows (prepared OUTSIDE the
    # timed region, so this is not the boundary number), one pinned block per mod type, copies overlapped with scans
    from nanomotif_b200.device import compact_rows
    from nanomotif_b200.pipeline import HostBlock, blocks_by_modtype, score_host_blocks

    n_rows = len(pile["position"])
    rows = compact_rows(np.zeros(n_rows, np.int32), pile["position"], pile["strand"], pile["fraction_mod"], pile["mod_type"], 1)
    blocks = [HostBlock(*(torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in b[:4]), b.modtypes)
              for b in blocks_by_modtype(rows["position"], rows["flags"], rows["percent_x100"], rows["contig_row_off"],
                                         len(MOD_TYPES))]
    jobs0 = jobs.copy()
    jobs0["tile_count"] = 0  # = every tile of the assembly
    ascii_h = torch.from_numpy(seq.copy()).pin_memory()
    out_h = torch.empty((len(work), 4), dtype=torch.int64).pin_memory()
    packed = progs.packed

    def streamed():
        return score_host_blocks(["contig_0"], [len(seq)], ascii_h, [0], blocks, packed, jobs0, len(packed), low=LOW,
                                 high=HIGH, n_modtypes=len(MOD_TYPES), device=device, reduce_over_ranks=False, out_host=out_h)

    for _ in range(2):
        got = streamed()
    assert torch.equal(got, out.cpu()), "streamed counts differ from the resident path"
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        streamed()
    torch.cuda.synchronize()
    s_ms = (time.perf_counter() - t0) / steps * 1e3
    res["streamed_compact"] = {"value": units / (s_ms * 1e-3), "ms_per_step": s_ms,
                               "h2d_bytes_per_step": len(seq) + 7 * n_rows + packed.nbytes + jobs0.nbytes,
                               "note": "pre-compacted 7-byte rows prepared outside the timed region (round-1 e2e leg)"}
    return res


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the regimes / stream / sweep / cfg2 sub-objects")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--only-stream", action="store_true", help="just the M = 1 streaming pass over cfg3 (profiling)")
    ap.add_argument("--only-sweep", action="store_true", help="just the cfg5 sweep passes (profiling)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--e2e-bins", type=int, default=8, help="bins of the end-to-end sample (host tables)")
    ap.add_argument("--bins", type=int, default=N_BINS, help="cfg3 bins (debug: smaller assemblies)")
    ap.add_argument("--ref-bins", type=int, default=2, help="--impl reference: bins held by the CPU pool")
    ap.add_argument("--ref-tasks-per-core", type=int, default=8, help="--impl reference: tasks per core and step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the counts of the last timed step to DIR/counts.npy: float64 [rows, 4] = n_mod '+', "
                         "n_nomod '+', n_mod '-', n_nomod '-'; rows round by round, within a round the (bin, mod type) "
                         "jobs in order, within a job its motifs of the round in work-list order")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the counts of the b200 path")
    if args.dump_outputs and (args.only_stream or args.only_sweep):
        ap.error("--dump-outputs needs the timed frontier schedule, which --only-stream / --only-sweep skip")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    # stdout carries exactly ONE line (the JSON): anything a library prints there (e.g. "NCCL version ...") goes to stderr
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    affinity = None
    if world > 1:  # one slice of the host cores per rank (contiguous: GPU i and core slice i share a NUMA node on HGX
        try:       # boards), so that the staging threads and pinned slots of a rank stay local to its GPU
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            affinity = cores[local * per:(local + 1) * per] or cores
            os.sched_setaffinity(0, affinity)
        except (AttributeError, OSError):
            affinity = None
    synth = load_synth()
    n_bins = args.bins
    extra = SWEEP_EXTRA_BINS if (n_bins == N_BINS and not args.no_extras) else 0
    plan = synth.cfg3_plan(N_BINS + SWEEP_EXTRA_BINS, BIN_BP)

    # ---- sharding (host logic, before CUDA): the product planner keeps bins whole ----
    from nanomotif_b200 import sharding  # imports the package: fails loudly without libnmb200.so

    def owners(b0, b1):
        sel = (plan["bin_of"] >= b0) & (plan["bin_of"] < b1)
        own = sharding.plan_shards(plan["lengths"][sel], world, plan["bin_of"][sel])
        first = np.array([plan["ranges"][b][0] for b in range(b0, b1)], dtype=np.int64) - plan["ranges"][b0][0]
        return own[first]  # bins stay whole: the owner of a bin = the owner of its first contig

    bin_owner = np.concatenate([owners(0, n_bins), owners(N_BINS, N_BINS + extra)])
    bin_ids = list(range(n_bins)) + list(range(N_BINS, N_BINS + extra))
    my_bins = [b for b, o in zip(bin_ids, bin_owner) if o == rank]
    # the e2e sample: its own shard plan (ShardedMultiBinScorer plans over the bins it is given)
    e2e_bins = list(range(min(args.e2e_bins, n_bins))) if not args.no_e2e else []
    e2e_lengths = [int(n) for b in e2e_bins for n in plan["lengths"][plan["ranges"][b][0]:plan["ranges"][b][1]]]
    e2e_groups = [b for b in e2e_bins for _ in range(*plan["ranges"][b])]
    e2e_owner = sharding.plan_shards(e2e_lengths, world, e2e_groups) if e2e_bins else np.zeros(0, np.int32)
    cpu_on = not args.no_cpu_baseline and world == 1 and rank == 0
    # host data of every sample bin with a contig on this rank (a bin above 1.25 / world of the sample is split)
    host_needed = sorted({b for b, o in zip(e2e_groups, e2e_owner.tolist()) if o == rank})
    t_setup = time.perf_counter()
    hb = host_bins(synth, plan, host_needed, workers=max(1, (os.cpu_count() or 1) // max(1, world)))

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    import nanomotif_b200 as nmb

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    res = Resident(synth, plan, my_bins, device)
    if args.only_stream or args.only_sweep:
        out = stream_leg(res) if args.only_stream else dict(zip(("ms", "increments"), sweep_leg(res, world)))
        if rank == 0:
            emit(out)
        return
    all_jobs = [(b, mt) for b in range(n_bins) for mt in range(len(MOD_TYPES))]
    worklists = job_worklists(synth, range(n_bins))
    sched = res.schedules(worklists, set(b for b in my_bins if b < N_BINS), all_jobs)
    max_rows = max(L["rows"] for ls in sched.values() for L in ls)
    outs = [torch.zeros((max_rows, 4), dtype=torch.int64, device=device) for _ in range(2)]
    total_bp = {b: int(plan["lengths"][plan["ranges"][b][0]:plan["ranges"][b][1]].sum()) for b in range(n_bins)}
    units_per_step = sum(sum(len(k) for k in worklists[(b, mt)]) * total_bp[b] for b, mt in all_jobs)  # whole job
    my_units = sum(L["units"] for L in sched["frontier4"])
    setup_s = time.perf_counter() - t_setup

    # ---- value: resident inputs, device-timed, 64 frontier rounds per step ----
    head = sched["frontier4"]
    pending = [None, None]
    for _ in range(args.warmup):
        run_schedule(res, head, outs, world, None, pending)
    drain(pending)
    barrier()
    sampler = ClockSampler(range(world)) if rank == 0 else None
    n_scans = sum(1 for L in head if L["progs"] is not None)
    step_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    scan_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps * n_scans)]
    scan_ev_all = list(scan_ev)
    keep = None
    if args.dump_outputs:  # the last step scans into one block of rows per launch, so that all of its counts remain
        launch_rows = [L["rows"] for L in head]
        last_counts = torch.zeros((sum(launch_rows), 4), dtype=torch.int64, device=device)
        keep = list(torch.split(last_counts, launch_rows))
    barrier()
    t_wall = time.perf_counter()
    torch.cuda.nvtx.range_push("timed")  # ncu --nvtx --nvtx-include "timed/" profiles exactly the timed region
    for i in range(args.steps):
        step_ev[i][0].record()
        run_schedule(res, head, outs, world, scan_ev, pending, keep if i == args.steps - 1 else None)
        if i == args.steps - 1:
            drain(pending)
        step_ev[i][1].record()
    torch.cuda.nvtx.range_pop()
    barrier()
    t_wall = time.perf_counter() - t_wall
    clocks = sampler.stop() if sampler else None
    dev_ms = max_over_ranks(step_ev[0][0].elapsed_time(step_ev[-1][1]))  # first record to last record, device clock
    scan_ms = float(np.mean([a.elapsed_time(b) for a, b in scan_ev_all])) if scan_ev_all else 0.0
    value = units_per_step * args.steps / (dev_ms * 1e-3)
    if keep is not None and rank == 0:  # after the all-reduce of the last step rank 0 holds the counts of every rank
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "counts.npy"), last_counts.cpu().numpy().astype(np.float64))

    peak, peak_kind = measured_peak_gbs()

    def timed_passes(launches, reps=3):
        run_schedule(res, launches, outs, world, None, pending)
        drain(pending)
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            run_schedule(res, launches, outs, world, None, pending)
        drain(pending)
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b)) / reps

    regimes = {}
    if not args.no_extras:
        for name, launches in sched.items():
            ms = timed_passes(launches)
            regimes[name] = {"launches_per_step": len(launches), "motifs_per_job_and_launch": round(
                float(np.mean([L["n_motifs"] / max(1, L["n_jobs"]) for L in launches])), 2),
                "ms_per_step": ms, "value": units_per_step / (ms * 1e-3),
                "alg_frac": ALG_BYTES_PER_UNIT * units_per_step / world / (ms * 1e-3) / 1e9 / peak}

    # ---- e2e: reference-shaped host table -> boundary -> counts on the host, nothing hoisted ----
    e2e = None
    e2e_counts = {}
    if e2e_bins:
        from nanomotif_b200.sharding import ShardedMultiBinScorer

        table = arrow_table(plan, hb) if hb else None
        bins_arg = {}
        for b in e2e_bins:  # every rank names every bin; contigs of other ranks are given by length only
            lo, hi = plan["ranges"][b]
            bins_arg[f"bin_{b}"] = contig_strings(plan, b, hb[b]) if b in hb else {
                f"contig_{i}": int(plan["lengths"][i]) for i in range(lo, hi)}
        e2e_lists = {k: v for k, v in worklists.items() if k[0] in e2e_bins}
        e2e_units = sum(sum(len(k) for k in rounds) * total_bp[b] for (b, mt), rounds in e2e_lists.items())
        motif_objs = {key: [[nmb.Motif(m, p) for m, p in kids] for kids in rounds] for key, rounds in e2e_lists.items()}
        keys = sorted(e2e_lists)
        # bytes that cross PCIe: the table's Arrow buffers -- with the int64 position column and the three large_utf8
        # offset columns narrowed to int32 inside the staging copy (4 bytes less per row and column) -- + the contigs
        h2d = (table_bytes(table) - 16 * table.num_rows if table is not None else 0) + sum(
            len(s) for b in hb for s in bins_arg[f"bin_{b}"].values())
        d2h = sum(sum(len(k) for k in rounds) for rounds in e2e_lists.values()) * 4 * 8

        def e2e_step(keep=None):
            scorer = ShardedMultiBinScorer(table, bins_arg, MOD_TYPES, LOW, HIGH, rank, world, device)
            ctx = {key: scorer.context(f"bin_{key[0]}", MOD_TYPES[key[1]]) for key in keys}
            for r in range(ROUNDS):  # a lock-step search: every round needs its counts on the host to go on
                got = scorer.score_batch([(ctx[key], motif_objs[key][r]) for key in keys])
                if keep is not None:
                    for key, c in zip(keys, got):
                        for (m, p), row in zip(e2e_lists[key][r], c):
                            keep[(key[0], m, p, key[1])] = (int(row[0]), int(row[1]))

        for _ in range(2):
            e2e_step(e2e_counts)
        e2e_steps = args.steps  # the same number of steps as the device-timed leg
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": e2e_units * e2e_steps / e2e_s, "unit": UNIT,
               "h2d_bytes_per_step": int(max_over_ranks(float(h2d))), "d2h_bytes_per_step": d2h,
               "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
               "sample": f"bins {e2e_bins} of cfg3 ({sum(total_bp[b] for b in e2e_bins)} bp, "
                         f"{int(max_over_ranks(float(table.num_rows if table is not None else 0)))} pileup rows on the "
                         f"largest rank), {len(keys)} jobs x {ROUNDS} rounds",
               "boundary": "ShardedMultiBinScorer(table, {bin: {contig: str}}, mod_types, 0.3, 0.7, rank, world) + "
                           "score_batch per frontier round (MultiBinScorer per rank inside)",
               "table_bytes_per_step": int(max_over_ranks(float(table_bytes(table) if table is not None else 0))),
               "host_format": "pyarrow Table as a polars frame holds it: contig / strand / mod_type large_utf8, position "
                              "int64, fraction_mod float64, pageable memory; contigs as Python str"}

    if rank == 0:
        alg_bytes = ALG_BYTES_PER_UNIT * my_units / max(1, n_scans)  # per scan launch on this rank
        achieved = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms else 0.0
        mpj = float(np.mean([sum(len(k) for k in worklists[j]) for j in all_jobs]))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 bit-planes / int64 counts", "data": "synthetic",
            "config": config_dict(plan, len(all_jobs), mpj, e2e_bins),
            "e2e": e2e,
            "gpu_launches": args.steps * 2 * n_scans,  # compile_motifs_kernel + scan_count_kernel per round
            "roofline": {"bound": "hbm", "kernel": "scan_count_kernel<1,1>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                         "traffic": recorded_traffic("cfg3_frontier4") if world == 1 else None, "launch_ms": scan_ms,
                         "alg_bytes_per_launch": alg_bytes,
                         "motifs_per_job_and_launch": round(
                             float(np.mean([L["n_motifs"] / max(1, L["n_jobs"]) for L in head])), 2),
                         "note": "3-4 motifs per tile visit: DRAM traffic (one 49.7 KB tile record per job and tile) is "
                                 "below the algorithmic bytes; `stream` is the M = 1 HBM-bound pass of the same kernel"},
            "clocks": clocks,
            "wall_s": t_wall, "setup_s": setup_s, "host_cores_per_rank": len(affinity) if affinity else os.cpu_count(),
            "resident": {"bins": len(my_bins), "contigs": res.asm.n_contigs, "bp": res.asm.total_bp,
                         "pileup_rows": res.n_rows, "tiles": res.asm.n_tiles},
        }
        if regimes:
            line["regimes"] = regimes
    if not args.no_extras:
        st = stream_leg(res) if world == 1 else None
        if extra:
            sweep_ms, n_inc = sweep_leg(res, world)
        if rank == 0:
            if st is not None:
                best = st["GATC"]
                line["stream"] = {"workload": "M = 1 motif per launch over the 1.5 Gbp of cfg3, one mod type",
                                  "bound": "hbm", "achieved": best["alg_gbs"], "peak": peak, "unit": "GB/s",
                                  "frac": best["alg_gbs"] / peak, "traffic": recorded_traffic("stream"), "detail": st}
            if extra:
                sweep_bp = int(plan["lengths"].sum())
                alg = 0.75 * sweep_bp / world  # the pass reads the sequence + one mod type's class planes once
                line["sweep"] = {
                    "workload": f"cfg5: all IUPAC 4-8-mers x every modified position + bipartite X{{3,4}}N{{4..8}}Y{{3,4}} "
                                f"over {sweep_bp} bp ({N_BINS + extra} bins), mod type 'a', contig-sharded over {world} GPU(s)",
                    "hist_ms": sweep_ms[0], "bipartite_ms": sweep_ms[1], "allreduce_ms": sweep_ms[2],
                    "roofline": {"bound": "hbm", "kernel": "sweep_hist_kernel", "achieved": alg / (sweep_ms[0] * 1e-3) / 1e9,
                                 "peak": peak, "unit": "GB/s", "frac": alg / (sweep_ms[0] * 1e-3) / 1e9 / peak,
                                 "alg_bytes_per_launch": alg, "traffic": recorded_traffic("sweep_hist")},
                    "equivalent_motifs": 1_450_000_000, "increments_rank0": n_inc}
        if world == 1:
            c2 = cfg2_leg(synth, device)
            c2["alg_frac"] = c2["alg_frac"] / peak
            line["cfg2"] = c2
    if rank == 0:
        if cpu_on and e2e_counts:
            line["cpu_baseline"] = cpu_leg(hb, worklists, plan, args.cpu_seconds, e2e_counts)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
