"""bench.py's contract pieces that run without a GPU: the reference arm prints exactly ONE JSON line with the keys
the driver reads and never imports the package (no repo library mapped); the host-side helpers of the e2e leg."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_and_maps_no_repo_library():
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0', "
            "'--ref-bins', '1', '--ref-tasks-per-core', '1']; runpy.run_path('bench.py', run_name='__main__'); "
            "sys.stderr.write('LOADED=' + str(any(m.startswith('nanomotif_b200') for m in sys.modules)) + chr(10)); "
            "sys.stderr.write('MAPPED=' + str('libnmb200' in open('/proc/self/maps').read()) + chr(10))")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1  # anything a library prints goes to stderr
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["unit"] == "motif*bp/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["config"]["workload"].startswith("cfg3") and line["config"]["bins"] == 300
    assert "LOADED=False" in res.stderr and "MAPPED=False" in res.stderr


def test_e2e_host_table_helpers():
    sys.path.insert(0, ROOT)
    import bench

    synth = bench.load_synth()
    plan = synth.cfg3_plan(12, 200_000)
    assert plan["lengths"].sum() >= 12 * 200_000 and len(plan["ranges"]) == 12
    hb = bench.host_bins(synth, plan, [3, 5], workers=2)
    table = bench.arrow_table(plan, hb)
    assert table.num_rows == sum(len(d["position"]) for d in hb.values())
    assert str(table.schema.field("contig").type) == "large_string" and str(table.schema.field("strand").type) == "large_string"
    names = table.column("contig").to_pylist()
    lo, hi = plan["ranges"][3]
    assert names[0] == f"contig_{lo}" and set(table.column("strand").to_pylist()) == {"+", "-"}
    strings = bench.contig_strings(plan, 3, hb[3])
    assert list(strings) == [f"contig_{i}" for i in range(lo, hi)]
    assert [len(s) for s in strings.values()] == hb[3]["lengths"].tolist()
    lists = bench.job_worklists(synth, [3, 5])
    tasks, bp = bench.cpu_work(lists, {3, 5}, plan)
    assert len(tasks) == sum(len(k) for r in lists.values() for k in r) and set(bp) == {3, 5}
    # every motif of a round shares all constrained positions but one with its siblings (a search expansion)
    for rounds in lists.values():
        for kids in rounds:
            assert 1 <= len(kids) <= bench.WIDTH and len({p for _, p in kids} | {len(m) for m, _ in kids}) <= 2 * len(kids)
    assert bench.table_bytes(table) > 40 * table.num_rows


def test_steps_below_one_are_refused():
    res = subprocess.run([sys.executable, "bench.py", "--steps", "0"], capture_output=True, text=True, cwd=ROOT, timeout=120)
    assert res.returncode == 2 and "--steps must be at least 1" in res.stderr


@pytest.mark.gpu
def test_dump_outputs_holds_the_counts_of_the_last_timed_step(tmp_path):
    """--steps sets the timed steps of both timed legs, and --dump-outputs writes the counts of the last one: the
    inputs are seeded, so they do not depend on the number of steps."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    sys.path.insert(0, ROOT)
    import bench

    lists = bench.job_worklists(bench.load_synth(), range(2))
    n_rows = sum(len(kids) for rounds in lists.values() for kids in rounds)
    dumped = []
    for steps in (1, 2):
        out = tmp_path / f"steps{steps}"
        res = subprocess.run([sys.executable, "bench.py", "--bins", "2", "--e2e-bins", "1", "--no-extras",
                              "--no-cpu-baseline", "--steps", str(steps), "--warmup", "0", "--dump-outputs", str(out)],
                             capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout)
        assert line["steps"] == steps and line["e2e"]["steps"] == steps
        assert sorted(os.listdir(out)) == ["counts.npy"]
        counts = np.load(out / "counts.npy")
        assert counts.dtype == np.float64 and counts.shape == (n_rows, 4)
        assert (counts >= 0).all() and (counts == np.round(counts)).all() and counts.sum() > 0
        dumped.append(counts)
    np.testing.assert_array_equal(dumped[0], dumped[1])
