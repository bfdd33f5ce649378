"""bench.py contract checks.  Without a GPU: the reference arm (`--impl reference`, the C restatement of the reference
env timed on the host cores) prints exactly one JSON line with the keys the driver reads, and names the same metric,
unit and workload as the device arm.  On the GPU: `--dump-outputs` writes the last timed step's outputs, the same ones
on every run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")  # what torchrun exports; the arm must not be starved by it
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    sys.path.insert(0, ROOT)
    import bench

    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT
    assert d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"] == bench.WORKLOADS["A"]["name"]
    # same `config` object as the device arm (VERDICT r1 weak #11: the driver compares them)
    assert d["config"] == bench.workload_config(bench.WORKLOADS["A"], bench.WORKLOADS["A"]["B"], 1)
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["sample"]
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    assert cb["cores"] == cores
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_needed_bytes_accounting():
    """The headline roofline numerator: bytes the incremental algorithm needs per env-step (bench.needed_bytes)."""
    sys.path.insert(0, ROOT)
    import bench

    nb = bench.needed_bytes(6, 6, 4, False, 4.5, 4.5, 1.0)
    assert nb["b_state"] == 1113                                   # SURVEY.md 8(d), config A
    assert nb["read"] == 1113 + 24 and nb["write"] == 206 + 41 + 32 + 30 + 4.5 * 48 + 4.5 * 10 + 32
    full = 8 + 2 * 1113 + (48 * 36 + 18 * 36 + 32 * 6 + 5 * 6 + 41)
    assert full == 4873 and nb["total"] < full                     # never credits bytes the kernel does not write
    assert bench.median([3, 1, 2]) == 2 and bench.median([4, 1, 2, 3]) == 2.5


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly_and_follow_steps(tmp_path):
    def run(name, steps):
        d = tmp_path / name
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "2",
                              "--repeats", "2", "--batch", "512", "--no-cpu-baseline", "--no-policy", "--no-dropin",
                              "--no-train", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert len([l for l in out.stdout.splitlines() if l.strip()]) == 1
        return {f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))}

    a, b, c = run("a", 5), run("b", 5), run("c", 6)
    assert set(a) == {"env_index", "op", "mach", "mfea1", "mach_mask", "reward5", "scaled4", "done", "invalid", "task_fea",
                      "mach_fea", "adj_w", "adj_src", "job_mask", "candidate"}
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    n = len(a["env_index"])
    assert n == 512 and (np.diff(a["env_index"]) > 0).all()
    for k, x in a.items():
        assert x.dtype in (np.float32, np.float64) and len(x) == n, k
        np.testing.assert_array_equal(x, b[k], err_msg=k)
    assert not (a["invalid"] != 0).any()
    assert any(not np.array_equal(a[k], c[k]) for k in ("op", "reward5", "task_fea"))   # two more timed steps
