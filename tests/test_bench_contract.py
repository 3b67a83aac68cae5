"""bench.py contract checks.  Without a GPU: the reference arm (CPU oracle on a bounded sample) prints one JSON line
with the documented keys; non-zero ranks of a torchrun launch stay silent; the clock sampler degrades cleanly.
On the GPU: the arrays --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)


def test_reference_arm_json_line():
    p = _run(["--impl", "reference", "--cpu-windows", "4", "--steps", "1", "--warmup", "1"])
    assert p.returncode == 0, p.stderr
    lines = [ln for ln in p.stdout.split("\n") if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "windows/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("C2") and d["config"]["window"] == 120 and d["config"]["shuffles"] == 100


def test_reference_arm_other_ranks_print_nothing():
    p = _run(["--impl", "reference", "--gpus", "2", "--cpu-windows", "4", "--steps", "1", "--warmup", "0"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_clock_sampler_without_gpu():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.start()
    out = s.stop()
    assert "reasons" in out and "sm_mhz" in out


@pytest.mark.gpu
def test_dump_outputs_repeatable(tmp_path):
    """--dump-outputs: float arrays of at most 64 MB in all, the same for two runs with the same arguments; --steps sets
    the timed steps of both arms"""
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        p = _run(["--windows", "3000", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(d)])
        assert p.returncode == 0, p.stderr[-3000:]
        line = json.loads(p.stdout.strip().split("\n")[-1])
        assert line["steps"] == 2 and line["e2e"]["steps"] == 2
        runs.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = runs
    assert sorted(a) == sorted(b) and "scan_mfe_dcal.npy" in a and "e2e_nt_part.npy" in a
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert len(a["scan_mfe_dcal.npy"]) == 3000 and len(a["e2e_window_z.npy"]) == 3000
    assert a["scan_shuffle_dcal.npy"].shape == (len(a["scan_sample_windows.npy"]), 100)
    for f in a:
        assert a[f].dtype in (np.float32, np.float64), f
        assert np.array_equal(a[f], b[f], equal_nan=True), f
