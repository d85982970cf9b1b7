"""The bench.py command line.  CPU: the reference arm prints exactly ONE JSON line on stdout with the result keys, whatever
else libraries print (stdout is claimed for the JSON line).  GPU: --dump-outputs writes the last timed step's arrays, the same
from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-users", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "user-seqs/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_bench_declares_the_baseline_metric():
    import ast
    src = open(os.path.join(ROOT, "bench.py")).read()
    ast.parse(src)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "train" in base["metric"] and "user-sequences/s" in src


def _bench_dump(out_dir, steps=2):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--users", "16", "--users-per-pass", "16", "--steps",
                        str(steps), "--warmup", "1", "--no-eval", "--no-variants", "--no-cpu-baseline", "--dump-outputs",
                        str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["steps"] == steps
    return {n: np.load(out_dir / (n + ".npy")) for n in ("loss", "params", "grads")}


@pytest.mark.gpu
def test_dump_outputs_repeat_across_runs(tmp_path):
    """--dump-outputs writes the loss, parameters and gradients of the last timed step; the same arguments give the same
    inputs and dropout masks, and the C2 step has no float atomics, so a second run computes the same arrays bit for bit."""
    a = _bench_dump(tmp_path / "a")
    b = _bench_dump(tmp_path / "b")
    assert a["loss"].dtype == np.float64 and a["loss"].shape == (1,) and np.isfinite(a["loss"]).all()
    for n in ("params", "grads"):
        assert a[n].dtype == np.float32 and a[n].ndim == 1 and a[n].shape == a["params"].shape and np.isfinite(a[n]).all()
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert np.abs(a["grads"]).max() > 0
    for n in ("loss", "params", "grads"):
        assert np.array_equal(a[n], b[n]), n
