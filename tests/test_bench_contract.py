"""bench.py's output contract, checked on CPU through the reference arm (`--impl reference` times the CPU port of the
hot path and needs no GPU): exactly one JSON line on stdout with the keys the driver reads, noise on stderr only."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "windows/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"] and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_our_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: without a CUDA device the product arm exits with an error instead of timing anything."""
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
    assert not [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]


@pytest.mark.parametrize("extra,message", [
    (["--steps", "0"], "--steps must be at least 1"),
    (["--dump-outputs", "unused"], "--dump-outputs writes the outputs of the CUDA path"),
])
def test_invalid_arguments_are_refused(tmp_path, extra, message):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *extra],
                       capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert r.returncode != 0 and message in r.stderr
    assert not r.stdout.strip() and not os.listdir(tmp_path)


def run_bench_dump(steps, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                        "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    """--steps sets the number of timed steps (the launches of the timed region scale with it), and --dump-outputs
    writes what the timed predict returned: float64 arrays under 64 MB in all, identical from run to run, status 0, the
    LML the result line sums, and the oracle's mean / variance for the first and the last window."""
    from corenav_gp_b200 import synthetic as syn
    from oracle import gp_oracle as go
    d1 = run_bench_dump(1, tmp_path / "one")
    d = run_bench_dump(3, tmp_path / "three")
    assert d1["steps"] == 1 and d["steps"] == 3
    assert d1["gpu_launches"] > 0 and d["gpu_launches"] == 3 * d1["gpu_launches"]
    assert d["roofline"]["launches_per_step"] == d1["roofline"]["launches_per_step"]
    names = ["lml.npy", "mean.npy", "status.npy", "var.npy"]
    assert sorted(os.listdir(tmp_path / "three")) == sorted(os.listdir(tmp_path / "one")) == names
    assert sum(os.path.getsize(tmp_path / "three" / f) for f in names) <= 64 << 20
    out = {k: np.load(tmp_path / "three" / f"{k}.npy") for k in ("mean", "var", "lml", "status")}
    for k, a in out.items():
        assert a.dtype == np.float64 and np.array_equal(a, np.load(tmp_path / "one" / f"{k}.npy")), k
    B, M = out["mean"].shape
    assert out["var"].shape == (B, M) and out["lml"].shape == out["status"].shape == (B,)
    assert np.all(out["status"] == 0)
    assert out["lml"].sum() == pytest.approx(d["checks"]["lml_checksum"], rel=1e-12)
    kernel = d["config"]["kernel"]
    x, y = syn.slip_windows(0, B, d["config"]["N"])
    xs = syn.test_grid(x[0], M)
    th = syn.theta_for(kernel)
    e = go.KernelExpr(kernel)
    for b in (0, B - 1):
        inf = go.inference(e, th[:-1], th[-1], x[b], y[b])
        mu, v = go.predict(e, th[:-1], th[-1], x[b], y[b], xs, inf)
        assert np.max(np.abs(out["mean"][b] - mu) / np.maximum(1, np.abs(mu))) < 1e-9
        assert np.max(np.abs(out["var"][b] - v) / np.maximum(1, np.abs(v))) < 1e-9
        assert abs(out["lml"][b] - inf.lml) < 1e-9 * max(1, abs(inf.lml))
