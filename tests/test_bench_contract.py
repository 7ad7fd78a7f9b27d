"""The bench.py contract that can be checked without a GPU: the reference arm (`--impl reference`, which
times the CPU oracle port — the reference itself is Julia and cannot run here) prints ONE well-formed JSON line,
and malformed arguments are refused. On a GPU: what `--dump-outputs` writes."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--config", "C2", "--cpu-sample", "20000"], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["unit"] == "locations/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["vs_baseline"] is None                       # BASELINE.md holds no published number for this metric
    assert d["value"] > 0 and d["steps"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_gpu_arm_fails_loudly_without_a_device():
    """No CPU fallback: on a box without a GPU the product arm must fail, not print a number."""
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline"],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(argv):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *argv], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 2 and "error" in r.stderr
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
@pytest.mark.parametrize("config,targets", [("C2", 65536), ("C3a", 1 << 22)])
def test_dump_outputs_hold_the_last_timed_step(gsk, ctx, tmp_path, config, targets):
    """--dump-outputs: the whole job when it fits in 64 MB, else a sorted, seeded sample of 2^20 targets; either way the
    values are the library's for those targets."""
    import numpy as np
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--config", config, "--targets", str(targets), "--steps", "2",
                        "--warmup", "1", "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 2
    target, mean, var = (np.load(out / f"{n}.npy") for n in ("target", "mean", "variance"))
    assert target.dtype == mean.dtype == var.dtype == np.float64
    assert target.nbytes + mean.nbytes + var.nbytes <= 64 << 20
    t = target.astype(np.int64)
    assert np.array_equal(t, target) and t.size == (targets if 24 * targets <= 64 << 20 else 1 << 20)
    assert (np.diff(t) > 0).all() and t[0] >= 0 and t[-1] < targets
    m, v = ctx.krige(gsk.synth.config_spec(config).with_slab(0, targets))
    assert np.array_equal(mean, m[t], equal_nan=True) and np.array_equal(var, v[t], equal_nan=True)
