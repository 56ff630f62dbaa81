"""bench.py's reference arm runs on the host CPU, so its JSON contract can be checked without a GPU: the keys the driver
reads, the `impl` tag, a zero-copy `e2e` that repeats the line's own value and a `cpu_baseline` that says what was timed
(oracle/_ref = the reference's own modules when the build container copied them, else the oracle port)."""
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-batch", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "FNO2d train samples/sec" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["vs_baseline"] is None                      # BASELINE.md publishes no number for this metric
    assert d["config"]["baseline_config"] == 1 and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "batch 2" in cb["sample"]


def _load_bench():
    spec = importlib.util.spec_from_file_location("_bench", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_cap_and_fixed_sample(tmp_path):
    """Above the cap every array keeps the same seeded share of its elements; complex tensors become (re, im) pairs."""
    bench = _load_bench()
    g = torch.Generator().manual_seed(1)
    arrays = {"loss": torch.tensor([0.5, 0.25]), "big": torch.randn(4, 1000, 1000, 2, generator=g, dtype=torch.cfloat),
              "wide": torch.randn(3, 1000, 1000, generator=g, dtype=torch.float64), "count": torch.tensor(7)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["big.npy", "count.npy", "loss.npy", "wide.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64_000_000
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert np.array_equal(a[f], np.load(tmp_path / "b" / f))
    assert a["big.npy"].dtype == np.float32 and a["wide.npy"].dtype == np.float64 and a["count.npy"].dtype == np.float32
    np.testing.assert_array_equal(a["loss.npy"], [0.5, 0.25])
    assert 0 < a["big.npy"].size < 4 * 1000 * 1000 * 2 * 2
    assert np.isin(a["wide.npy"], arrays["wide"].numpy()).all()


def test_reference_arm_joint_step_dumps_outputs(tmp_path):
    """The config-2 reference arm runs with or without oracle/_ref (the port covers the two-head model) and dumps the
    last CPU step: its loss and every parameter of both heads."""
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--config", "2", "--steps", "1",
                          "--warmup", "0", "--cpu-batch", "1", "--dump-outputs", str(tmp_path / "d")],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["config"]["baseline_config"] == 2 and d["cpu_baseline"]["kind"] in ("reference", "port")
    got = {p.name: np.load(p) for p in (tmp_path / "d").iterdir()}
    assert {"loss.npy", "param.fc2_primary.weight.npy", "param.fc2_auxiliary.weight.npy",
            "param.conv0.weights1.npy"} <= set(got)
    assert got["param.conv0.weights1.npy"].shape == (20, 20, 12, 12, 2)
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in got.values())
    assert 0 < float(got["loss.npy"]) < 10


@pytest.mark.gpu
def test_dump_outputs_reproducible_and_follow_steps(tmp_path):
    """Same arguments -> same inputs, so two runs agree to fp32 rounding; one more timed step changes what is dumped."""
    def run(steps, name):
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", str(steps), "--warmup", "3", "--batch", "8",
                              "--no-e2e", "--no-cpu-baseline", "--no-torch-gpu", "--dump-outputs", str(tmp_path / name)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
        return {p.name: np.load(p) for p in (tmp_path / name).iterdir()}

    a, b, c = run(2, "a"), run(2, "b"), run(3, "c")
    assert "loss.npy" in a and "param.conv0.weights1.npy" in a and sorted(a) == sorted(b) == sorted(c)
    for f in a:
        assert a[f].dtype in (np.float32, np.float64)
        np.testing.assert_allclose(a[f], b[f], rtol=1e-5, atol=1e-6)
    assert not np.allclose(a["param.conv0.weights1.npy"], c["param.conv0.weights1.npy"], rtol=1e-7, atol=0)
