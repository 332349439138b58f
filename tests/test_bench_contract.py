"""bench.py prints ONE JSON line with the keys the driver's contract names (both arms)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(args, timeout=600):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, res.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--model", "tiny", "--steps", "2", "--warmup", "1"])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == "gram_cache_samples_per_sec" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["gpu_launches"] == 0 and "workload" in d["config"] and d["vs_baseline"] is None


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    import numpy as np

    d = _run(["--model", "tiny", "--steps", "3", "--warmup", "3", "--batch", "8", "--dump-outputs", str(tmp_path)])
    logits = np.load(tmp_path / "logits.npy")
    assert logits.shape == (8, 8) and logits.dtype == np.float32 and np.isfinite(logits).all()
    grams = sorted(tmp_path.glob("gram.*.npy"))
    assert len(grams) == 96 and sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20
    g = np.load(grams[0])
    assert g.dtype == np.float32 and g.shape == (192 + (1 << 15),) and (g[:192] > 0).all()   # diagonal, then the sample
    assert BASE_KEYS | {"roofline", "clocks", "merge"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["value"] > 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3
    assert d["gpu_launches"] > 0 and r["launches_timed"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 0
    assert d["merge"]["roofline"]["bound"] == "hbm" and d["merge"]["e2e"]["bit_exact_vs_torch"] is True
    assert d["cpu_baseline"]["kind"] == "port" and max(d["gram_parity_rel_fro"].values()) < 1e-3
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
