"""CPU suite: the reference arm of bench.py (`--impl reference`) runs without a GPU and prints ONE JSON line with the contract keys
(the driver launches it beside our arm and divides the two `e2e` / `value` figures itself)."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line(tmp_path):
    dump = tmp_path / "out"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(dump)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images_per_sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("SD1.5-arch UNet 512^2") and d["config"]["unet_batch_per_gpu"] == 2
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert sorted(p.name for p in dump.iterdir()) == ["latent.npy"]
    lat = np.load(dump / "latent.npy")
    assert lat.dtype == np.float32 and lat.shape[:2] == (1, 4) and np.isfinite(lat).all()


def test_dump_outputs_samples_large_tensors(tmp_path, monkeypatch):
    """Outputs over the size cap are stored as a fixed seeded sample: the same elements in every run."""
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4 * 1000)
    t = torch.arange(5000, dtype=torch.float64).view(5, 1000)
    bench.dump_outputs(str(tmp_path / "a"), {"x": t})
    bench.dump_outputs(str(tmp_path / "b"), {"x": t})
    a, b = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "b" / "x.npy")
    assert a.dtype == np.float32 and a.shape == (1000,) and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and np.array_equal(a, a.astype(np.int64))   # distinct original elements, in order
    small = torch.ones((2, 3))
    bench.dump_outputs(str(tmp_path / "c"), {"y": small})
    assert np.load(tmp_path / "c" / "y.npy").shape == (2, 3)


def test_split_steps_times_exactly_k_steps():
    import bench
    for k in (1, 2, 5, 7, 50):
        for regions in (1, 3, 5, 9):
            parts = bench.split_steps(k, regions)
            assert sum(parts) == k and len(parts) == min(regions, k) and max(parts) - min(parts) <= 1
