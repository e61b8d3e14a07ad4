"""CPU: bench.py's reference arm honours the driver contract (one JSON line, required keys)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "spectra/sec" and d["unit"] == "spectra/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_non_zero_rank_of_reference_arm_exits_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--gpus", "2", "--steps", "1", "--warmup", "1"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_fits_budget_and_samples_rows_reproducibly(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    big = torch.arange(300 * 60000, dtype=torch.float32).reshape(300, 60000)    # 72 MB
    small = torch.linspace(0, 1, 1000, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs({"big": big, "small": small}, str(tmp_path / d))
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and 0 < a.shape[0] < 300 and np.array_equal(a, b)
    rows = a[:, 0] / 60000
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, big.numpy()[rows.astype(int)])
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())
    # one dim-0 slice above the share (the gathered [chunks, ranks, C, F, bins] layout), and one
    # last-dim row above it: every file still fits, rows of the flattened output are sampled
    monkeypatch.setattr(bench, "DUMP_BYTES", 1_000_000)
    gathered = torch.arange(2 * 300 * 1000, dtype=torch.float32).reshape(2, 3, 100, 1000)      # 2.4 MB
    wide = torch.arange(200_000, dtype=torch.float64).reshape(1, 200_000)                     # 1.6 MB
    bench.dump_outputs({"gathered": gathered, "wide": wide}, str(tmp_path / "c"))
    files = sorted(os.listdir(tmp_path / "c"))
    assert sum(os.path.getsize(tmp_path / "c" / f) for f in files) <= bench.DUMP_BYTES
    g, w = np.load(tmp_path / "c" / "gathered.npy"), np.load(tmp_path / "c" / "wide.npy")
    assert g.ndim == 2 and g.shape[1] == 1000 and 0 < g.shape[0] < 600
    assert np.array_equal(g, gathered.numpy().reshape(-1, 1000)[(g[:, 0] / 1000).astype(int)])
    assert w.dtype == np.float64 and w.shape[1] == 1 and 0 < w.shape[0] < 200_000
    assert np.all(np.diff(w[:, 0]) > 0) and np.array_equal(w, wide.numpy().reshape(-1, 1)[w[:, 0].astype(int)])
