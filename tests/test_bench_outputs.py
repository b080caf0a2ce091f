"""bench.py --dump-outputs: what the timed path returned in its last step, written as .npy files that two builds of the
project can compare array for array."""
import json
import subprocess
import sys
from argparse import Namespace
from pathlib import Path

import numpy as np
import pytest
import torch

import bench

ROOT = Path(__file__).resolve().parent.parent


def test_dump_writes_float32_and_keeps_float64(tmp_path):
    arrays = {"refmap": torch.rand(2, 4, 4, 3), "refmask": torch.rand(2, 4, 4) > 0.5,
              "counts": torch.arange(32, dtype=torch.int32).reshape(2, 4, 4), "scale": torch.rand(2, dtype=torch.float64)}
    bench.dump_outputs(arrays, tmp_path / "out")
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == [f"{n}.npy" for n in sorted(arrays)]
    for name, t in arrays.items():
        a = np.load(tmp_path / "out" / f"{name}.npy")
        assert a.dtype == (np.float64 if t.dtype == torch.float64 else np.float32) and a.shape == tuple(t.shape)
        assert np.array_equal(a, t.numpy().astype(a.dtype))


def test_dump_past_the_limit_is_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100_000)
    arrays = {"big": torch.rand(40, 1000), "wide": torch.rand(10_000, dtype=torch.float64)}
    for d in ("a", "b"):
        bench.dump_outputs(arrays, tmp_path / d)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 100_000
    for name, t in arrays.items():
        idx = np.load(tmp_path / "a" / f"{name}.sample_index.npy")
        vals = np.load(tmp_path / "a" / f"{name}.npy")
        assert idx.dtype == np.float64 and len(idx) == len(vals) > 0 and (np.diff(idx) > 0).all()
        assert np.array_equal(vals, t.numpy().reshape(-1)[idx.astype(np.int64)].astype(vals.dtype))
        assert np.array_equal(idx, np.load(tmp_path / "b" / f"{name}.sample_index.npy"))
        assert np.array_equal(vals, np.load(tmp_path / "b" / f"{name}.npy"))


@pytest.mark.gpu
def test_render_dump_is_the_last_step_on_the_seeded_inputs(tmp_path):
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "render", "--batch", "2", "--steps", "2",
                        "--warmup", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout)["steps"] == 2
    dumped = np.load(tmp_path / "refmaps.npy")
    W = bench.wl_render(Namespace(batch=2, footprint="auto"), 0, torch.device("cuda:0"))
    ours = W["step"]().cpu().numpy()
    assert dumped.dtype == np.float32 and dumped.shape == (2, 3, 128, 128)
    assert np.array_equal(dumped, ours)
