"""bench.py --dump-outputs on the CPU: the sample it writes of a batch output depends only on the output's shape,
holds the first and last instances and frames, stays within its byte budget and keeps the output's dtype."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sample_positions_are_fixed_and_within_budget(tmp_path, monkeypatch):
    monkeypatch.setitem(bench.DUMP_BYTES, "cfg3", 64 << 10)
    y = torch.from_numpy(np.random.default_rng(0).standard_normal((20, 2, 50000)))
    bench.dump_sample(str(tmp_path / "a"), "cfg3", y)
    bench.dump_sample(str(tmp_path / "b"), "cfg3", 2 * y)
    a, b = np.load(tmp_path / "a" / "cfg3.npy"), np.load(tmp_path / "b" / "cfg3.npy")
    assert a.dtype == np.float64 and a.nbytes <= 64 << 10 and a.shape[:2] == (8, 2)
    assert np.array_equal(b, 2 * a)                                   # same positions for the same shape
    yn = y.numpy()
    edge = min(1024, a.shape[2] // 4)
    assert np.array_equal(a[0, :, :edge], yn[0, :, :edge]) and np.array_equal(a[-1, :, -edge:], yn[-1, :, -edge:])
    pos = {v: i for i, v in enumerate(yn[0, 0])}
    idx = [pos[v] for v in a[0, 0]]
    assert idx == sorted(set(idx))                                    # distinct frames, in order
    assert np.array_equal(a[0], yn[0][:, idx])                        # channels sampled at the same frames


def test_small_output_is_written_whole(tmp_path):
    y = torch.from_numpy(np.random.default_rng(1).standard_normal((3, 1, 100)).astype(np.float32))
    bench.dump_sample(str(tmp_path), "cfg4", y)
    got = np.load(tmp_path / "cfg4.npy")
    assert got.dtype == np.float32 and np.array_equal(got, y.numpy())


def test_reference_arm_refuses_dump_outputs(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                        str(tmp_path)], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)
