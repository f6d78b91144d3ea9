"""CPU: bench.py --dump-outputs writes float32 arrays within its size limit and, above it, the same seeded sample of
rays from every array; arguments it cannot honour are refused before anything runs."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_small_outputs_whole(tmp_path):
    depth, color = torch.rand(100), torch.rand(100, 3)
    bench.dump_outputs(str(tmp_path), {"depth": depth, "color": color})
    got = _load(tmp_path)
    assert sorted(got) == ["color", "depth"]
    assert got["depth"].dtype == np.float32 and np.array_equal(got["depth"], depth.numpy())
    assert got["color"].dtype == np.float32 and np.array_equal(got["color"], color.numpy())


def test_dump_outputs_samples_the_same_rays_of_every_array(tmp_path):
    n, limit = 10000, 1 << 20
    ray = torch.arange(n, dtype=torch.float32)
    arrays = {"depth": ray, "weights": ray[:, None].repeat(1, 128)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, limit_bytes=limit)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= limit
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == ["depth", "ray_index", "weights"]
    idx = a["ray_index"]
    assert a["ray_index"].dtype == np.float64 and 0 < idx.shape[0] < n and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["depth"], idx) and np.array_equal(a["weights"], np.repeat(idx[:, None], 128, 1))
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_dump_outputs_samples_gathered_frames_along_the_ray_axis(tmp_path):
    n = 4096
    frames = torch.arange(n, dtype=torch.float32)[None, :, None].repeat(3, 1, 4)
    bench.dump_outputs(str(tmp_path), {"frames": frames}, ray_axis=1, limit_bytes=64 << 10)
    got = _load(tmp_path)
    assert got["frames"].shape == (3, got["ray_index"].shape[0], 4)
    assert np.array_equal(got["frames"][1, :, 2], got["ray_index"])


def test_bench_refuses_arguments_it_cannot_honour(tmp_path):
    for extra in (["--steps", "0"], ["--workload", "sweep", "--dump-outputs", str(tmp_path)],
                  ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, bench.__file__, *extra], capture_output=True, text=True)
        assert r.returncode == 2 and "error" in r.stderr, extra
    assert os.listdir(tmp_path) == []
