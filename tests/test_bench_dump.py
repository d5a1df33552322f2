"""bench.py --dump-outputs: the files it writes (names, float32, the size cap of the pixel sample) and, on the GPU,
that two runs with the same arguments write the same outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("conf", "depthmaps", "focals", "poses", "principal_points")


class _Scene:
    """The getters of LightPointCloudGroupOptimizer that dump_outputs reads, on seeded CPU tensors."""

    def __init__(self, T, H, W):
        g = torch.Generator().manual_seed(1)
        self.T, self.H, self.W = T, H, W
        self.depth = torch.rand(T, H * W, generator=g)
        self.conf = torch.rand(T, H, W, generator=g)

    def get_depthmaps(self):
        return [d.view(self.H, self.W) for d in self.depth]

    def get_conf(self):
        return list(self.conf)

    def get_im_poses(self):
        return torch.eye(4).repeat(self.T, 1, 1).requires_grad_()

    def get_focals(self):
        return torch.full((self.T, 1), 300.0)

    def get_principal_points(self):
        return torch.tensor([(self.W / 2, self.H / 2)] * self.T)


def _load(d):
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in NAMES)
    return {n: np.load(os.path.join(d, n + ".npy")) for n in NAMES}


def test_dump_outputs_whole_and_sampled(tmp_path, monkeypatch):
    import bench
    small = _Scene(4, 8, 16)
    bench.dump_outputs(small, str(tmp_path / "small"))
    out = _load(tmp_path / "small")
    assert all(a.dtype == np.float32 for a in out.values())
    assert np.array_equal(out["depthmaps"], small.depth.view(4, 8, 16).numpy())
    assert np.array_equal(out["conf"], small.conf.numpy())
    assert out["poses"].shape == (4, 4, 4) and out["focals"].shape == (4, 1) and out["principal_points"].shape == (4, 2)
    # a clip above the cap: the same sorted pixel sample for depth and confidence in every call
    monkeypatch.setattr(bench, "DUMP_MAX_PIXELS", 100)
    big = _Scene(3, 8, 16)
    for d in ("a", "b"):
        bench.dump_outputs(big, str(tmp_path / d))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(np.array_equal(a[n], b[n]) for n in NAMES)
    assert a["depthmaps"].shape == a["conf"].shape == (100,)
    flat_d, flat_c = big.depth.reshape(-1).numpy(), big.conf.reshape(-1).numpy()
    idx = np.nonzero(np.isin(flat_d, a["depthmaps"]))[0]
    assert len(idx) == 100 and np.array_equal(flat_d[idx], a["depthmaps"]) and np.array_equal(flat_c[idx], a["conf"])


@pytest.mark.gpu
def test_bench_dump_is_reproducible(cuda_device, tmp_path):
    """A tiny workload (2 windows of 16 frames at 128x192, 2 DDIM steps, 20 alignment iterations) twice, each in
    its own process; the tile autotuner is off so that the GEMM configuration, and with it the rounding, is fixed."""
    env = dict(os.environ, GEO4D_AUTOTUNE="0")
    outs = []
    for run in ("a", "b"):
        d = str(tmp_path / run)
        cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
               "--frames", "24", "--height", "128", "--width", "192", "--ddim-steps", "2", "--align-iters", "20",
               "--single-window-steps", "0", "--no-cpu-baseline", "--dump-outputs", d]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=REPO, env=env)
        assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["warmup"] == 1
        outs.append(_load(d))
    a, b = outs
    assert a["depthmaps"].shape == a["conf"].shape == (24, 128, 192)
    assert a["poses"].shape == (24, 4, 4) and a["focals"].shape == (24, 1)
    assert all(a[n].dtype == np.float32 and np.isfinite(a[n]).all() for n in NAMES)
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for n in NAMES:
        assert np.array_equal(a[n], b[n]), n
