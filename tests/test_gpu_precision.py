"""Every scenario of tests/precision.py on the GPU, through the C ABI with each step-kernel family, judged block by
block against the long-double oracle; and P2 and O1 advanced 50 ticks per launch by ukfb_run_dev, so that the
multi-tick loop carries the state between ticks on chip.  Run with `pytest -m gpu` on a B200."""
from __future__ import annotations

import numpy as np
import pytest

import precision as PR

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Ukf():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from slam_pose_estimation_b200 import UkfBatch

    return UkfBatch


@pytest.mark.parametrize("kernel", ["fast", "thread", "warp"])
@pytest.mark.parametrize("name", [n for n in PR.SCENARIOS if n not in PR.TICK_SCENARIOS])
def test_gpu_kernel_per_block_precision(Ukf, monkeypatch, name, kernel):
    monkeypatch.setenv("UKFB_KERNEL", kernel)  # read by ukfb_create
    _, fn = PR.SCENARIOS[name]
    PR.check(name, fn(Ukf), what=f"gpu {kernel}")


@pytest.mark.parametrize("kernel", ["fast", "thread", "warp"])
@pytest.mark.parametrize("name", PR.TICK_SCENARIOS)
def test_gpu_run_dev_per_block_precision(Ukf, monkeypatch, name, kernel):
    import torch

    monkeypatch.setenv("UKFB_KERNEL", kernel)
    K = 50
    kind, _ = PR.SCENARIOS[name]
    x = PR.run_ticks(name, lambda *a: _NoTicks(Ukf(*a)))  # set up as the single-call form does, without its ticks
    dev = torch.device("cuda:0")
    d_dt = torch.full((K,), PR.syn.DT, dtype=torch.float64, device=dev)
    ticks = PR.ticks(name)
    assert len(ticks) % K == 0
    for c in range(0, len(ticks), K):
        win = ticks[c:c + K]
        kinds = np.array([t[0] for t in win], np.int8)
        zs = np.stack([t[1] for t in win])
        Rs = np.stack([t[2] for t in win])
        imu = torch.from_numpy(np.stack([t[3] for t in win])).to(dev) if kind == 1 else None
        x.g.run_dev(K, d_dt, False, kinds, torch.from_numpy(zs).to(dev), torch.from_numpy(Rs).to(dev), False, imu)
        x.g.synchronize()  # the engine's stream reads this window's tensors: keep them alive until it is done
    PR.check(name, x.g, what=f"gpu {kernel} run_dev K={K}")


class _NoTicks:
    """a UkfBatch whose per-tick calls are dropped: run_ticks() then only creates, initialises and parametrises it"""

    def __init__(self, g):
        self.g = g

    def initialize(self, mu, sg):
        self.g.initialize(mu, sg)

    def set_process_noise(self, Q):
        self.g.set_process_noise(Q)

    def set_orientation_params(self, *a):
        self.g.set_orientation_params(*a)

    def set_rotation_rate(self, *a):
        pass

    def set_acceleration(self, *a):
        pass

    def predict_dt(self, *a):
        pass

    def update(self, *a):
        pass
