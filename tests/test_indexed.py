"""Per-filter access to a batch: indexed state read-back, indexed re-initialisation, status lookup and indexed clear.

A caller of the reference owns N filter objects and calls getCurrentState / initializeFilter on the one it needs
(UnscentedKalmanFilter.hpp:40-75).  The indexed entry points must do exactly that to the listed filters and nothing to
the others: bit for bit what the whole-batch workaround (get_state, patch rows, get_last_time, initialize,
set_last_time) gives, on one device and on sharded handles, for both filter kinds and every kernel family
(UKFB_KERNEL=warp / thread run this file too)."""
from __future__ import annotations

import math
import os
import subprocess

import numpy as np
import pytest

import parity as P
from oracle.oracle_lib import OracleBatch
from slam_pose_estimation_b200 import _build, synthetic as syn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NOT_SPD, NONFINITE_MEAS = 8, 4


def device_lists():
    import torch

    n = torch.cuda.device_count()
    return [[0, 0, 0]] + ([list(range(n))] if n >= 2 else [])


def c3_from_sample_time(x, B, start, steps):
    """C3 schedule driven by predictionStepFromSampleTime: a filter whose time latch is 0 only latches"""
    for k in range(start, start + steps):
        x.predict_time(np.array([syn.T0_US + 1000 * k], np.int64))
        for kind in syn.pose_schedule(k):
            z, R = syn.pose_measurement(kind, B, k)
            x.update(kind, z, R)


def ori_steps(x, B, start, steps):
    P.run_ori_c1(x, B, steps, start=start, every=5)


def make(kind, cls, B, **kw):
    return P.make_pose(cls, B, **kw) if kind == 0 else P.make_ori(cls, B, **kw)


def run(kind, x, B, start, steps):
    (c3_from_sample_time if kind == 0 else ori_steps)(x, B, start, steps)


def new_rows(kind, S, seed):
    """fresh states for the filters S: the initial states of other filters, slightly moved"""
    rng = np.random.default_rng(seed)
    mu, sg = syn.pose_initial(len(S), perturb=True, first=1000 + seed) if kind == 0 else syn.orientation_initial(len(S))
    mu = mu.copy()
    mu[:, 0 if kind == 0 else 4] += rng.standard_normal(len(S)) * 0.1
    return mu, sg


def reinit_by_workaround(x, S, mu_s, sg_s):
    """what a caller can do without the indexed calls: the whole batch through the host"""
    mu, sg = x.get_state()
    mu[S], sg[S] = mu_s, sg_s
    t = x.get_last_time()
    x.initialize(mu, sg)
    t[S] = 0
    x.set_last_time(t)


def assert_same(a, b, what=""):
    (ma, sa), (mb, sb) = a.get_state(), b.get_state()
    assert np.array_equal(ma, mb) and np.array_equal(sa, sb), f"{what}: states differ"
    assert np.array_equal(a.get_status(), b.get_status()), f"{what}: status differs"
    assert np.array_equal(a.get_last_time(), b.get_last_time()), f"{what}: time latches differ"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_get_state_indexed_is_rows_of_get_state(kind):
    import torch

    from slam_pose_estimation_b200 import UkfBatch

    B = 203
    x = make(kind, UkfBatch, B)
    run(kind, x, B, 1, 12)
    mu, sg = x.get_state()
    rng = np.random.default_rng(kind)
    for idx in (np.arange(B), np.sort(rng.choice(B, 50, replace=False)), rng.permutation(B)[:77],
                np.array([5, 5, 202, 0, 5]), np.array([117])):
        m, s = x.get_state_indexed(idx)
        assert np.array_equal(m, mu[idx]) and np.array_equal(s, sg[idx])
        assert np.array_equal(x.get_state_indexed(idx, with_sigma=False), mu[idx])
        d_idx = torch.as_tensor(idx, dtype=torch.int64, device="cuda")
        d_mu = torch.empty((idx.size, x.MU), dtype=torch.float64, device="cuda")
        d_sg = torch.empty((idx.size, x.n, x.n), dtype=torch.float64, device="cuda")
        x.get_state_indexed_dev(d_idx, d_mu, d_sg)
        assert np.array_equal(d_mu.cpu().numpy(), mu[idx]) and np.array_equal(d_sg.cpu().numpy(), sg[idx])
        d_mu2 = torch.empty((idx.size, x.MU), dtype=torch.float64, device="cuda")
        x.get_state_indexed_dev(d_idx, d_mu2)
        assert np.array_equal(d_mu2.cpu().numpy(), mu[idx])
    assert x.get_state_indexed(np.array([], np.int64))[0].shape == (0, x.MU)


def _equivalence(kind, B, S, devices=None, steps=(12, 25), dev_path=False):
    """handle A: initialize_indexed(S); handle B: the whole-batch workaround; both continue and must stay identical"""
    import torch

    from slam_pose_estimation_b200 import UkfBatch

    kw = {} if devices is None else {"devices": devices}
    a, b = make(kind, UkfBatch, B, **kw), make(kind, UkfBatch, B)
    for x in (a, b):
        run(kind, x, B, 1, steps[0])
        x.clear_mean_iter_hist()
    mu_s, sg_s = new_rows(kind, S, seed=len(S))
    if dev_path:
        a.initialize_indexed_dev(torch.as_tensor(S, device="cuda"), torch.as_tensor(mu_s, device="cuda"),
                                 torch.as_tensor(sg_s, device="cuda"))
    else:
        a.initialize_indexed(S, mu_s, sg_s)
    reinit_by_workaround(b, S, mu_s, sg_s)
    assert_same(a, b, "right after the re-initialisation")
    for x in (a, b):
        run(kind, x, B, 1 + steps[0], steps[1])
    assert_same(a, b, "after more steps")
    assert np.array_equal(a.get_mean_iter_hist(), b.get_mean_iter_hist())
    return a, b


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_initialize_indexed_equals_the_whole_batch_workaround(kind):
    B = 203
    rng = np.random.default_rng(7)
    for S in (rng.permutation(B)[:40], np.array([0, 31, 32, 202]), np.arange(B)):
        _equivalence(kind, B, S)
    _equivalence(kind, B, rng.permutation(B)[:40], dev_path=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_initialize_indexed_between_overlapping_step_launches(kind):
    """64 Ki filters: consecutive step launches overlap tile by tile; the indexed calls sit between them in stream order"""
    B = 64 * 1024
    rng = np.random.default_rng(11)
    S = rng.permutation(B)[:5000]
    a, _ = _equivalence(kind, B, S, steps=(6, 12))
    if os.environ.get("UKFB_KERNEL", "fast") == "fast" and os.environ.get("UKFB_OVERLAP_LAUNCHES", "1") != "0":
        assert a.overlapped_launch_count() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_initialize_indexed_against_the_oracle(kind):
    from slam_pose_estimation_b200 import UkfBatch

    B = 203
    S = np.random.default_rng(3).permutation(B)[:60]
    g, o = make(kind, UkfBatch, B), make(kind, OracleBatch, B)
    mu_s, sg_s = new_rows(kind, S, seed=5)
    for x in (g, o):
        run(kind, x, B, 1, 10)
    g.initialize_indexed(S, mu_s, sg_s)
    reinit_by_workaround(o, S, mu_s, sg_s)
    for x in (g, o):
        run(kind, x, B, 11, 20)
    P.assert_parity(kind, g.get_state(), o.get_state(), what="initialize_indexed vs oracle")
    assert np.array_equal(g.get_last_time(), o.get_last_time())


def _recovery(devices=None):
    """PoseUKF: a covariance that is not positive definite makes the next prediction fail (NOT_SPD), sticky.
    OrientationUKF: a NaN velocity measurement is refused (NONFINITE_MEAS).  find_status names exactly those
    filters; initialize_indexed + clear_status_indexed brings them back; 50 more steps match the oracle."""
    from slam_pose_estimation_b200 import UkfBatch

    kw = {} if devices is None else {"devices": devices}
    B = 203
    F = np.array([4, 40, 41, 100, 202])
    out = []
    for kind in (0, 1):
        g, o = make(kind, UkfBatch, B, **kw), make(kind, OracleBatch, B)
        run(kind, g, B, 1, 5)
        run(kind, o, B, 1, 5)
        if kind == 0:
            mu, sg = g.get_state_indexed(F)
            sg[:, 0, 0] = -1.0
            g.initialize_indexed(F, mu, sg)
            run(kind, g, B, 6, 3)  # g's F latch, then fail at every prediction
            run(kind, o, B, 6, 3)
            bit = NOT_SPD
        else:
            z, R = syn.orientation_velocity(B, 6)
            z[F] = np.nan
            g.update(9, z, R)
            o.update(9, z, R)
            bit = NONFINITE_MEAS
        assert np.array_equal(g.find_status(bit), F)
        assert np.array_equal(g.find_status(), F)
        mu_s, sg_s = new_rows(kind, F, seed=9)
        g.initialize_indexed(F, mu_s, sg_s)
        g.clear_status_indexed(F)
        reinit_by_workaround(o, F, mu_s, sg_s)
        o.clear_status()
        assert g.find_status().size == 0
        run(kind, g, B, 20, 50)
        run(kind, o, B, 20, 50)
        P.assert_parity(kind, g.get_state(), o.get_state(), what=f"recovery kind {kind}")
        assert not g.get_status().any() and g.find_status().size == 0
        out.append(g.get_state())
    return out


@pytest.mark.gpu
def test_recovery_of_failed_filters():
    _recovery()


@pytest.mark.gpu
def test_sharded_handles_equal_one_device():
    from slam_pose_estimation_b200 import UkfBatch, UkfbError
    import torch

    B = 203
    rng = np.random.default_rng(21)
    S = rng.permutation(B)[:90]  # unsorted, every shard
    ref = _recovery()
    for devs in device_lists():
        for kind in (0, 1):
            a, b = _equivalence(kind, B, S, devices=devs)
            idx = rng.permutation(B)[:120]
            assert np.array_equal(a.get_state_indexed(idx)[0], b.get_state_indexed(idx)[0])
            assert np.array_equal(a.get_state_indexed(idx)[1], b.get_state_indexed(idx)[1])
            d = torch.zeros(4, dtype=torch.int64, device="cuda")
            m = torch.zeros((4, a.MU), dtype=torch.float64, device="cuda")
            s = torch.zeros((4, a.n, a.n), dtype=torch.float64, device="cuda")
            for call in (lambda: a.get_state_indexed_dev(d, m, s), lambda: a.initialize_indexed_dev(d, m, s)):
                with pytest.raises(UkfbError) as e:
                    call()
                assert e.value.code == -1
        got = _recovery(devices=devs)
        for (m1, s1), (m2, s2) in zip(got, ref):
            assert np.array_equal(m1, m2) and np.array_equal(s1, s2)


@pytest.mark.gpu
def test_find_status_and_clear_on_sharded_handle():
    from slam_pose_estimation_b200 import UkfBatch

    B = 203
    for devs in device_lists():
        s, g = P.make_ori(UkfBatch, B, devices=devs), P.make_ori(UkfBatch, B)
        z, R = syn.orientation_velocity(B, 1)
        bad = np.array([1, 60, 67, 68, 69, 135, 136, 200])  # around the shard boundaries of [0, 0, 0]
        z[bad] = np.nan
        for x in (s, g):
            x.update(9, z, R)
        assert np.array_equal(s.find_status(), bad) and np.array_equal(g.find_status(), bad)
        for x in (s, g):
            x.clear_status_indexed(bad[::2])
        assert np.array_equal(s.find_status(NONFINITE_MEAS), bad[1::2])
        assert np.array_equal(s.get_status(), g.get_status())


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0, 0]])
def test_rejected_calls_change_nothing(devices):
    from slam_pose_estimation_b200 import UkfBatch, UkfbError

    B = 203
    kw = {} if devices is None else {"devices": devices}
    x = P.make_ori(UkfBatch, B, **kw)
    ori_steps(x, B, 1, 5)
    z, R = syn.orientation_velocity(B, 6)
    z[[3, 150]] = np.nan
    x.update(9, z, R)
    before = (*x.get_state(), x.get_status(), x.get_last_time())
    mu, sg = syn.orientation_initial(3)
    for idx in (np.array([1, 150, 1]), np.array([0, B, 2]), np.array([-1, 5, 6])):  # duplicate, out of range
        with pytest.raises(UkfbError) as e:
            x.initialize_indexed(idx, mu, sg)
        assert e.value.code == -1
    for idx in (np.array([0, B]), np.array([-1])):
        with pytest.raises(UkfbError):
            x.get_state_indexed(idx)
        with pytest.raises(UkfbError):
            x.clear_status_indexed(idx)
    after = (*x.get_state(), x.get_status(), x.get_last_time())
    for u, v in zip(before, after):
        assert np.array_equal(u, v)
    assert np.array_equal(x.find_status(), np.array([3, 150]))


@pytest.mark.gpu
def test_initialize_indexed_needs_an_initialized_handle():
    from slam_pose_estimation_b200 import UkfBatch, UkfbError

    x = UkfBatch(0, 40)
    mu, sg = syn.pose_initial(1)
    with pytest.raises(UkfbError) as e:
        x.initialize_indexed([3], mu, sg)
    assert e.value.code == -2


# ---- C++ mirror: initializeFilter(index, ...), getCurrentState(index, ...), lastFailedFilters() -----------------------

@pytest.fixture(scope="module")
def recovery_demo(tmp_path_factory):
    _build.build()
    exe = str(tmp_path_factory.mktemp("cpp") / "recovery_demo")
    libdir = os.path.dirname(_build.LIB)
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "recovery_demo.cpp"), "-L", libdir, "-lukfb", f"-Wl,-rpath,{libdir}",
                    "-o", exe], check=True)
    return exe


def test_recovery_demo_compiles_and_fails_loudly_without_gpu(recovery_demo):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([recovery_demo, "64"], capture_output=True, text=True)
    assert r.returncode != 0 and ("no CPU path" in r.stderr or "CUDA" in r.stderr)


def _wobble(b, k, c):
    return math.sin(0.37 * b + 1.3 * k + 0.71 * c)


def _oracle_for_recovery_demo(B):
    """the calls of tests/cpp/recovery_demo.cpp on the oracle, its failing filters re-initialised the long way"""
    d0 = np.array([1, 1, 1, 0.01, 0.01, 0.01, 0.1, 0.1, 0.1, 0.01, 0.01, 0.01])
    mu0, sg0 = np.zeros((B, 13)), np.zeros((B, 12, 12))
    for b in range(B):
        yaw = 0.3 * _wobble(b, 20, 0)
        mu0[b, 0], mu0[b, 1] = _wobble(b, 21, 0), _wobble(b, 21, 1)
        mu0[b, 5], mu0[b, 6] = math.sin(0.5 * yaw), math.cos(0.5 * yaw)
        mu0[b, 7] = 1.0 + 0.1 * _wobble(b, 22, 0)
        mu0[b, 12] = 0.05
        sg0[b] = np.diag([d0[i] * (1.0 + 0.2 * _wobble(b, 23, i)) for i in range(12)])
    o = OracleBatch(0, B)
    o.initialize(mu0, sg0)
    failed = np.array([b for b in range(B) if b % 13 == 5])
    o.predict_time(np.array([1000000], np.int64))
    o.predict_time(np.array([1010000], np.int64))
    reinit_by_workaround(o, failed, mu0[failed], sg0[failed])
    o.predict_time(np.array([1020000], np.int64))
    w = np.array([[(0.05 if i == 2 else 0.0) + 1e-3 * _wobble(b, 0, i) for i in range(3)] for b in range(B)])
    o.update(8, w, np.tile(np.eye(3) * 1e-6, (B, 1, 1)))
    o.predict_time(np.array([1030000], np.int64))
    o.update(4, np.tile([1.01, 0.0, 0.0], (B, 1)), np.eye(3) * 1e-4)
    return o, failed


@pytest.mark.gpu
def test_cpp_recovery_through_the_batch_object(recovery_demo):
    B = 64
    r = subprocess.run([recovery_demo, str(B)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == "after_latch_failed 0"
    assert lines[1] == "caught ukfom: covariance is not positive definite"  # the same text as before this API existed
    o, failed = _oracle_for_recovery_demo(B)
    assert lines[2].split()[1:] == [str(b) for b in failed]
    assert lines[3] == "after_steps_failed 0" and lines[4] == "indexed_equals_batch 1"
    vals = np.array([[float(v) for v in ln.split()[2:]] for ln in lines[5:]])
    assert vals.shape == (B, 13 + 144)
    P.assert_parity(0, (vals[:, :13], vals[:, 13:].reshape(B, 12, 12)), o.get_state(), what="C++ recovery")
