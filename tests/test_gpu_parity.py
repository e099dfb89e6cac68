"""GPU parity tests: the CUDA engine, called through the C ABI (lib/libukfb.so), against the
CPU oracle on identical seeded inputs.  Tolerance: 1e-9 (north star), norm-wise metrics
of SURVEY.md section 8(d) -- see tests/parity.py.  Run with `pytest -m gpu` on a B200.
"""
from __future__ import annotations

import numpy as np
import pytest

import parity as P
from oracle.oracle_lib import OracleBatch
from slam_pose_estimation_b200 import synthetic as syn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Ukf():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from slam_pose_estimation_b200 import UkfBatch

    return UkfBatch


def both(Ukf, kind, B, **kw):
    if kind == 0:
        return P.make_pose(Ukf, B, **kw), P.make_pose(OracleBatch, B, **kw)
    return P.make_ori(Ukf, B), P.make_ori(OracleBatch, B)


# ---- single operations -----------------------------------------------------------------------

@pytest.mark.parametrize("B", [1, 3, 4, 5, 33, 1000])
def test_pose_predict(Ukf, B):
    g, o = both(Ukf, 0, B)
    for x in (g, o):
        x.predict_dt(0.01)
    P.assert_parity(0, g.get_state(), o.get_state(), what=f"pose predict B={B}")
    assert P.spd_ok(g.get_state()[1])


def test_pose_predict_per_filter_dt(Ukf):
    B = 70
    g, o = both(Ukf, 0, B)
    dt = np.linspace(1e-3, 0.5, B)
    for x in (g, o):
        x.predict_dt(dt)
    P.assert_parity(0, g.get_state(), o.get_state(), what="per-filter dt")


@pytest.mark.parametrize("kind", list(range(9)))
def test_pose_update_kinds(Ukf, kind):
    B = 37
    g, o = both(Ukf, 0, B)
    z, R = syn.pose_measurement(kind, B, 7)
    for x in (g, o):
        x.predict_dt(0.05)
        x.update(kind, z, R)
    P.assert_parity(0, g.get_state(), o.get_state(), what=f"pose update kind {kind}")


def test_pose_update_per_filter_cov_and_mask(Ukf):
    B = 50
    g, o = both(Ukf, 0, B)
    z, R = syn.pose_measurement(4, B, 3, r_scale=np.linspace(0.25, 4.0, B))
    mask = (np.arange(B) % 3 != 0).astype(np.uint8)
    before = None
    for x in (g, o):
        x.predict_dt(0.02)
        before = x.get_state()
        x.update(4, z, R, mask)
    gs, os_ = g.get_state(), o.get_state()
    P.assert_parity(0, gs, os_, what="masked update")
    # masked-out filters are untouched by the update
    assert np.array_equal(os_[0][mask == 0], before[0][mask == 0])


def test_pose_acceleration_branch(Ukf):
    """finite stored acceleration: the shadowed process noise of PoseUKF.cpp:188-193"""
    B = 19
    g, o = both(Ukf, 0, B)
    acc = 0.01 * syn.noise(np.arange(B), 1, 13, 3)
    cov = np.eye(3) * 1e-4
    part = (np.arange(B) % 2).astype(np.uint8)  # half the filters keep the NaN sentinel
    for x in (g, o):
        x.set_acceleration(acc, cov, part)
        x.predict_dt(0.01)
        x.predict_dt(0.01)
    P.assert_parity(0, g.get_state(), o.get_state(), what="acceleration branch")


def test_orientation_predict_and_update(Ukf):
    B = 41
    g, o = both(Ukf, 1, B)
    for k in range(1, 4):
        gyro, acc = syn.orientation_imu(B, k)
        z, R = syn.orientation_velocity(B, k)
        for x in (g, o):
            x.set_rotation_rate(gyro)
            x.set_acceleration(acc)
            x.predict_dt(syn.DT)
            x.update(9, z, R)
    P.assert_parity(1, g.get_state(), o.get_state(), what="orientation predict+update")
    assert np.allclose(g.get_rotation_rate(), o.get_rotation_rate(), rtol=0, atol=1e-15)


def test_fused_step_equals_predict_then_update(Ukf):
    B = 21
    a, _ = both(Ukf, 0, B)
    b = P.make_pose(Ukf, B)
    z, R = syn.pose_measurement(8, B, 2)
    a.step(0.01, 8, z, R)
    b.predict_dt(0.01)
    b.update(8, z, R)
    sa, sb = a.get_state(), b.get_state()
    assert np.array_equal(sa[0], sb[0]) and np.array_equal(sa[1], sb[1])


def test_update_mixed(Ukf):
    B = 64
    g, o = both(Ukf, 0, B)
    kinds = (np.arange(B) % 10 - 1).astype(np.int8)  # -1 .. 8
    mu3 = np.zeros((B, 3))
    cov33 = np.tile(np.eye(3), (B, 1, 1))
    for b in range(B):
        k = int(kinds[b])
        if k < 0:
            continue
        z, R = syn.pose_measurement(k, B, 5)
        m = z.shape[1]
        mu3[b, :m] = z[b]
        cov33[b, :m, :m] = R
    for x in (g, o):
        x.predict_dt(0.01)
        x.update_mixed(kinds, mu3, cov33)
    P.assert_parity(0, g.get_state(), o.get_state(), what="mixed kinds")


# ---- guards (UnscentedKalmanFilter.hpp:83-125, :142-147) ----------------------------------------

def test_time_guards(Ukf):
    B = 6
    g, o = both(Ukf, 0, B)
    dt = np.array([-1.0, 0.0, 1e-10, 0.01, 5.0, 0.02])
    for x in (g, o):
        x.set_time_bounds(1e-9, 1.0)
        x.predict_dt(dt)
    sg, so = g.get_status(), o.get_status()
    assert np.array_equal(sg, so)
    assert sg[0] == 1 and sg[4] == 2 and sg[1] == 0 and sg[2] == 0
    P.assert_parity(0, g.get_state(), o.get_state(), what="time guards")
    n, bits = g.status_summary()
    assert n == 2 and bits == 3


def test_sample_time_latching(Ukf):
    B = 5
    g, o = both(Ukf, 0, B)
    seq = [syn.T0_US, syn.T0_US + 1000, syn.T0_US + 1000, syn.T0_US + 500, syn.T0_US + 3000]
    for ts in seq:
        for x in (g, o):
            x.predict_time(np.array([ts], np.int64))
    assert np.array_equal(g.get_last_time(), o.get_last_time())
    assert np.array_equal(g.get_status(), o.get_status())
    assert (g.get_status() == 1).all()  # one negative delta each
    P.assert_parity(0, g.get_state(), o.get_state(), what="sample-time path")


def test_nonfinite_measurement_orientation(Ukf):
    B = 4
    g, o = both(Ukf, 1, B)
    z, R = syn.orientation_velocity(B, 1)
    z[1, 0] = np.nan
    gyro, acc = syn.orientation_imu(B, 1)
    gyro[2, 1] = np.inf
    for x in (g, o):
        x.set_rotation_rate(gyro)
        x.set_acceleration(acc)
        x.predict_dt(syn.DT)
        x.update(9, z, R)
    assert np.array_equal(g.get_status(), o.get_status())
    assert g.get_status()[1] == 4 and g.get_status()[2] == 4
    P.assert_parity(1, g.get_state(), o.get_state(), what="non-finite measurement")


def test_not_initialized_and_wrong_kind(Ukf):
    from slam_pose_estimation_b200 import UkfbError

    x = Ukf(0, 4)
    with pytest.raises(UkfbError) as e:
        x.get_state()
    assert e.value.code == -2
    mu, sg = syn.pose_initial(4)
    x.initialize(mu, sg)
    with pytest.raises(UkfbError) as e:
        x.update(9, np.zeros((4, 3)), np.eye(3))
    assert e.value.code == -1


def test_reinitialize_resets_time(Ukf):
    B = 3
    g, o = both(Ukf, 0, B)
    mu, sg = syn.pose_initial(B)
    for x in (g, o):
        x.predict_time(np.array([syn.T0_US], np.int64))
        x.initialize(mu, sg)
    assert (g.get_last_time() == 0).all() and np.array_equal(g.get_last_time(), o.get_last_time())


def test_process_noise_roundtrip_and_per_filter(Ukf):
    B = 9
    g, o = both(Ukf, 0, B)
    rng = np.random.default_rng(1)
    A = rng.normal(size=(B, 12, 12)) * 0.01
    Q = A @ np.transpose(A, (0, 2, 1))
    for x in (g, o):
        x.set_process_noise(Q)
        x.predict_dt(0.1)
    assert np.allclose(g.get_process_noise(per_filter=True), Q, rtol=0, atol=0)
    P.assert_parity(0, g.get_state(), o.get_state(), what="per-filter Q")


@pytest.mark.parametrize("filt", [0, 1])
def test_dense_and_diagonal_broadcast_process_noise(Ukf, filt):
    """a broadcast Q without off-diagonal entries takes the 12/13-load path of the fast kernels, a dense one the general path"""
    B = 40
    n = 12 if filt == 0 else 13
    rng = np.random.default_rng(11)
    A = rng.normal(size=(n, n)) * 0.01
    for Q in (A @ A.T, np.diag(rng.uniform(1e-6, 1e-3, n))):
        g, o = both(Ukf, filt, B)
        for x in (g, o):
            x.set_process_noise(Q)
            if filt == 0:
                P.run_pose_c3(x, B, 8)
            else:
                P.run_ori_c1(x, B, 8, every=4)
        assert np.array_equal(np.tril(g.get_process_noise()), np.tril(Q))  # the engine keeps the lower triangle
        P.assert_parity(filt, g.get_state(), o.get_state(), what="broadcast Q")


# ---- streams ---------------------------------------------------------------------------------------

def test_pose_c3_200_steps(Ukf):
    B = 256
    g, o = both(Ukf, 0, B)
    P.run_pose_c3(g, B, 200)
    P.run_pose_c3(o, B, 200)
    em, es = P.assert_parity(0, g.get_state(), o.get_state(), what="C3 200 steps")
    assert np.array_equal(g.get_status(), o.get_status()) and not g.get_status().any()
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())


def test_orientation_c1_10k_steps(Ukf):
    """BASELINE config 1: a single OrientationUKF on a 1 kHz IMU stream for 10k steps."""
    g, o = both(Ukf, 1, 1)
    P.run_ori_c1(g, 1, 10_000)
    P.run_ori_c1(o, 1, 10_000)
    P.assert_parity(1, g.get_state(), o.get_state(), what="C1 10k steps")
    assert not g.get_status().any()


def test_pose_10k_steps_run_dev(Ukf):
    """10k fused predict+update ticks advanced on-chip K at a time (ukfb_run_dev) vs the oracle."""
    import torch

    B, steps, K = 8, 10_000, 100
    g, o = both(Ukf, 0, B)
    dev = torch.device("cuda:0")
    d_dt = torch.full((K,), syn.DT, dtype=torch.float64, device=dev)
    kinds = np.full(K, 8, np.int8)
    R = np.eye(3) * syn.SIGMA_GYRO**2
    d_R = torch.from_numpy(np.tile(R, (K, 1, 1))).to(dev)
    for c in range(steps // K):
        zs = np.stack([syn.pose_measurement(8, B, c * K + j + 1)[0] for j in range(K)])
        d_z = torch.from_numpy(zs).to(dev)
        g.run_dev(K, d_dt, False, kinds, d_z, d_R, False)
        g.synchronize()
        for j in range(K):
            o.step(syn.DT, 8, zs[j], R)
    P.assert_parity(0, g.get_state(), o.get_state(), what="10k steps run_dev")
    assert not g.get_status().any()


def test_run_dev_with_a_schedule_that_changes_between_calls(Ukf):
    """ukfb_run_dev keeps the K tick kinds of its last call on the device and rewrites them only when they change (a copy
    between two launches is a full ordering point): same schedule twice, another schedule, a longer one, the first again"""
    import torch

    B = 70
    g, o = both(Ukf, 0, B)
    dev = torch.device("cuda:0")
    tick = 0
    for kinds in ([8, 8, 4, 8], [8, 8, 4, 8], [0, -1, 8, 7], [8, 4, 8, 8, 0, 8, -1, 2, 8], [8, 8, 4, 8]):
        K = len(kinds)
        zs, Rs = np.zeros((K, B, 3)), np.tile(np.eye(3), (K, 1, 1))
        for j, kind in enumerate(kinds):
            tick += 1
            if kind >= 0:
                z, R = syn.pose_measurement(kind, B, tick)
                m = z.shape[1]
                zs[j, :, :m], Rs[j, :m, :m] = z, R
        g.run_dev(K, torch.full((K,), syn.DT, dtype=torch.float64, device=dev), False, np.array(kinds, np.int8),
                  torch.from_numpy(zs).to(dev), torch.from_numpy(Rs).to(dev), False)
        for j, kind in enumerate(kinds):
            o.predict_dt(syn.DT)
            if kind >= 0:
                m = g.meas_dim(kind)
                o.update(kind, zs[j, :, :m], Rs[j, :m, :m])
    P.assert_parity(0, g.get_state(), o.get_state(), what="run_dev, changing schedules")
    assert np.array_equal(g.get_status(), o.get_status())


def test_pose_c3_10k_steps_mixed_updates(Ukf):
    """north star: 1e-9 after 10k steps on the C3 schedule (angular velocity every tick, velocity every 10th, position
    every 100th), through the single calls"""
    B = 6
    g, o = both(Ukf, 0, B)
    P.run_pose_c3(g, B, 10_000)
    P.run_pose_c3(o, B, 10_000)
    em, es = P.assert_parity(0, g.get_state(), o.get_state(), what="C3, 10k steps")
    assert not g.get_status().any()
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())


def test_shard_invariance(Ukf):
    """a filter's result does not depend on the batch it is in or its position in it (section 8e)"""
    B = 101
    whole = P.make_pose(Ukf, B)
    P.run_pose_c3(whole, B, 12)
    mu_w, sg_w = whole.get_state()
    lo, hi = 37, 64
    part = P.make_pose(Ukf, hi - lo, first=lo)
    P.run_pose_c3(part, hi - lo, 12, first=lo)
    mu_p, sg_p = part.get_state()
    assert np.array_equal(mu_w[lo:hi], mu_p) and np.array_equal(sg_w[lo:hi], sg_p)


def test_large_batch_invariants(Ukf):
    """full BASELINE size (65,536 PoseUKF): finite, symmetric PSD, unit quaternions; a strided sample matches the oracle."""
    B = 65_536
    g = P.make_pose(Ukf, B)
    P.run_pose_c3(g, B, 10)
    mu, sg = g.get_state()
    assert np.isfinite(mu).all() and np.isfinite(sg).all()
    assert np.abs(np.linalg.norm(mu[:, 3:7], axis=1) - 1.0).max() < 1e-12
    assert P.spd_ok(sg[::257])
    assert not g.get_status().any()
    idx = np.arange(0, B, 4099)
    for i in idx:
        o = P.make_pose(OracleBatch, 1, first=int(i))
        P.run_pose_c3(o, 1, 10, first=int(i))
        P.assert_parity(0, (mu[i:i + 1], sg[i:i + 1]), o.get_state(), what=f"filter {i} of 65536")


def test_full_size_c4_invariants_and_shards(Ukf):
    """BASELINE config 4 at its full size (1,048,576 PoseUKF, Monte-Carlo initial states): size-independent
    properties -- finite, unit quaternions, symmetric positive definite covariances, no status bits, one mean pass --
    a strided sample against the oracle, and a shard of the sweep run on its own is bitwise equal to its slice."""
    B = 1 << 20
    g = P.make_pose(Ukf, B)
    for k in range(1, 4):
        z, R = syn.pose_measurement(8, B, k)
        g.step(syn.DT, 8, z, R)
    mu, sg = g.get_state()
    assert np.isfinite(mu).all() and np.isfinite(sg).all()
    assert np.abs(np.linalg.norm(mu[:, 3:7], axis=1) - 1.0).max() < 1e-12
    assert P.spd_ok(sg[::4099])
    assert not g.get_status().any()
    assert g.get_mean_iter_hist()[1] == 2 * 3 * B
    for i in np.arange(0, B, 65_537):
        o = P.make_pose(OracleBatch, 1, first=int(i))
        for k in range(1, 4):
            z, R = syn.pose_measurement(8, 1, k, first=int(i))
            o.step(syn.DT, 8, z, R)
        P.assert_parity(0, (mu[i:i + 1], sg[i:i + 1]), o.get_state(), what=f"filter {i} of 1 Mi")
    lo, n = 5 * (B // 8), 4096  # inside the shard rank 5 of 8 owns
    part = P.make_pose(Ukf, n, first=lo)
    for k in range(1, 4):
        z, R = syn.pose_measurement(8, n, k, first=lo)
        part.step(syn.DT, 8, z, R)
    mu_p, sg_p = part.get_state()
    assert np.array_equal(mu[lo:lo + n], mu_p) and np.array_equal(sg[lo:lo + n], sg_p)


def test_full_size_c2_orientation_invariants(Ukf):
    """BASELINE config 2 at its full size (65,536 OrientationUKF on the IMU stream)."""
    B = 65_536
    g = P.make_ori(Ukf, B)
    P.run_ori_c1(g, B, 20, every=10)
    mu, sg = g.get_state()
    assert np.isfinite(mu).all() and np.isfinite(sg).all()
    assert np.abs(np.linalg.norm(mu[:, 0:4], axis=1) - 1.0).max() < 1e-12
    assert P.spd_ok(sg[::257])
    assert not g.get_status().any()
    for i in np.arange(0, B, 8191):
        o = P.make_ori(OracleBatch, 1)
        P.run_ori_c1(o, 1, 20, first=int(i), every=10)
        P.assert_parity(1, (mu[i:i + 1], sg[i:i + 1]), o.get_state(), what=f"filter {i} of 65536")


# ---- kernel variants and the streaming calls ------------------------------------------------------

@pytest.mark.parametrize("kernel", ["fast", "thread", "warp"])
def test_pose_kernels_agree_with_the_oracle(Ukf, kernel, monkeypatch):
    """UKFB_KERNEL selects the step kernel at ukfb_create: 'fast' (default, ukf_pose_fast.cuh), 'thread' (literal
    lane-per-filter, ukf_thread.cuh), 'warp' (literal warp-per-group, ukf_device.cuh).  All three against the oracle
    on the C3 schedule plus one update of every kind."""
    monkeypatch.setenv("UKFB_KERNEL", kernel)
    B = 77
    g, o = both(Ukf, 0, B)
    for x in (g, o):
        P.run_pose_c3(x, B, 30)
        for kind in range(9):
            z, R = syn.pose_measurement(kind, B, 40 + kind)
            x.step(0.02, kind, z, R)
    P.assert_parity(0, g.get_state(), o.get_state(), what=f"kernel={kernel}")
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())
    assert not g.get_status().any()


def test_pose_fast_kernel_fallback_lanes(Ukf):
    """lanes that leave the polynomial ranges / the selector-update guard run the literal code inside the fast kernel"""
    B = 64
    mu, sg = syn.pose_initial(B)
    sg[0::4, 3:6, 3:6] *= 150.0
    sg[1::4, 3:6, 3:6] *= 400.0  # trace 12: the out-of-line column check keeps the structured update
    sg[3::4, 5, 5] = 3.13**2  # a factor column next to pi: the literal update
    mu[2::4, 10:13] = [3.0, -40.0, 25.0]
    g, o = Ukf(0, B), OracleBatch(0, B)
    for x in (g, o):
        x.initialize(mu, sg)
        for k, kind in enumerate([8, 4, 0, 7, 3]):
            z, R = syn.pose_measurement(kind, B, k + 1)
            x.step(0.05, kind, z, R)
    assert np.array_equal(g.get_status(), o.get_status())
    P.assert_parity(0, g.get_state(), o.get_state(), tol=1e-9, what="fast kernel fallback lanes")
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())


def test_orientation_fast_kernel_wide_attitude_lanes(Ukf):
    """OrientationUKF filters that barely know their attitude (0.7 ... 3 rad per axis, an unknown heading, a factor column
    at the branch cut) next to ordinary ones in the same warps: the any-angle instance of the structured code, the literal
    update for the last kind, all against the oracle with equal status and mean-pass histogram"""
    B = 96
    mu, sg = syn.orientation_initial(B)
    for start, sig in ((0, (0.7, 0.7, 0.7)), (1, (1.0, 1.0, 1.0)), (2, (2.0, 2.0, 2.0)), (3, (0.1, 0.1, 2.9)), (4, (3.0, 3.0, 3.0)),
                       (5, (0.1, 0.1, 3.13))):
        sg[start::8, 0:3, 0:3] = np.diag(np.square(sig))
    g, o = P.make_ori(Ukf, B), P.make_ori(OracleBatch, B)
    for x in (g, o):
        x.initialize(mu, sg)
        for k in range(1, 9):
            gyro, acc = syn.orientation_imu(B, k)
            x.set_rotation_rate(gyro)
            x.set_acceleration(acc)
            if k % 2 == 0:
                z, R = syn.orientation_velocity(B, k)
                x.step(0.01, 9, z, R)
            else:
                x.predict_dt(0.01)
    assert np.array_equal(g.get_status(), o.get_status()) and not o.get_status().any()
    P.assert_parity(1, g.get_state(), o.get_state(), tol=1e-9, what="orientation wide attitude lanes")
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())


@pytest.mark.parametrize("filt", [0, 1])
def test_unnormalised_quaternions_match_the_scale_invariant_log(Ukf, filt):
    """the fast kernels' reciprocal-free log assumes |q| = 1; states initialised with other norms run the literal code
    (the reference's log is scale invariant) and agree with the oracle"""
    B = 96
    mu, sg = syn.pose_initial(B) if filt == 0 else syn.orientation_initial(B)
    qs = slice(3, 7) if filt == 0 else slice(0, 4)
    mu[1::3, qs] *= 1.001
    mu[2::7, qs] *= 0.97
    g, o = Ukf(filt, B), OracleBatch(filt, B)
    for x in (g, o):
        if filt == 1:
            x.set_process_noise(syn.ORI_Q)
            x.set_orientation_params(syn.ORI_TAU, syn.ORI_TAU, syn.LATITUDE_BREMEN)
        x.initialize(mu, sg)
        if filt == 0:
            P.run_pose_c3(x, B, 20)
        else:
            P.run_ori_c1(x, B, 20, every=5)
    P.assert_parity(filt, g.get_state(), o.get_state(), tol=1e-9, what="unnormalised quaternions")
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())


@pytest.mark.parametrize("kernel", ["fast", "thread", "warp"])
def test_orientation_kernels_agree_with_the_oracle(Ukf, kernel, monkeypatch):
    """OrientationUKF through each step kernel ('fast' = ukf_ori_fast.cuh): IMU stream with velocity updates, finite
    bias time constants, fused steps."""
    monkeypatch.setenv("UKFB_KERNEL", kernel)
    B = 77
    g, o = Ukf(1, B), OracleBatch(1, B)
    mu, sg = syn.orientation_initial(B)
    for x in (g, o):
        x.set_orientation_params(60.0, 30.0, syn.LATITUDE_BREMEN)
        x.initialize(mu, sg)
        x.set_process_noise(syn.ORI_Q)
        P.run_ori_c1(x, B, 40, every=5)
        for k in range(41, 46):
            z, R = syn.orientation_velocity(B, k)
            x.step(0.02, 9, z, R)
    P.assert_parity(1, g.get_state(), o.get_state(), what=f"orientation kernel={kernel}")
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())
    assert not g.get_status().any()


def test_orientation_per_filter_parameters(Ukf):
    """one (gyro_bias_tau, acc_bias_tau, latitude) per filter, as separately constructed reference objects would have"""
    from test_emu_lane_kernels import _per_filter_orientation

    B = 200
    g, o = _per_filter_orientation(Ukf, B), _per_filter_orientation(OracleBatch, B)
    P.assert_parity(1, g.get_state(), o.get_state(), what="per-filter tau / latitude")
    assert np.abs(g.get_rotation_rate() - o.get_rotation_rate()).max() < 1e-12


def test_orientation_fast_kernel_fallback_lanes(Ukf):
    """lanes that leave the polynomial ranges / the update guard run the literal code inside ukf_ori_fast_kernel"""
    B = 64
    mu, sg = syn.orientation_initial(B)
    sg[0::4, 0:3, 0:3] *= 150.0
    sg[1::4, 0:3, 0:3] *= 400.0
    gyro = np.tile([0.0, 0.0, 0.05], (B, 1))
    gyro[2::4] = [3.0, -40.0, 25.0]
    g, o = P.make_ori(Ukf, B), P.make_ori(OracleBatch, B)
    for x in (g, o):
        x.initialize(mu, sg)
        for k in range(1, 4):
            x.set_rotation_rate(gyro)
            x.set_acceleration(syn.orientation_imu(B, k)[1])
            z, R = syn.orientation_velocity(B, k)
            x.step(0.05, 9, z, R)
    assert np.array_equal(g.get_status(), o.get_status())
    P.assert_parity(1, g.get_state(), o.get_state(), tol=1e-9, what="orientation fast kernel fallback lanes")
    assert np.array_equal(g.get_mean_iter_hist(), o.get_mean_iter_hist())


def test_orientation_run_dev_imu_stream(Ukf):
    """K ticks per launch with the IMU stream stored before each predict and a velocity update on the last tick"""
    import torch

    B, K, rounds = 40, 25, 4
    g, o = P.make_ori(Ukf, B), P.make_ori(OracleBatch, B)
    dev = torch.device("cuda:0")
    d_dt = torch.full((K,), syn.DT, dtype=torch.float64, device=dev)
    kinds = np.full(K, -1, np.int8)
    kinds[K - 1] = 9
    for c in range(rounds):
        imu = np.empty((K, B, 6))
        for j in range(K):
            imu[j, :, :3], imu[j, :, 3:] = syn.orientation_imu(B, c * K + j + 1)
        z, R = syn.orientation_velocity(B, c + 1)
        zs = np.zeros((K, B, 3))
        zs[K - 1] = z
        g.run_dev(K, d_dt, False, kinds, torch.from_numpy(zs).to(dev), torch.from_numpy(np.tile(R, (K, 1, 1))).to(dev), False,
                  torch.from_numpy(imu).to(dev))
        g.synchronize()
        for j in range(K):
            o.set_rotation_rate(imu[j, :, :3])
            o.set_acceleration(imu[j, :, 3:])
            o.predict_dt(syn.DT)
        o.update(9, z, R)
    P.assert_parity(1, g.get_state(), o.get_state(), what="orientation run_dev")
    assert np.abs(g.get_rotation_rate() - o.get_rotation_rate()).max() < 1e-12


def test_streaming_calls_match_the_blocking_ones(Ukf):
    import torch

    B, steps = 5000, 7
    a, b = P.make_pose(Ukf, B), P.make_pose(Ukf, B)
    zs = [torch.from_numpy(syn.pose_measurement(8, B, k + 1)[0]).pin_memory() for k in range(steps)]
    R = np.eye(3) * syn.SIGMA_GYRO**2
    outs = [torch.empty((B, 13), dtype=torch.float64).pin_memory() for _ in range(steps)]
    sig = torch.empty((B, 12, 12), dtype=torch.float64).pin_memory()
    want = []
    for k in range(steps):
        a.step(syn.DT, 8, zs[k].numpy(), R)
        want.append(a.get_state()[0])
    for k in range(steps):
        b.step_async(syn.DT, 8, zs[k].numpy(), R)
        b.get_state_async(outs[k].numpy(), sig.numpy() if k == steps - 1 else None)
    b.synchronize()
    for k in range(steps):
        assert np.array_equal(outs[k].numpy(), want[k]), f"streamed estimates of step {k} differ"
    assert np.array_equal(sig.numpy(), a.get_state()[1])
    # mixing blocking calls after streamed ones keeps the order
    b.step(syn.DT, 8, zs[0].numpy(), R)
    a.step(syn.DT, 8, zs[0].numpy(), R)
    assert np.array_equal(a.get_state()[0], b.get_state()[0])


@pytest.mark.parametrize("devices", [None, [0, 0, 0]])
def test_streaming_calls_match_the_blocking_ones_over_every_staged_layout(Ukf, devices):
    """step_async / get_state_async / get_mu_range_async against their blocking twins on a second handle, bit for bit,
    over every set of arrays a call stages: dt broadcast or per filter; no measurement, a broadcast R, a per-filter R or
    the R kept by set_measurement_cov (cov=None); with and without a mask; mu alone, mu and sigma, or a range of mu.
    36 000 filters, 12 000 per shard on three: the third step lands in the input slot of the first (dt alone, 1 MiB) and
    needs more (97 bytes per filter with a per-filter R and a mask), the third read-back (sigma) in the output slot of
    the first (a range of mu), so both slots grow between pipelined calls."""
    import torch

    B = 36000
    rng = np.random.default_rng(11)
    keep = []

    def pinned(x):
        t = torch.from_numpy(np.ascontiguousarray(x)).pin_memory()
        keep.append(t)
        return t.numpy()

    a, b = P.make_pose(Ukf, B), P.make_pose(Ukf, B, devices=devices)
    kept_R = syn.pose_measurement(0, B, 1)[1] * rng.uniform(0.5, 2.0, (B, 1, 1))
    for x in (a, b):
        x.set_measurement_cov(0, kept_R)
    # (dt per filter, measurement, mask): the 14 combinations, starting with the ones that make the slots grow
    seq = [(False, "none", False), (True, "per", True), (False, "per", True), (True, "bcast", False), (False, "kept", True),
           (True, "none", False), (False, "bcast", True), (True, "kept", False), (False, "per", False), (True, "bcast", True),
           (False, "kept", False), (True, "per", False), (True, "kept", True), (False, "bcast", False)]
    assert len(set(seq)) == 14
    want, got = [], []
    for k, (dt_per, meas, masked) in enumerate(seq):
        dt = pinned(syn.DT * rng.uniform(0.5, 1.5, B)) if dt_per else syn.DT
        kind, mu, cov = -1, None, None
        if meas == "bcast":
            kind = 8
            mu, cov = syn.pose_measurement(kind, B, k + 1)
        elif meas == "per":
            kind = 4
            mu, R = syn.pose_measurement(kind, B, k + 1)
            cov = pinned(R * rng.uniform(0.5, 2.0, (B, 1, 1)))
        elif meas == "kept":
            kind = 0
            mu = syn.pose_measurement(kind, B, k + 1)[0]
        mu = pinned(mu) if mu is not None else None
        mask = pinned(rng.integers(0, 2, B, dtype=np.uint8)) if masked else None
        a.step(dt, kind, mu, cov, mask)
        b.step_async(dt, kind, mu, cov, mask)
        if k % 3 == 0:
            want.append((a.get_mu_range(0, 7),))
            got.append((pinned(np.empty((B, 7))),))
            b.get_mu_range_async(0, 7, *got[-1])
        elif k % 3 == 1:
            want.append((a.get_state(with_sigma=False),))
            got.append((pinned(np.empty((B, 13))),))
            b.get_state_async(*got[-1])
        else:
            want.append(a.get_state())
            got.append((pinned(np.empty((B, 13))), pinned(np.empty((B, 12, 12)))))
            b.get_state_async(*got[-1])
    b.synchronize()
    for k, (w, g) in enumerate(zip(want, got)):
        for wi, gi in zip(w, g):
            assert np.array_equal(gi, wi), f"step {k} {seq[k]}: streamed read-back differs from the blocking one"


@pytest.mark.gpu
def test_fast_kernel_not_spd_deferral_is_one_factorisation():
    """see tests/test_emu_lane_kernels.py::check_not_spd_deferral: the documented one-step deferral, on the device"""
    from slam_pose_estimation_b200 import UkfBatch
    from test_emu_lane_kernels import check_not_spd_deferral

    check_not_spd_deferral(UkfBatch, {})


@pytest.mark.parametrize("filt", [0, 1])
def test_overlapped_launches_equal_launches_in_stream_order(Ukf, filt):
    """A handle whose batch is a few waves of warps orders its step launches tile by tile (launch n starts in the slots
    the last wave of launch n - 1 leaves empty: include/ukf_batch.h, ukfb_overlapped_launch_count).  64 Ki filters are 1.7
    waves on a B200; its four quarters, one handle each, are less than half a wave and launch in plain stream order.  Same
    device inputs, launches back to back: the results must be equal bit for bit, and match the oracle on a sample."""
    import torch

    B, H, K = 65536, 16384, 12
    dev = torch.device("cuda", 0)
    mu, sg = syn.pose_initial(B) if filt == 0 else syn.orientation_initial(B)
    whole, halves = Ukf(filt, B), [Ukf(filt, H) for _ in range(B // H)]
    objs = [(whole, slice(0, B))] + [(h, slice(i * H, (i + 1) * H)) for i, h in enumerate(halves)]
    d_dt = torch.full((1,), syn.DT, dtype=torch.float64, device=dev)
    for x, sl in objs:
        x.initialize(mu[sl], sg[sl])
        if filt == 1:
            x.set_process_noise(syn.ORI_Q)
            x.set_orientation_params(syn.ORI_TAU, syn.ORI_TAU, syn.LATITUDE_BREMEN)
    if filt == 0:
        zs = [syn.pose_measurement(8, B, k + 1) for k in range(K)]
        for x, sl in objs:
            d_z = [torch.from_numpy(np.ascontiguousarray(z[sl])).to(dev) for z, _ in zs]
            d_R = torch.from_numpy(zs[0][1]).to(dev)
            torch.cuda.synchronize()
            for k in range(K):  # nothing but step launches in the stream
                x.step_dev(d_dt, False, 8, d_z[k], d_R, False)
            x.synchronize()
    else:
        imu = np.stack([np.concatenate(syn.orientation_imu(B, k + 1), axis=1) for k in range(K)])  # K x B x 6
        for x, sl in objs:
            d_imu = torch.from_numpy(np.ascontiguousarray(imu[:, sl])).to(dev)
            torch.cuda.synchronize()
            d_dt3 = torch.full((3,), syn.DT, dtype=torch.float64, device=dev)
            for k in range(0, K, 3):  # launches of three ticks each
                x.run_dev(3, d_dt3, False, d_imu=d_imu[k:k + 3])
            x.synchronize()
    n_launches = K if filt == 0 else K // 3
    assert whole.overlapped_launch_count() == n_launches, "the 64 Ki handle did not overlap its launches (not a B200?)"
    assert halves[0].overlapped_launch_count() == 0
    m, s = whole.get_state()
    for h, (_, sl) in zip(halves, objs[1:]):
        mh, sh = h.get_state()
        assert np.array_equal(m[sl], mh) and np.array_equal(s[sl], sh)
    assert not whole.get_status().any()
    idx = np.arange(0, B, B // 16)
    o = OracleBatch(filt, idx.size)
    o.initialize(mu[idx], sg[idx])
    if filt == 0:
        for k in range(K):
            o.step(syn.DT, 8, zs[k][0][idx], zs[k][1])
    else:
        o.set_process_noise(syn.ORI_Q)
        o.set_orientation_params(syn.ORI_TAU, syn.ORI_TAU, syn.LATITUDE_BREMEN)
        for k in range(K):
            o.set_rotation_rate(imu[k, idx, 0:3])
            o.set_acceleration(imu[k, idx, 3:6])
            o.predict_dt(syn.DT)
    P.assert_parity(filt, (m[idx], s[idx]), o.get_state(), what="overlapped launches")


def test_overlapped_launches_with_other_stream_work_in_between(Ukf):
    """The same question on 128 Ki PoseUKF filters (3.5 waves: what one GPU holds of the 1 Mi batch sharded over eight), 30
    launches, and with everything else a caller puts into the stream between two steps -- a field readback on the device,
    a stored acceleration (its own small kernel), a status summary -- each of which is a full ordering point that the
    overlapped launches before and after it have to respect.  Reference: eight handles of 16 Ki filters (under one wave:
    plain stream order) given the same calls."""
    import torch

    B, H, K = 131072, 16384, 30
    dev = torch.device("cuda", 0)
    mu, sg = syn.pose_initial(B)
    whole, parts = Ukf(0, B), [Ukf(0, H) for _ in range(B // H)]
    objs = [(whole, slice(0, B))] + [(h, slice(i * H, (i + 1) * H)) for i, h in enumerate(parts)]
    d_dt = torch.full((1,), syn.DT, dtype=torch.float64, device=dev)
    zs = [syn.pose_measurement(8, B, k + 1)[0] for k in range(4)]
    R = syn.pose_measurement(8, B, 1)[1]
    acc = np.tile([0.02, -0.01, 0.03], (B, 1))
    reads = {}
    for x, sl in objs:
        n = sl.stop - sl.start
        x.initialize(mu[sl], sg[sl])
        d_z = [torch.from_numpy(np.ascontiguousarray(z[sl])).to(dev) for z in zs]
        d_R = torch.from_numpy(R).to(dev)
        d_pose = torch.empty((n, 7), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        got = []
        for k in range(K):
            x.step_dev(d_dt, False, 8, d_z[k % 4], d_R, False)
            if k % 7 == 3:
                x.get_mu_range_dev(0, 7, d_pose)  # unpack kernel on the handle's stream
                x.synchronize()
                got.append(d_pose.cpu().numpy().copy())
            if k == 11:
                x.set_acceleration(acc[sl], np.eye(3) * 1e-4)  # host-pointer call: copy + store kernel; the next predicts use it
            if k == 20:
                got.append(np.array(x.status_summary()))
        x.synchronize()
        reads[sl.start, n] = got
    assert whole.overlapped_launch_count() == K and parts[0].overlapped_launch_count() == 0
    m, s = whole.get_state()
    for h, (_, sl) in zip(parts, objs[1:]):
        mh, sh = h.get_state()
        assert np.array_equal(m[sl], mh) and np.array_equal(s[sl], sh)
        for a, b in zip(reads[0, B], reads[sl.start, H]):
            if a.ndim == 2:
                assert np.array_equal(a[sl], b), "a readback between two overlapped launches saw another state"
    assert not whole.get_status().any()
