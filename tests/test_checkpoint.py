"""Checkpoint and restore of a whole batch (include/ukf_batch.h, "checkpoint / restore").

A job stopped after k ticks and resumed from its image must continue exactly as the job that was never stopped: bit
for bit, for both filter kinds, with every part of a filter's state in use (a stored PoseUKF acceleration on some
filters and the NaN sentinel on others, an OrientationUKF IMU stream, per-filter and broadcast Q, per-filter
orientation parameters, kept measurement covariances, a finite gate, non-default time bounds, flagged filters).  The
image does not depend on the shard count or the kernel family, is in stream order with the pipelined calls, rolls a
batch back on the device, and a rejected image changes nothing."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import parity as P
from oracle.oracle_lib import OracleBatch
from slam_pose_estimation_b200 import _build, synthetic as syn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NOT_SPD = 8
HEADER = 768
FAILED = np.array([3, 40, 41, 150])  # given a covariance that is not positive definite: NOT_SPD from their next predict


def device_lists():
    import torch

    n = torch.cuda.device_count()
    return [[0, 0, 0]] + ([list(range(n))] if n >= 2 else [])


def _kw(devices):
    return {} if devices is None else {"devices": devices}


def _rng_q(n, B, seed):
    rng = np.random.default_rng(seed)
    d = np.abs(rng.standard_normal((B, n))) * 1e-3 + 1e-4
    return np.stack([np.diag(r) for r in d])


def setup(kind, B, per_filter_q, devices=None, cls=None):
    """a batch with every handle-wide setting away from its default"""
    from slam_pose_estimation_b200 import UkfBatch

    cls = cls or UkfBatch
    x = (P.make_pose if kind == 0 else P.make_ori)(cls, B, **_kw(devices))
    x.set_time_bounds(1e-7, 0.5)
    x.set_mahalanobis_gate(400.0)
    n = 12 if kind == 0 else 13
    if per_filter_q:
        x.set_process_noise(_rng_q(n, B, 1 + kind))
    elif kind == 0:
        x.set_process_noise(np.diag(np.repeat([2e-3, 1e-4, 5e-3, 1e-4], 3)))  # broadcast, diagonal, not the default
    if kind == 0:
        acc = 0.2 * syn.noise(np.arange(B), 1, 30, 3)
        x.set_acceleration(acc, np.eye(3) * 1e-3, mask=(np.arange(B) % 3 == 0).astype(np.uint8))  # the rest keep NaN
        x.set_measurement_cov(4, np.eye(3) * syn.SIGMA_DVL ** 2)                                 # broadcast
        x.set_measurement_cov(8, np.tile(np.eye(3) * syn.SIGMA_GYRO ** 2, (B, 1, 1)) * (1 + np.arange(B))[:, None, None] / B)
    else:
        x.set_orientation_params(syn.ORI_TAU * (1 + 0.01 * np.arange(B)), syn.ORI_TAU, syn.LATITUDE_BREMEN + 1e-3 * np.arange(B))
        x.set_measurement_cov(9, np.tile(np.eye(3) * syn.SIGMA_DVL ** 2, (B, 1, 1)))           # per filter
    return x


def fail_some(x, kind):
    mu, sg = x.get_state_indexed(FAILED)
    sg[:, 0, 0] = -1.0
    x.initialize_indexed(FAILED, mu, sg)


def _ori_events(B, k):
    """one tick of an OrientationUKF sensor stream: rotation rate and acceleration at t_k, a velocity every 4th tick"""
    t = syn.T0_US + 1000 * k
    gyro, acc = syn.orientation_imu(B, k)
    z, _ = syn.orientation_velocity(B, k)
    ts = np.array([np.full(B, t), np.full(B, t), np.full(B, t + 300)], np.int64)
    kinds = np.array([np.full(B, 11), np.full(B, 12), np.full(B, 9 if k % 4 == 0 else -2)], np.int8)
    return ts, kinds, np.stack([gyro, acc, z])


def ticks(x, kind, B, start, count, pipelined=False):
    """the history: PoseUKF C3 ticks with kept covariances; OrientationUKF event streams plus kept-covariance updates"""
    for k in range(start, start + count):
        if kind == 0:
            z, _ = syn.pose_measurement(8, B, k)
            (x.step_async if pipelined else x.step)(syn.DT, 8, z, None)  # the kept per-filter covariance
            if k % 5 == 0:
                z, _ = syn.pose_measurement(4, B, k)
                (x.step_async if pipelined else x.step)(syn.DT, 4, z, None)
        else:
            ts, kinds, mu3 = _ori_events(B, k)
            (x.run_events_async if pipelined else x.run_events)(ts, kinds, mu3, syn.sensor_cov_table())
            if not pipelined and k % 7 == 0:
                z, _ = syn.orientation_velocity(B, k)
                x.update(9, z, None)


def observe(x, kind):
    """everything the public API reads back"""
    mu, sg = x.get_state()
    out = {"mu": mu, "sigma": sg, "status": x.get_status(), "t_last": x.get_last_time(),
           "Q": x.get_process_noise(per_filter=True), "hist": x.get_mean_iter_hist(), "bounds": np.array(x.get_time_bounds()),
           "gate": np.array([x.get_mahalanobis_gate()]), "init": np.array([x.is_initialized()])}
    if kind == 1:
        out["rate"] = x.get_rotation_rate()
    return out


def assert_same(a, b, kind, what):
    oa, ob = observe(a, kind), observe(b, kind)
    for k in oa:
        assert np.array_equal(oa[k].view(np.uint8), ob[k].view(np.uint8)), f"{what}: {k} differs"
    assert np.array_equal(a.checkpoint(), b.checkpoint()), f"{what}: images differ"


def payload_bytes(kind, B, per_filter_q):
    """the sections of setup()'s batch: 860 / 972 bytes per filter, + 624 / 728 with per-filter Q, + 40 with per-filter
    orientation parameters (OrientationUKF here), + its kept covariances (PoseUKF: kind 4 broadcast, kind 8 per filter;
    OrientationUKF: kind 9 per filter), + Q once when broadcast"""
    per = (860 if kind == 0 else 972) + (per_filter_q and (624 if kind == 0 else 728)) + (0 if kind == 0 else 40) + 72
    once = (72 if kind == 0 else 0) + (0 if per_filter_q else (624 if kind == 0 else 728))
    return B * per + once


@pytest.mark.gpu
@pytest.mark.parametrize("per_filter_q", [False, True])
@pytest.mark.parametrize("kind", [0, 1])
def test_resume_equals_uninterrupted(kind, per_filter_q):
    from slam_pose_estimation_b200 import UkfBatch

    B, k = 203, 12
    a = setup(kind, B, per_filter_q)
    ticks(a, kind, B, 1, k)
    fail_some(a, kind)
    ticks(a, kind, B, 1 + k, 3)
    assert (a.get_status()[FAILED] & NOT_SPD).all()
    img = a.checkpoint()
    size = a.checkpoint_size()
    assert img.dtype == np.uint8 and img.size == size
    assert HEADER + payload_bytes(kind, B, per_filter_q) <= size <= HEADER + payload_bytes(kind, B, per_filter_q) + 256 * 18
    r = UkfBatch(kind, B)  # never initialized
    assert not r.is_initialized()
    r.restore(img)
    assert_same(a, r, kind, "right after the restore")
    assert np.array_equal(r.checkpoint(), img)
    for x in (a, r):
        ticks(x, kind, B, 4 + k, k)
    assert_same(a, r, kind, "after more ticks")
    if kind == 1:  # initialize does not apply the constructor's IMU defaults to a restored handle
        mu, sg = syn.orientation_initial(B)
        for x in (a, r):
            x.initialize(mu, sg)
            ticks(x, kind, B, 100, 2)
        assert_same(a, r, kind, "after a later initialize")
    shifted = np.empty(img.size + 1, np.uint8)[1:]  # an image at an odd address: the restore may not assume alignment
    shifted[:] = img
    for src in (bytes(img), bytearray(img), shifted):
        r.restore(src)
        assert np.array_equal(r.checkpoint(), img)


@pytest.mark.gpu
def test_resume_without_the_stored_acceleration_would_differ():
    """what the image adds over the old getters: restoring only mu, sigma, Q and t_last loses the stored acceleration
    and the next predictions take the other branch of PoseUKF.cpp:188-192"""
    from slam_pose_estimation_b200 import UkfBatch

    B = 96
    a = setup(0, B, False)
    ticks(a, 0, B, 1, 4)
    mu, sg = a.get_state()
    r, old = UkfBatch(0, B), UkfBatch(0, B)
    r.restore(a.checkpoint())
    old.initialize(mu, sg)
    old.set_process_noise(a.get_process_noise())
    old.set_last_time(a.get_last_time())
    for x in (a, r, old):
        x.set_mahalanobis_gate(400.0)
        x.predict_dt(syn.DT)
    assert np.array_equal(a.get_state()[0], r.get_state()[0])
    moved = np.any(a.get_state()[0] != old.get_state()[0], axis=1)
    assert moved[::3].all() and not moved[1::3].any()  # exactly the filters with a stored acceleration


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_image_does_not_depend_on_the_shard_count(kind):
    from slam_pose_estimation_b200 import UkfBatch

    B, k = 203, 8
    one = setup(kind, B, kind == 0)
    ticks(one, kind, B, 1, k)
    fail_some(one, kind)
    ticks(one, kind, B, 1 + k, 2)
    img = one.checkpoint()
    for devs in device_lists():
        sh = setup(kind, B, kind == 0, devices=devs)
        ticks(sh, kind, B, 1, k)
        fail_some(sh, kind)
        ticks(sh, kind, B, 1 + k, 2)
        assert np.array_equal(sh.checkpoint(), img), f"{devs}: a sharded handle's image differs"
        for dst_devs, src in ((devs, img), (None, sh.checkpoint())):  # 1 -> n and n -> 1
            r = UkfBatch(kind, B, **_kw(dst_devs))
            r.restore(src)
            assert np.array_equal(r.checkpoint(), img), f"{devs} -> {dst_devs}: re-saved image differs"
        r = UkfBatch(kind, B, devices=devs)
        r.restore(img)
        for x in (one, r):
            ticks(x, kind, B, 3 + k, 6)
        assert_same(one, r, kind, f"restored onto {devs}")
        one.restore(img)  # back to the saved point for the next device list


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["thread", "warp"])
@pytest.mark.parametrize("kind", [0, 1])
def test_image_moves_between_kernel_families(kind, family, monkeypatch):
    """an image of the fast kernels restores into a literal-kernel handle (other record layout for warp), re-saves to the
    same bytes, and the continuation agrees with the oracle"""
    from slam_pose_estimation_b200 import UkfBatch

    B = 203
    g, o = (P.make_pose if kind == 0 else P.make_ori)(UkfBatch, B), (P.make_pose if kind == 0 else P.make_ori)(OracleBatch, B)
    if kind == 0:
        acc = 0.2 * syn.noise(np.arange(B), 1, 30, 3)
        mask = (np.arange(B) % 3 == 0).astype(np.uint8)
        for x in (g, o):
            x.set_acceleration(acc, np.eye(3) * 1e-3, mask=mask)
            P.run_pose_c3(x, B, 10)
    else:
        for x in (g, o):
            P.run_ori_c1(x, B, 10, every=5)
    img = g.checkpoint()
    monkeypatch.setenv("UKFB_KERNEL", family)
    r = UkfBatch(kind, B)
    monkeypatch.delenv("UKFB_KERNEL")
    r.restore(img)
    assert np.array_equal(r.checkpoint(), img)
    for x in (r, o):
        if kind == 0:
            P.run_pose_c3(x, B, 20, start=11)
        else:
            P.run_ori_c1(x, B, 20, start=11, every=5)
    P.assert_parity(kind, r.get_state(), o.get_state(), what=f"fast image continued by the {family} kernel")
    assert np.array_equal(r.get_last_time(), o.get_last_time())


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_stream_order_with_pipelined_calls(kind):
    """64 Ki filters, where consecutive step launches overlap tile by tile: a save issued right after the _async calls
    equals one taken after synchronize, and a restore followed by _async calls continues the uninterrupted run"""
    from slam_pose_estimation_b200 import UkfBatch

    B = 64 * 1024
    a, b = setup(kind, B, False), setup(kind, B, False)
    for x in (a, b):
        ticks(x, kind, B, 1, 3)
    ticks(a, kind, B, 4, 4, pipelined=True)
    img_now = a.checkpoint()  # no synchronize before it
    ticks(b, kind, B, 4, 4, pipelined=True)
    b.synchronize()
    assert np.array_equal(img_now, b.checkpoint())
    r = UkfBatch(kind, B)
    r.restore(img_now)
    ticks(r, kind, B, 8, 4, pipelined=True)
    ticks(a, kind, B, 8, 4, pipelined=True)
    r.synchronize()
    a.synchronize()
    assert_same(a, r, kind, "pipelined continuation")
    if os.environ.get("UKFB_KERNEL", "fast") == "fast" and os.environ.get("UKFB_OVERLAP_LAUNCHES", "1") != "0":
        assert a.overlapped_launch_count() > 0 and r.overlapped_launch_count() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_device_snapshot_rolls_back(kind):
    import torch

    B = 203
    x, y = setup(kind, B, kind == 1), setup(kind, B, kind == 1)
    for h in (x, y):
        ticks(h, kind, B, 1, 5)
    snap = x.checkpoint_dev()
    assert snap.device.type == "cuda" and snap.dtype == torch.uint8
    assert np.array_equal(snap.cpu().numpy(), x.checkpoint())
    ticks(x, kind, B, 6, 6)  # a speculative block
    assert not np.array_equal(x.checkpoint(), y.checkpoint())
    x.restore_dev(snap)
    assert np.array_equal(x.checkpoint(), y.checkpoint())
    ticks(x, kind, B, 6, 6)  # the same block again
    ticks(y, kind, B, 6, 6)
    assert_same(x, y, kind, "rolled back and re-applied")
    out = torch.zeros(x.checkpoint_size() + 100, dtype=torch.uint8, device="cuda")
    x.checkpoint_dev(out)
    assert np.array_equal(out[: x.checkpoint_size()].cpu().numpy(), x.checkpoint())


def _patched(img, at, value, dtype):
    bad = img.copy()
    bad[at: at + np.dtype(dtype).itemsize] = np.array([value], dtype).view(np.uint8)
    return bad


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 0, 0]])
def test_rejected_images_change_nothing(devices):
    import torch

    from slam_pose_estimation_b200 import UkfBatch, UkfbError

    B = 203
    x = setup(0, B, True, devices=devices)
    ticks(x, 0, B, 1, 4)
    fail_some(x, 0)
    ticks(x, 0, B, 5, 2)
    img = x.checkpoint()
    other_kind = setup(1, B, False)
    other_size = setup(0, B + 1, True)
    sec1_bytes = 256 + 24 * 1 + 16  # the bytes field of section 1 (t_last): table at 256, 24 bytes per entry
    bad = {
        "kind": other_kind.checkpoint(),
        "B": other_size.checkpoint(),
        "version": _patched(img, 8, 2, np.uint32),
        "magic": _patched(img, 0, 0x5A, np.uint8),
        "truncated": img[:-1],
        "header only": img[:HEADER],
        "short header": img[:100],
        "section size": _patched(img, sec1_bytes, B * 8 + 8, np.uint64),
        "mode": _patched(img, 192, 0, np.uint32),  # per-filter Q declared broadcast: the sections no longer match
    }
    for what, b in bad.items():
        with pytest.raises(UkfbError) as e:
            x.restore(b)
        assert e.value.code == -1, what
        assert np.array_equal(x.checkpoint(), img), f"{what}: the handle changed"
    lib = x.lib
    assert lib.ukfb_checkpoint_restore(x.h, None, img.size) == -1
    assert lib.ukfb_checkpoint_save(x.h, None, img.size) == -1
    small = np.zeros(img.size - 1, np.uint8)
    assert lib.ukfb_checkpoint_save(x.h, small.ctypes.data_as(C.c_void_p), small.size) == -1
    assert not small.any()
    if devices is not None:
        for call in (lambda: x.checkpoint_dev(), lambda: x.restore_dev(torch.as_tensor(img, device="cuda"))):
            with pytest.raises(UkfbError) as e:
                call()
            assert e.value.code == -1
    else:
        d = torch.as_tensor(_patched(img, 8, 2, np.uint32), device="cuda")
        with pytest.raises(UkfbError) as e:
            x.restore_dev(d)
        assert e.value.code == -1
        with pytest.raises(UkfbError):
            x.restore_dev(torch.as_tensor(img[:-1], device="cuda"))
        assert lib.ukfb_checkpoint_save_dev(x.h, C.c_void_p(d.data_ptr()), d.numel() - 1) == -1
    assert np.array_equal(x.checkpoint(), img)
    fresh = UkfBatch(0, 40, **_kw(devices))
    with pytest.raises(UkfbError) as e:
        fresh.checkpoint()
    assert e.value.code == -2  # UKFB_ERR_NOT_INITIALIZED


# ---- C++ mirror: saveCheckpoint / restoreCheckpoint ------------------------------------------------------------------

@pytest.fixture(scope="module")
def checkpoint_demo(tmp_path_factory):
    _build.build()
    exe = str(tmp_path_factory.mktemp("cpp") / "checkpoint_demo")
    libdir = os.path.dirname(_build.LIB)
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "checkpoint_demo.cpp"), "-L", libdir, "-lukfb", f"-Wl,-rpath,{libdir}",
                    "-o", exe], check=True)
    return exe


def test_checkpoint_demo_compiles_and_fails_loudly_without_gpu(checkpoint_demo):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([checkpoint_demo, "64"], capture_output=True, text=True)
    assert r.returncode != 0 and ("no CPU path" in r.stderr or "CUDA" in r.stderr)


@pytest.mark.gpu
def test_cpp_checkpoint_through_the_batch_object(checkpoint_demo):
    B = 64
    r = subprocess.run([checkpoint_demo, str(B)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[0].startswith("image_bytes ") and int(lines[0].split()[1]) >= HEADER + B * 860
    assert lines[1] == "resaved_equal 1" and lines[2] == "states_equal 1"
