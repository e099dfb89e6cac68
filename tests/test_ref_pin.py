"""Pinning the oracle on the reference's own text.

oracle/_ref/libref.so (oracle/ref_recipe.mk) is the reference's PoseUKF.cpp, OrientationUKF.cpp and
UnscentedKalmanFilter.hpp compiled UNMODIFIED from /root/reference against stand-in dependency headers (oracle/ref_shim).

  layer                                                        in oracle/_ref            checked here
  L2 shell: guards, time latch, init (UnscentedKalmanFilter.hpp) REFERENCE TEXT           oracle == _ref, bit for bit
  L3 PoseUKF / OrientationUKF: models, Q shaping, quirks        REFERENCE TEXT           oracle == _ref, bit for bit
  L1 ukfom::ukf, MTK SO(3) / vect, Eigen arithmetic             restatement (App. A)     NOT pinned: still a recollection
                                                                                          of the un-vendored slam/mtk

So a green run means: everything the reference tree itself contains on the hot path is reproduced exactly by the oracle
(and, through the committed fixtures, by the CUDA engine at 1e-9); the engine underneath remains pinned only by the
independent NumPy restatement and the analytic known answers of tests/test_oracle.py.

The reference's sources are not part of this repository.  Where _ref is built, the live comparisons run and the
fixtures tests/golden/ref_*.npz (made by tests/golden/make_ref_golden.py from _ref) are checked against a fresh _ref;
everywhere else the fixtures stand in for it: the oracle must reproduce them bit for bit, and the quirks are checked on
the oracle alone."""
from __future__ import annotations

import importlib.util
import os

import numpy as np
import pytest

import parity as P
from oracle import oracle_lib as O
from oracle.oracle_lib import OracleBatch
from slam_pose_estimation_b200 import synthetic as syn

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_ref_golden", os.path.join(HERE, "golden", "make_ref_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)
NAMES = sorted(G.SCENARIOS)


def have_ref() -> bool:
    try:
        return O.build_ref()
    except Exception:
        return False


HAVE_REF = have_ref()
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="oracle/_ref/libref.so absent and the reference's sources not here to build it")
# the oracle's quirk runs are compared with _ref's where it is built
VARIANTS = ("left", "ref") if HAVE_REF else ("left",)


def fixture(name):
    return np.load(os.path.join(HERE, "golden", name + ".npz"))


def same(a, b, kind):
    """bitwise: the oracle restates the same expressions in the same order as the reference text"""
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), f"{k} differs (max |d| = {np.nanmax(np.abs(a[k].astype(float) - b[k].astype(float)))})"


@needs_ref
def test_reference_sources_compile_unmodified_and_are_the_ones_hashed():
    """the recipe compiles the files where they lie; the hashes next to the library are those of the files there now"""
    assert os.path.exists(O.REF_LIB)
    listed = open(os.path.join(os.path.dirname(O.REF_LIB), "sources.sha256")).read().split("\n")
    names = [line.split()[-1] for line in listed if line.strip()]
    assert [os.path.basename(n) for n in names] == ["PoseUKF.cpp", "OrientationUKF.cpp", "UnscentedKalmanFilter.hpp"]
    if os.path.isdir(O.REF_ROOT):
        import hashlib
        for line in listed:
            if line.strip():
                digest, path = line.split()
                assert hashlib.sha256(open(path, "rb").read()).hexdigest() == digest
        # nothing of the reference is copied into the repo: the include directory is a link into /root/reference
        link = os.path.join(os.path.dirname(O.REF_LIB), "include", "pose_estimation")
        assert os.path.islink(link) and os.path.realpath(link) == os.path.realpath(os.path.join(O.REF_ROOT, "src"))


@pytest.mark.parametrize("name", NAMES)
def test_oracle_equals_the_reference_sources(name):
    """bit for bit: against _ref where it is built, else against _ref's committed outputs"""
    kind, B, script = G.SCENARIOS[name]
    o = G.make(OracleBatch, kind, B)
    script(o, B)
    if HAVE_REF:
        r = G.make(OracleBatch, kind, B, variant="ref")
        script(r, B)
        ref = G.outputs(r, kind)
    else:
        ref = fixture(name)
    same(G.outputs(o, kind), ref, kind)


def test_quirks_one_by_one():
    """each reference quirk SURVEY.md lists, isolated, shown to matter -- and oracle vs the reference text where _ref is
    built"""
    B = 6
    # (1) PoseUKF.cpp:188-193: with a finite acceleration the process noise is the UNROTATED, UNSCALED Q with
    #     block(6,6,3,3) = 2 acc.cov (the shadowing local), not delta * rotated Q
    Q = G.dense_spd(12, 5, 1e-3)
    acc, acov = 0.1 * syn.noise(np.arange(B), 2, 13, 3), G.dense_spd(3, 6, 2e-3)
    res = {}
    for variant in VARIANTS:
        x = P.make_pose(OracleBatch, B, variant=variant)
        x.set_process_noise(Q)
        x.predict_dt(0.01)
        plain = x.get_state()[1].copy()
        x.set_acceleration(acc, acov)
        x.predict_dt(0.01)
        res[variant] = (plain, x.get_state()[1].copy())
    assert all(np.array_equal(res["left"][0], res[v][0]) and np.array_equal(res["left"][1], res[v][1]) for v in VARIANTS)
    grow_plain = np.trace(res["left"][0][0]) - np.trace(syn.pose_initial(B, perturb=True)[1][0])
    grow_acc = np.trace(res["left"][1][0]) - np.trace(res["left"][0][0])
    assert grow_acc > 20 * grow_plain  # unscaled Q (1e-3 per entry) against 0.01 s x Q
    # (2) OrientationUKF.cpp:86: process noise scales with dt^2 -- doubling dt quadruples the added noise
    add = {}
    for variant in VARIANTS:
        for dt in (0.01, 0.02):
            x = P.make_ori(OracleBatch, 1, variant=variant)
            x.set_process_noise(np.eye(13) * 1e-2)
            s0 = x.get_state()[1][0, 12, 12]  # gravity: passes through the model, only noise is added
            x.predict_dt(dt)
            add[variant, dt] = x.get_state()[1][0, 12, 12] - s0
    assert all(add["left", 0.01] == add[v, 0.01] and add["left", 0.02] == add[v, 0.02] for v in VARIANTS)
    assert abs(add["left", 0.02] / add["left", 0.01] - 4.0) < 1e-9
    # (3) UnscentedKalmanFilter.hpp:86-97,110-122: first call latches only; dt <= min_dt neither predicts nor latches;
    #     dt > max_dt throws AFTER the latch moved; a negative dt throws without moving it
    for variant in VARIANTS:
        x = P.make_pose(OracleBatch, 2, variant=variant)
        x.set_time_bounds(1e-3, 0.5)
        m0 = x.get_state()[0].copy()
        t = lambda us: np.full(2, us, np.int64)
        x.predict_time(t(5_000_000))
        assert np.array_equal(x.get_state()[0], m0) and (x.get_last_time() == 5_000_000).all() and not x.get_status().any()
        x.predict_time(t(5_000_900))  # 0.9 ms <= min_dt
        assert np.array_equal(x.get_state()[0], m0) and (x.get_last_time() == 5_000_000).all() and not x.get_status().any()
        x.predict_time(t(4_000_000))  # backwards
        assert (x.get_status() == 1).all() and (x.get_last_time() == 5_000_000).all()
        x.predict_time(t(6_000_000))  # 1 s > max_dt
        assert (x.get_status() == 3).all() and (x.get_last_time() == 6_000_000).all() and np.array_equal(x.get_state()[0], m0)
        x.predict_time(t(6_010_000))
        assert not np.array_equal(x.get_state()[0], m0)
    # (4) PoseUKF never finite-checks a measurement (PoseUKF.cpp:112-173), OrientationUKF does (OrientationUKF.cpp:55,61,67)
    for variant in VARIANTS:
        p = P.make_pose(OracleBatch, 2, variant=variant)
        z = np.array([[np.nan, 0, 0], [0.0, 0, 0.05]])
        p.update(8, z, np.eye(3) * 1e-6)
        assert not (p.get_status() & 4).any() and np.isnan(p.get_state()[0][0]).any() and np.isfinite(p.get_state()[0][1]).all()
        q = P.make_ori(OracleBatch, 2, variant=variant)
        q.update(9, z, np.eye(3) * 1e-4)
        assert q.get_status().tolist() == [4, 0] and np.isfinite(q.get_state()[0]).all()


@needs_ref
@pytest.mark.parametrize("name", NAMES)
def test_fixtures_are_what_the_reference_sources_give(name):
    kind, B, script = G.SCENARIOS[name]
    r = G.make(OracleBatch, kind, B, variant="ref")
    script(r, B)
    fx = fixture(name)
    out = G.outputs(r, kind)
    for k in out:
        if out[k].dtype.kind == "f":
            assert np.allclose(out[k], fx[k], rtol=0, atol=1e-12 * max(1.0, np.nanmax(np.abs(fx[k]))), equal_nan=True), k
        else:
            assert np.array_equal(out[k], fx[k]), k


@pytest.mark.parametrize("name", NAMES)
def test_oracle_reproduces_the_reference_fixtures(name):
    """runs on any host: the committed outputs of the reference's own sources"""
    kind, B, script = G.SCENARIOS[name]
    fx = fixture(name)
    assert int(fx["kind"]) == kind and int(fx["B"]) == B and "PoseUKF.cpp" in str(fx["source_sha256"])
    o = G.make(OracleBatch, kind, B)
    script(o, B)
    P.assert_parity(kind, o.get_state(), (fx["mu"], fx["sigma"]), tol=1e-12, what=name)
    assert np.array_equal(o.get_status(), fx["status"]) and np.array_equal(o.get_last_time(), fx["last_time"])
    assert np.array_equal(o.get_mean_iter_hist(), fx["hist"])
    if kind == 1:
        assert np.abs(o.get_rotation_rate() - fx["rotation_rate"]).max() < 1e-15


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_engine_matches_the_reference_fixtures(name):
    """the CUDA engine, through the C ABI, against outputs of the reference's own sources (north-star tolerance)"""
    from slam_pose_estimation_b200 import UkfBatch

    kind, B, script = G.SCENARIOS[name]
    fx = fixture(name)
    g = G.make(UkfBatch, kind, B)
    script(g, B)
    P.assert_parity(kind, g.get_state(), (fx["mu"], fx["sigma"]), tol=P.TOL, what=name)
    assert np.array_equal(g.get_status(), fx["status"]) and np.array_equal(g.get_last_time(), fx["last_time"])
    if name != "ref_pose_quirks":  # that scenario re-initialises: the reference's fresh ukfom::ukf starts a new count, the
        assert np.array_equal(g.get_mean_iter_hist(), fx["hist"])  # engine's histogram is per handle
    if kind == 1:
        assert np.abs(g.get_rotation_rate() - fx["rotation_rate"]).max() < 1e-12
    assert g.launch_count() > 0
