"""Per-block accuracy against the extended-precision oracle.

TEST INFRASTRUCTURE.  tests/parity.py judges a state with two norm-wise numbers (the mean error over max(1, ||mu||_inf),
the covariance error over ||S||_F).  Both are dominated by the largest components, so a block that is small in
absolute terms (the orientation at UTM-scale positions, the bias and gravity variances of OrientationUKF) can be wrong
by many of its own standard deviations and still pass.  At UTM-scale positions the FP64 oracle itself is about 5e-8
standard deviations away from the exact result of its own algorithm, so 1e-9 against it decides nothing there.

Here every implementation, the FP64 oracle included, is compared with the same algorithm computed in long double
(oracle/build/liboracle_ld.so), and each block is judged on its own scale, in units of the reference filter's
standard deviations:
  mean:        |(x [-] x_ref)_i| / sqrt(S_ref[i,i])                  (orientation in tangent coordinates)
  covariance:  |S[i,j] - S_ref[i,j]| / sqrt(S_ref[i,i] S_ref[j,j])   (row i in the block, every column j)
each reduced by max over the block's rows and the batch.  An implementation passes a block when its error is at most
max(C * the FP64 oracle's error, F), and every error, the FP64 oracle's included, is below CAP.

The scenarios drive any object with the UkfBatch method names, like the scripts of tests/parity.py.
"""
from __future__ import annotations

import numpy as np

import parity as P
from slam_pose_estimation_b200 import synthetic as syn

C = 4.0  # an implementation may be this many times less accurate than the FP64 oracle ...
F = 1e-12  # ... or this far from the exact result, whichever is larger
CAP = 1e-6  # and no block of anyone, the FP64 oracle included, may be further off than this

BLOCKS = {
    0: (("position", 0, 3), ("orientation", 3, 6), ("velocity", 6, 9), ("angular_velocity", 9, 12)),
    1: (("orientation", 0, 3), ("velocity", 3, 6), ("gyro_bias", 6, 9), ("acc_bias", 9, 12), ("gravity", 12, 13)),
}

B = 33  # one full warp and a ragged lane
UTM = np.array([487_000.0, 5_880_000.0, 50.0])  # easting, northing, height of a UTM zone 32 fix (Bremen)


# ---- metric ----------------------------------------------------------------------------------------

def tangent_error(kind: int, mu: np.ndarray, mu_ref: np.ndarray) -> np.ndarray:
    """mu [-] mu_ref per filter and tangent coordinate (B x n): Euclidean differences, orientation as log(q q_ref^-1)"""
    rot = 3 if kind == 0 else 0
    dq = P._qlog(P._qmul(mu[:, rot:rot + 4], mu_ref[:, rot:rot + 4] * np.array([-1.0, -1.0, -1.0, 1.0])))
    rest = np.delete(mu - mu_ref, np.s_[rot:rot + 4], axis=1)
    return np.concatenate([rest[:, :rot], dq, rest[:, rot:]], axis=1)


def block_errors(kind: int, got, ref) -> dict:
    """{block: (mean error, covariance error)} in standard deviations of the reference state `ref`"""
    (mu, sg), (mu_r, sg_r) = got, ref
    sd = np.sqrt(np.einsum("bii->bi", sg_r))
    em = np.abs(tangent_error(kind, mu, mu_r)) / sd
    es = np.abs(sg - sg_r) / (sd[:, :, None] * sd[:, None, :])
    return {name: (float(em[:, a:b].max()), float(es[:, a:b, :].max())) for name, a, b in BLOCKS[kind]}


def judge(kind: int, got, fp64, ref) -> list:
    """rows (block, 'mean' | 'cov', err, err_fp64_oracle) of an implementation's result `got`, the FP64 oracle's `fp64`
    and the long-double oracle's `ref`"""
    e, e64 = block_errors(kind, got, ref), block_errors(kind, fp64, ref)
    return [(blk, what, e[blk][j], e64[blk][j]) for blk, _, _ in BLOCKS[kind] for j, what in enumerate(("mean", "cov"))]


def failures(rows) -> list:
    """the rows that break the acceptance rule, as text"""
    out = []
    for blk, what, err, e64 in rows:
        if not (np.isfinite(err) and np.isfinite(e64)) or err > max(C * e64, F) or err > CAP or e64 > CAP:
            out.append(f"{blk} {what}: {err:.2e} std (FP64 oracle {e64:.2e}, bound {max(C * e64, F):.2e}, cap {CAP:g})")
    return out


# ---- scenarios -------------------------------------------------------------------------------------

def _pose(cls, mu, sg, **kw):
    x = cls(0, mu.shape[0], **kw)
    x.initialize(mu, sg)
    return x


def _gps(kind: int, Bn: int, k: int, offset):
    """a GPS fix of `kind` (0: xyz, 1: xy, 2: z) with a per-filter offset (Bn x 3) added to the local-frame value"""
    z, R = syn.pose_measurement(kind, Bn, k)
    cols = {0: slice(0, 3), 1: slice(0, 2), 2: slice(2, 3)}[kind]
    return z + offset[:, cols], R


def p1(cls, **kw):
    """C3, 300 ticks"""
    x = P.make_pose(cls, B, **kw)
    P.run_pose_c3(x, B, 300)
    return x


def p2(cls, **kw):
    """P1 at UTM-scale positions: GPS kinds 0, 1 and 2 take turns every 100 ticks, each with the offset"""
    mu, sg = syn.pose_initial(B, perturb=True)
    mu[:, 0:3] += UTM
    x = _pose(cls, mu, sg, **kw)
    off = np.broadcast_to(UTM, (B, 3))
    for k in range(1, 301):
        x.step(syn.DT, 8, *syn.pose_measurement(8, B, k))
        if k % 10 == 0:
            x.update(4, *syn.pose_measurement(4, B, k))
        if k % 100 == 0:
            g = k // 100 - 1
            x.update(g, *_gps(g, B, k, off))
    return x


def p3(cls, **kw):
    """dead reckoning: position variance 1e4, velocity variance 1, 1000 ticks of dt 0.01 with angular-velocity updates
    only, then one position fix with R = 0.25 I (condition number about 1e8, a downdate of 4 to 5 digits)"""
    mu, sg = syn.pose_initial(B, perturb=True)
    sg[:, 0:3, 0:3] = np.eye(3) * 1e4
    sg[:, 6:9, 6:9] = np.eye(3)
    x = _pose(cls, mu, sg, **kw)
    for k in range(1, 1001):
        x.step(0.01, 8, *syn.pose_measurement(8, B, k))
    z, _ = syn.pose_measurement(0, B, 1000)
    x.update(0, z, np.eye(3) * 0.25)
    return x


def p4(cls, **kw):
    """an accurate velocity update (R = 1e-10 I, not the R = 0 deferral) between C3 ticks, then predicts: a nearly
    singular predicted covariance"""
    x = P.make_pose(cls, B, **kw)
    P.run_pose_c3(x, B, 50)
    z, _ = syn.pose_measurement(4, B, 50)
    x.update(4, z, np.eye(3) * 1e-10)
    for _ in range(50):
        x.predict_dt(syn.DT)
    return x


def dense_pose_cov(rho: float = 1 - 1e-6) -> np.ndarray:
    """a dense 12 x 12 PoseUKF covariance in which each velocity axis has correlation `rho` with its position axis"""
    sd9 = np.sqrt(np.array([1.0, 2.0, 0.5] + [0.01] * 3 + [0.01, 0.02, 0.03]))  # position, orientation, ang. velocity
    C9 = 0.7 * np.eye(9) + 0.3 * np.ones((9, 9))  # dense and well conditioned
    G = sd9[:, None] * C9 * sd9[None, :]
    # velocity = 0.1 position + e, with var(e) chosen for corr(position_i, velocity_i) = rho
    T = np.zeros((12, 12))
    T[0:3, 0:3] = np.eye(3)
    T[3:6, 3:6] = np.eye(3)
    T[6:9, 0:3] = 0.1 * np.eye(3)
    T[9:12, 6:9] = np.eye(3)
    T[6:9, 9:12] = np.eye(3)
    Ge = np.zeros((12, 12))  # (position, orientation, angular velocity, e)
    Ge[:9, :9] = G
    Ge[9:, 9:] = np.diag(0.01 * sd9[:3] ** 2 * (1 / rho**2 - 1))
    S = T @ Ge @ T.T
    return 0.5 * (S + S.T)


def p5(cls, **kw):
    """C3 for 300 ticks from a dense initial covariance with position-velocity correlation 1 - 1e-6"""
    mu, _ = syn.pose_initial(B, perturb=True)
    x = _pose(cls, mu, np.broadcast_to(dense_pose_cov(), (B, 12, 12)).copy(), **kw)
    P.run_pose_c3(x, B, 300)
    return x


P6_B = 64
P6_LANES = ("p1", "p2", "p4", "wide_orientation", "rotation_below", "rotation_above")


def p6(cls, **kw):
    """B = 64 with unlike lanes next to each other in one warp.  Lane i is P6_LANES[i % 6]: P1; P2 (UTM offset, GPS
    kinds taking turns); P4 (one velocity update with R = 1e-10 I at tick 150); an orientation standard deviation of
    2 rad; a yaw rate with |w| dt / 2 just below and just above the 0.58 rad range of the fast kernels' SO(3)
    polynomials."""
    Bn = P6_B
    lane = np.array([P6_LANES[i % len(P6_LANES)] for i in range(Bn)])
    utm, acc = lane == "p2", lane == "p4"
    rate = np.zeros((Bn, 3))
    rate[lane == "rotation_below", 2] = 2 * 0.57 / syn.DT
    rate[lane == "rotation_above", 2] = 2 * 0.59 / syn.DT
    off = np.where(utm[:, None], UTM, 0.0)
    mu, sg = syn.pose_initial(Bn, perturb=True)
    mu[:, 0:3] += off
    mu[:, 10:13] += rate
    sg[lane == "wide_orientation", 3:6, 3:6] = np.eye(3) * 4.0
    x = _pose(cls, mu, sg, **kw)
    for k in range(1, 301):
        z, R = syn.pose_measurement(8, Bn, k)
        x.step(syn.DT, 8, z + rate, R)
        if k % 10 == 0:
            z, R = syn.pose_measurement(4, Bn, k)
            R = np.broadcast_to(R, (Bn, 3, 3)).copy()
            if k == 150:
                R[acc] = np.eye(3) * 1e-10
            x.update(4, z, R)
        if k % 100 == 0:
            g = k // 100 - 1
            x.update(0, *_gps(0, Bn, k, off), mask=(~utm).astype(np.uint8))
            x.update(g, *_gps(g, Bn, k, off), mask=utm.astype(np.uint8))
    return x


def _ori(cls, Bn, sg=None, **kw):
    mu, sg0 = syn.orientation_initial(Bn)
    x = cls(1, Bn, **kw)
    x.initialize(mu, sg0 if sg is None else sg)
    x.set_process_noise(syn.ORI_Q)
    return x


def per_filter_orientation_params(Bn: int):
    """gyro / acc bias time constants from 1 s to 1000 s and latitudes over +-1.5 rad, one set per filter"""
    rng = np.random.default_rng(17)
    return 10.0 ** rng.uniform(0, 3, Bn), 10.0 ** rng.uniform(0, 3, Bn), rng.uniform(-1.5, 1.5, Bn)


def o1(cls, **kw):
    """C1 for 1000 ticks with a velocity update every 10th, per-filter tau and latitude"""
    x = _ori(cls, B, **kw)
    x.set_orientation_params(*per_filter_orientation_params(B))
    P.run_ori_c1(x, B, 1000, every=10)
    return x


O2_DT = np.geomspace(1e-5, 0.5, B)


def o2(cls, **kw):
    """per-filter dt from 1e-5 to 0.5 (Q scaled by dt^2 down to about 1e-22), 500 ticks, a velocity update every 10th"""
    x = _ori(cls, B, **kw)
    x.set_orientation_params(syn.ORI_TAU, syn.ORI_TAU, syn.LATITUDE_BREMEN)
    for k in range(1, 501):
        gyro, acc = syn.orientation_imu(B, k)
        x.set_rotation_rate(gyro)
        x.set_acceleration(acc)
        x.predict_dt(O2_DT)
        if k % 10 == 0:
            x.update(9, *syn.orientation_velocity(B, k))
    return x


def o3(cls, **kw):
    """attitude standard deviation 2 rad and heading 3 rad: the any-angle instance, C1 for 300 ticks"""
    _, sg = syn.orientation_initial(B)
    sg[:, 0:3, 0:3] = np.diag([4.0, 4.0, 9.0])
    x = _ori(cls, B, sg, **kw)
    x.set_orientation_params(syn.ORI_TAU, syn.ORI_TAU, syn.LATITUDE_BREMEN)
    P.run_ori_c1(x, B, 300, every=10)
    return x


SCENARIOS = {"P1": (0, p1), "P2": (0, p2), "P3": (0, p3), "P4": (0, p4), "P5": (0, p5), "P6": (0, p6),
             "O1": (1, o1), "O2": (1, o2), "O3": (1, o3)}


# ---- one update per tick: the form the multi-tick call ukfb_run_dev takes ----------------------------

def ticks(name: str):
    """P2 and O1 with one update per tick (the velocity update replaces the angular-velocity one, a GPS fix the
    velocity one) and dt = DT from the first tick: a list of (kind or -1, z (B x 3, leading m used), R (3 x 3, leading
    m x m used), imu (B x 6) or None)"""
    out = []
    for k in range(1, (301 if name == "P2K" else 1001)):
        z, R = np.zeros((B, 3)), np.eye(3)
        if name == "P2K":
            imu = None
            kind = (k // 100 - 1) if k % 100 == 0 else 4 if k % 10 == 0 else 8
            zk, Rk = _gps(kind, B, k, np.broadcast_to(UTM, (B, 3))) if k % 100 == 0 else syn.pose_measurement(kind, B, k)
        else:
            imu = np.concatenate(syn.orientation_imu(B, k), axis=1)
            kind = 9 if k % 10 == 0 else -1
            zk, Rk = syn.orientation_velocity(B, k) if kind == 9 else (z[:, :0], R[:0, :0])
        m = zk.shape[1]
        z[:, :m], R[:m, :m] = zk, Rk
        out.append((kind, z, R, imu))
    return out


def run_ticks(name: str, cls, **kw):
    """the ticks of ticks(name) through the single calls"""
    if name == "P2K":
        mu, sg = syn.pose_initial(B, perturb=True)
        mu[:, 0:3] += UTM
        x = _pose(cls, mu, sg, **kw)
    else:
        x = _ori(cls, B, **kw)
        x.set_orientation_params(*per_filter_orientation_params(B))
    for kind, z, R, imu in ticks(name):
        if imu is not None:
            x.set_rotation_rate(imu[:, :3])
            x.set_acceleration(imu[:, 3:])
        x.predict_dt(syn.DT)
        if kind >= 0:
            m = {1: 2, 2: 1}.get(kind, 3)
            x.update(kind, z[:, :m], R[:m, :m])
    return x


SCENARIOS["P2K"] = (0, lambda cls, **kw: run_ticks("P2K", cls, **kw))
SCENARIOS["O1K"] = (1, lambda cls, **kw: run_ticks("O1K", cls, **kw))
TICK_SCENARIOS = ("P2K", "O1K")  # driven tick by tick; the emulator and single-call runs use the other nine


# ---- references, cached per process -----------------------------------------------------------------

_REFS: dict = {}


def oracle_runs(name: str):
    """(long-double oracle, FP64 oracle) objects after scenario `name`"""
    if name not in _REFS:
        from oracle.oracle_lib import OracleBatch

        kind, fn = SCENARIOS[name]
        _REFS[name] = (fn(lambda k, b: OracleBatch(k, b, variant="ld")), fn(lambda k, b: OracleBatch(k, b)))
    return _REFS[name]


def check(name: str, impl, what: str = "") -> list:
    """Judge the object `impl` after scenario `name` against both oracles: the same status words and mean-pass
    histogram as the FP64 oracle, and every block within the acceptance rule.  Returns the rows of judge()."""
    kind, _ = SCENARIOS[name]
    ld, d = oracle_runs(name)
    assert np.array_equal(impl.get_status(), d.get_status()), f"{what} {name}: status words differ from the oracle's"
    assert np.array_equal(impl.get_mean_iter_hist(), d.get_mean_iter_hist()), \
        f"{what} {name}: mean-pass histogram differs from the oracle's"
    got = impl.get_state()
    assert np.isfinite(got[0]).all() and np.isfinite(got[1]).all(), f"{what} {name}: non-finite state"
    rows = judge(kind, got, d.get_state(), ld.get_state())
    bad = failures(rows)
    assert not bad, f"{what} {name}:\n  " + "\n  ".join(bad)
    return rows
