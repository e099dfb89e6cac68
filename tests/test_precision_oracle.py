"""The long-double oracle (oracle/build/liboracle_ld.so) that tests/precision.py uses as its reference.

It is the FP64 oracle's algorithm with every intermediate in x87 long double: it must agree with the FP64 oracle where
FP64 is accurate, take the same branches on every scenario, be exact to far below FP64 rounding on a case with a
closed-form answer, and make the per-block checker see errors that the norm-wise parity metric cannot.
"""
from __future__ import annotations

import mpmath
import numpy as np
import pytest

import parity as P
import precision as PR
from oracle.oracle_lib import OracleBatch
from slam_pose_estimation_b200 import synthetic as syn

TIGHT = 1e-11  # as in test_oracle.py: two restatements of one algorithm in local-frame coordinates


@pytest.mark.parametrize("name", ["P1", "O1"])
def test_ld_oracle_matches_the_fp64_oracle_in_local_coordinates(name):
    ld, d = PR.oracle_runs(name)
    P.assert_parity(PR.SCENARIOS[name][0], d.get_state(), ld.get_state(), tol=TIGHT, what=f"{name} FP64 vs LD")


@pytest.mark.parametrize("name", list(PR.SCENARIOS))
def test_ld_and_fp64_oracles_take_the_same_branches(name):
    """equal status words and mean-pass histograms: no scenario sits on a decision boundary of the algorithm"""
    ld, d = PR.oracle_runs(name)
    assert np.array_equal(ld.get_status(), d.get_status())
    assert np.array_equal(ld.get_mean_iter_hist(), d.get_mean_iter_hist())


def test_kat_linear_measurement_is_the_kalman_update():
    """test_oracle.py's known answer (a velocity measurement, no orientation coupling: the unscented update equals the
    Kalman update) with the closed form in 30-digit mpmath: the LD oracle is exact to 1e-17 beyond the one rounding of
    the read-back to double"""
    mpmath.mp.dps = 30
    rng = np.random.default_rng(7)
    n = 12
    A = rng.normal(size=(9, 9)) * 0.3
    S9 = A @ A.T + np.eye(9) * 0.05
    idx = [0, 1, 2, 6, 7, 8, 9, 10, 11]
    sigma = np.zeros((n, n))
    sigma[np.ix_(idx, idx)] = S9
    sigma[3:6, 3:6] = np.eye(3) * 1e-4
    mu, _ = syn.pose_initial(1)
    R = np.diag([0.01, 0.02, 0.03])
    z = np.array([[1.1, -0.2, 0.05]])
    o = OracleBatch(0, 1, variant="ld")
    o.initialize(mu, sigma[None])
    o.update(4, z, R)
    mu_o, sg_o = o.get_state()

    M = mpmath.matrix
    S, H = M(sigma.tolist()), mpmath.zeros(3, n)
    for i in range(3):
        H[i, 6 + i] = 1
    x = M([*mu[0, 0:3], 0, 0, 0, *mu[0, 7:13]])
    Sm = H * S * H.T + M(R.tolist())
    K = S * H.T * mpmath.inverse(Sm)
    x_new = x + K * (M(z[0].tolist()) - H * x)
    s_new = S - K * Sm * K.T

    got = np.concatenate([mu_o[0, 0:3], np.zeros(3), mu_o[0, 7:13]])
    pairs = [(got[i], x_new[i]) for i in range(n)] + [(sg_o[0, i, j], s_new[i, j]) for i in range(n) for j in range(n)]
    for g, e in pairs:
        bound = 0.5 * np.spacing(abs(float(e))) + 1e-17 * max(1.0, abs(float(e)))
        assert abs(mpmath.mpf(float(g)) - e) <= bound, (g, e)
    assert np.array_equal(mu_o[0, 3:7], mu[0, 3:7])  # orientation untouched


def _yawed(mu, angle):
    out = mu.copy()
    q = np.tile([0.0, 0.0, np.sin(angle / 2), np.cos(angle / 2)], (mu.shape[0], 1))
    out[:, 3:7] = P._qmul(q, out[:, 3:7])
    return out


def test_per_block_checker_sees_what_the_norm_wise_metric_cannot():
    """Two states that assert_parity accepts against the LD reference and the per-block rule rejects:
    - P2 (UTM coordinates) with the yaw moved by 1e-7 rad, 1e-6 of its standard deviation.  The FP64 oracle's own
      orientation error there is about 1e-8 standard deviations (1e-9 rad), so a smaller yaw error is indistinguishable
      from FP64 rounding; the norm-wise metric divides by 5.9e6 m and would pass yaw errors up to 6e-3 rad;
    - O1 with the gyro-bias covariance block scaled by 1 + 1e-9, which the Frobenius metric sees as 3e-13."""
    ld, d = PR.oracle_runs("P2")
    mu, sg = ld.get_state()
    moved = (_yawed(mu, 1e-7), sg)
    P.assert_parity(0, moved, (mu, sg), what="P2, yaw + 1e-7 rad")
    bad = PR.failures(PR.judge(0, moved, d.get_state(), (mu, sg)))
    assert bad and all(b.startswith("orientation mean") for b in bad), bad

    ld, d = PR.oracle_runs("O1")
    mu, sg = ld.get_state()
    scaled = sg.copy()
    scaled[:, 6:9, 6:9] *= 1 + 1e-9
    P.assert_parity(1, (mu, scaled), (mu, sg), what="O1, gyro-bias covariance x (1 + 1e-9)")
    bad = PR.failures(PR.judge(1, (mu, scaled), d.get_state(), (mu, sg)))
    assert bad and all(b.startswith("gyro_bias cov") for b in bad), bad


@pytest.mark.parametrize("name", list(PR.SCENARIOS))
def test_fp64_oracle_is_within_the_cap(name):
    """the FP64 oracle carries the acceptance rule, so it must itself be close to the exact result on every block"""
    ld, d = PR.oracle_runs(name)
    kind = PR.SCENARIOS[name][0]
    rows = PR.judge(kind, d.get_state(), d.get_state(), ld.get_state())
    assert not PR.failures(rows), PR.failures(rows)
