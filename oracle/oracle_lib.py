"""oracle/oracle_lib.py -- ctypes loader for the CPU oracle.  TEST INFRASTRUCTURE ONLY.

Builds (make) and loads oracle/build/liboracle.so and wraps the orc_* batch calls
with the same method names as slam_pose_estimation_b200.UkfBatch, so a parity test
drives both with identical arguments.  Only tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
_LIBS: dict[str, C.CDLL] = {}

POSE, ORIENTATION = 0, 1


def build(quiet: bool = True) -> None:
    subprocess.run(["make", "-C", _DIR], check=True, stdout=subprocess.DEVNULL if quiet else None)


REF_LIB = os.path.join(_DIR, "_ref", "libref.so")
REF_ROOT = "/root/reference"


def build_ref(quiet: bool = True) -> bool:
    """oracle/_ref/libref.so: the reference's own UKF sources compiled unmodified against oracle/ref_shim
    (oracle/ref_recipe.mk).  Needs /root/reference, which exists in the build container only: elsewhere the file built
    there is used as it is.  Returns whether the library exists afterwards."""
    if os.path.isdir(os.path.join(REF_ROOT, "src")):
        subprocess.run(["make", "-f", os.path.join("oracle", "ref_recipe.mk")], check=True, cwd=os.path.dirname(_DIR),
                       stdout=subprocess.DEVNULL if quiet else None)
    return os.path.exists(REF_LIB)


def load(variant: str = "left") -> C.CDLL:
    """variant: 'left' (default SO(3) convention), 'right' (upstream body-frame), 'tight' (tighter manifold-mean
    tolerance), 'ld' (the default oracle computed in long double, tests/precision.py) or 'ref' (the reference's own
    wrapper sources over the oracle's engine, oracle/_ref)."""
    if variant in _LIBS:
        return _LIBS[variant]
    if variant == "ref":
        if not build_ref():
            raise RuntimeError("oracle/_ref/libref.so is missing and /root/reference is not here to build it")
        path = REF_LIB
    else:
        name = {"left": "liboracle.so", "right": "liboracle_right.so", "tight": "liboracle_tight.so",
                "ld": "liboracle_ld.so"}[variant]
        path = os.path.join(_DIR, "build", name)
        if not os.path.exists(path):
            build()
    lib = C.CDLL(path)
    lib.orc_create.restype = C.c_void_p
    lib.orc_create.argtypes = [C.c_int, C.c_int64]
    lib.orc_destroy.argtypes = [C.c_void_p]
    lib.orc_max_threads.restype = C.c_int
    _LIBS[variant] = lib
    return lib


def _p(a, dtype):
    if a is None:
        return None, None
    a = np.ascontiguousarray(a, dtype=dtype)
    return a, a.ctypes.data_as(C.c_void_p)


class OracleBatch:
    def __init__(self, kind: int, B: int, variant: str = "left", threads: int | None = None):
        self.lib = load(variant)
        self.kind, self.B = kind, int(B)
        self.n = 12 if kind == POSE else 13
        self.MU = 13 if kind == POSE else 14
        if threads:
            self.lib.orc_set_threads(C.c_int(threads))
        self.h = C.c_void_p(self.lib.orc_create(kind, self.B))
        if not self.h:
            raise RuntimeError("orc_create failed")

    def __del__(self):
        try:
            if self.h:
                self.lib.orc_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def _chk(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} -> {rc}")

    def initialize(self, mu, sigma):
        mu, pm = _p(mu, np.float64)
        sg, ps = _p(sigma, np.float64)
        assert mu.size == self.B * self.MU and sg.size == self.B * self.n * self.n
        self._chk(self.lib.orc_initialize(self.h, pm, ps), "orc_initialize")

    def get_state(self):
        mu = np.empty((self.B, self.MU))
        sg = np.empty((self.B, self.n, self.n))
        self._chk(self.lib.orc_get_state(self.h, mu.ctypes.data_as(C.c_void_p), sg.ctypes.data_as(C.c_void_p)),
                  "orc_get_state")
        return mu, sg

    def set_process_noise(self, Q):
        Q, pq = _p(Q, np.float64)
        per = 1 if Q.ndim == 3 else 0
        self._chk(self.lib.orc_set_process_noise(self.h, pq, C.c_int(per)), "orc_set_process_noise")

    def set_time_bounds(self, min_dt, max_dt):
        self._chk(self.lib.orc_set_time_bounds(self.h, C.c_double(min_dt), C.c_double(max_dt)), "set_time_bounds")

    def set_orientation_params(self, tau_g, tau_a, latitude):
        if np.ndim(tau_g) == 0 and np.ndim(tau_a) == 0 and np.ndim(latitude) == 0:
            self._chk(self.lib.orc_set_orientation_params(self.h, C.c_double(tau_g), C.c_double(tau_a),
                                                          C.c_double(latitude)), "set_orientation_params")
            return
        arrs = [np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.B,))) for a in (tau_g, tau_a, latitude)]
        self._chk(self.lib.orc_set_orientation_params_per_filter(self.h, *[a.ctypes.data_as(C.c_void_p) for a in arrs]),
                  "set_orientation_params_per_filter")

    def set_mahalanobis_gate(self, max_d2):
        self._chk(self.lib.orc_set_mahalanobis_gate(self.h, C.c_double(max_d2)), "set_mahalanobis_gate")

    def set_last_time(self, ts):
        ts = np.atleast_1d(np.asarray(ts, np.int64))
        ts, pt = _p(ts, np.int64)
        self._chk(self.lib.orc_set_last_time(self.h, pt, C.c_int(1 if ts.size == self.B else 0)),
                  "set_last_time")

    def get_last_time(self):
        out = np.empty(self.B, np.int64)
        self._chk(self.lib.orc_get_last_time(self.h, out.ctypes.data_as(C.c_void_p)), "get_last_time")
        return out

    def predict_dt(self, dt):
        dt = np.atleast_1d(np.asarray(dt, np.float64))
        per = 1 if dt.size == self.B else 0
        dt, pd = _p(dt, np.float64)
        self._chk(self.lib.orc_predict_dt(self.h, pd, C.c_int(per)), "orc_predict_dt")

    def predict_time(self, ts):
        ts = np.atleast_1d(np.asarray(ts, np.int64))
        per = 1 if ts.size == self.B else 0
        ts, pt = _p(ts, np.int64)
        self._chk(self.lib.orc_predict_time(self.h, pt, C.c_int(per)), "orc_predict_time")

    def update(self, kind, mu, cov, mask=None):
        m = self.lib.orc_meas_dim(C.c_int(kind))
        mu, pm = _p(mu, np.float64)
        cov, pc = _p(cov, np.float64)
        assert mu.size == self.B * m
        per = 1 if cov.ndim == 3 else 0
        mask, pk = _p(mask, np.uint8)
        self._chk(self.lib.orc_update(self.h, C.c_int(kind), pm, pc, C.c_int(per), pk), "orc_update")

    def update_mixed(self, kinds, mu3, cov33):
        kinds, pk = _p(kinds, np.int8)
        mu3, pm = _p(mu3, np.float64)
        cov33, pc = _p(cov33, np.float64)
        self._chk(self.lib.orc_update_mixed(self.h, pk, pm, pc), "orc_update_mixed")

    def run_events(self, ts, kinds, mu3, cov):
        ts, pt = _p(ts, np.int64)
        kinds, pk = _p(kinds, np.int8)
        mu3, pm = _p(mu3, np.float64)
        cov, pc = _p(cov, np.float64)
        K = ts.size // self.B
        per_event = cov.shape != (13, 3, 3)  # a (13, 3, 3) array is the per-sensor table
        assert not per_event or cov.size == K * self.B * 9
        self._chk(self.lib.orc_run_events(self.h, C.c_int(K), pt, pk, pm, pc, C.c_int(1 if per_event else 0)),
                  "orc_run_events")

    def set_acceleration(self, mu, cov=None, mask=None):
        mu, pm = _p(mu, np.float64)
        cov, pc = _p(cov, np.float64)
        per = 1 if (cov is not None and cov.ndim == 3) else 0
        mask, pk = _p(mask, np.uint8)
        self._chk(self.lib.orc_set_acceleration(self.h, pm, pc, C.c_int(per), pk), "orc_set_acceleration")

    def set_rotation_rate(self, mu, cov=None, mask=None):
        mu, pm = _p(mu, np.float64)
        cov, pc = _p(cov, np.float64)
        per = 1 if (cov is not None and cov.ndim == 3) else 0
        mask, pk = _p(mask, np.uint8)
        self._chk(self.lib.orc_set_rotation_rate(self.h, pm, pc, C.c_int(per), pk), "orc_set_rotation_rate")

    def get_rotation_rate(self):
        out = np.empty((self.B, 3))
        self._chk(self.lib.orc_get_rotation_rate(self.h, out.ctypes.data_as(C.c_void_p)), "get_rotation_rate")
        return out

    def step(self, dt, kind, mu, cov, mask=None):
        self.predict_dt(dt)
        if kind >= 0:
            self.update(kind, mu, cov, mask)

    def get_status(self):
        out = np.empty(self.B, np.uint32)
        self._chk(self.lib.orc_get_status(self.h, out.ctypes.data_as(C.c_void_p)), "get_status")
        return out

    def clear_status(self):
        self._chk(self.lib.orc_clear_status(self.h), "clear_status")

    def get_mean_iter_hist(self):
        out = np.zeros(8, np.uint64)
        self._chk(self.lib.orc_get_mean_iter_hist(self.h, out.ctypes.data_as(C.c_void_p)), "hist")
        return out

    def max_threads(self):
        return int(self.lib.orc_max_threads())


def from_body_states(rbs):
    """BodyStateMeasurement::fromRigidBodyState over B records (B x 49) -> mu (B,13), sigma (B,12,12)"""
    lib = load()
    rbs = np.ascontiguousarray(rbs, np.float64).reshape(-1, 49)
    B = rbs.shape[0]
    mu, sg = np.empty((B, 13)), np.empty((B, 12, 12))
    lib.orc_from_body_states(rbs.ctypes.data_as(C.c_void_p), C.c_int64(B), mu.ctypes.data_as(C.c_void_p),
                             sg.ctypes.data_as(C.c_void_p))
    return mu, sg


def to_body_states(mu, sigma):
    """BodyStateMeasurement::toRigidBodyState over B filters -> B x 49"""
    lib = load()
    mu = np.ascontiguousarray(mu, np.float64).reshape(-1, 13)
    sigma = np.ascontiguousarray(sigma, np.float64).reshape(-1, 12, 12)
    out = np.empty((mu.shape[0], 49))
    lib.orc_to_body_states(mu.ctypes.data_as(C.c_void_p), sigma.ctypes.data_as(C.c_void_p), C.c_int64(mu.shape[0]),
                           out.ctypes.data_as(C.c_void_p))
    return out
