"""UkfBatch -- thin Python driver over the C ABI (include/ukf_batch.h).

One UkfBatch is B independent PoseUKF / OrientationUKF filters on one B200, or -- with `devices=[...]` -- split by
filter index over several B200s of the box behind ONE handle (ukfb_create_sharded).  Method names
and argument meaning follow the ABI, which in turn follows the reference classes
(UnscentedKalmanFilter.hpp:27-137, PoseUKF.hpp:32-86, OrientationUKF.hpp:28-48).  Host
(NumPy) arguments are copied by the library inside the call; `*_dev` methods take device
pointers (torch CUDA tensors or raw ints) and only enqueue work on the handle's stream: for
torch tensors the handle's stream is first made to wait for the torch stream that is current
on the tensor's device (ukfb_wait_for_stream), so that a kernel never reads inputs that torch
is still writing; outputs of `*_dev` getters are ordered the other way round (ukfb_stream_wait).
PyTorch is used for device memory only -- all filter arithmetic is in lib/libukfb.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi

POSE, ORIENTATION = 0, 1

MEAS_NONE = -1
MEAS_POSE_POSITION, MEAS_POSE_XY, MEAS_POSE_Z, MEAS_POSE_ORIENTATION = 0, 1, 2, 3
MEAS_POSE_VELOCITY, MEAS_POSE_XY_VELOCITY, MEAS_POSE_Z_VELOCITY = 4, 5, 6
MEAS_POSE_XVEL_YAWVEL, MEAS_POSE_ANGULAR_VELOCITY, MEAS_ORI_VELOCITY = 7, 8, 9

EVENT_IDLE, EVENT_POSE_ACCELERATION, EVENT_ORI_ROTATION_RATE, EVENT_ORI_ACCELERATION, EVENT_KIND_COUNT = -2, 10, 11, 12, 13

STATUS_NEG_DT, STATUS_DT_TOO_LARGE, STATUS_NONFINITE_MEAS, STATUS_NOT_SPD, STATUS_MEAN_NO_CONVERGE = 1, 2, 4, 8, 16
STATUS_BAD_EVENT, STATUS_MEAS_REJECTED = 32, 64

RBS_DOUBLES = 49

FIND_STATUS_FIRST = 1024  # matches UkfBatch.find_status fetches with the count

ERR_INVALID, ERR_NOT_INITIALIZED, ERR_CUDA, ERR_NOMEM = -1, -2, -3, -4


class UkfbError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"ukfb error {code}: {text}")
        self.code = code


def _host(a, dtype):
    if a is None:
        return None, None
    a = np.ascontiguousarray(a, dtype=dtype)
    return a, a.ctypes.data_as(C.c_void_p)


def _dev(t):
    """device pointer of a torch CUDA tensor (must be contiguous) or a raw int / None"""
    if t is None:
        return None
    if isinstance(t, int):
        return C.c_void_p(t)
    if not t.is_cuda or not t.is_contiguous():
        raise ValueError("device arguments must be contiguous CUDA tensors")
    return C.c_void_p(t.data_ptr())


def _index_array(idx, who):
    """a 1-D int64 array of filter indices (integer input of another width is widened; anything else is refused)"""
    a = np.asarray(idx)
    if a.ndim != 1:
        raise ValueError(f"{who}: idx must be one-dimensional, got shape {a.shape}")
    if a.size and not np.issubdtype(a.dtype, np.integer):
        raise TypeError(f"{who}: idx must hold integers, got {a.dtype}")
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(C.c_void_p)


def _rows(a, shape, what):
    """float64 rows of exactly `shape`, or the same flattened to one dimension"""
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.shape != tuple(shape) and a.shape != (int(np.prod(shape)),):
        raise ValueError(f"{what} must be {shape}, got {a.shape}")
    return a


def _dev_index(t, who):
    """number of indices in a device index tensor (int64, 1-D, contiguous)"""
    if isinstance(t, int):
        raise TypeError(f"{who}: pass the indices as a torch tensor (its length is the row count)")
    import torch

    if t.dtype != torch.int64 or t.dim() != 1:
        raise TypeError(f"{who}: d_idx must be a 1-D int64 CUDA tensor, got {t.dtype} of shape {tuple(t.shape)}")
    return int(t.numel())


def _dev_rows(t, shape, what):
    if isinstance(t, int):
        return
    import torch

    if t.dtype != torch.float64 or tuple(t.shape) != tuple(shape):
        raise ValueError(f"{what} must be a float64 CUDA tensor of shape {tuple(shape)}, got {t.dtype} {tuple(t.shape)}")


def _torch_stream_of(*tensors):
    """the raw cudaStream_t torch has current on the device of the first torch tensor among the arguments (None if
    there is none: raw device pointers are the caller's own business)"""
    for t in tensors:
        if t is not None and not isinstance(t, int):
            import torch

            return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)
    return None


class UkfBatch:
    def __init__(self, kind: int, B: int, device: int = 0, devices=None, _borrowed=None):
        """devices = [d0, d1, ...]: one handle whose filters are split by index over those devices (contiguous shards,
        one host worker thread and one set of CUDA streams per device, no inter-device traffic)."""
        self.lib = _capi.load()
        self.kind, self.B = int(kind), int(B)
        self._owned = _borrowed is None
        if _borrowed is not None:
            self.h = _borrowed
            self.device = self.lib.ukfb_device(self.h)
        else:
            h = C.c_void_p()
            if devices is not None:
                arr = (C.c_int * len(devices))(*[int(d) for d in devices])
                self._chk(self.lib.ukfb_create_sharded(self.kind, self.B, arr, len(devices), C.byref(h)))
                self.device = int(devices[0])
            else:
                self.device = int(device)
                self._chk(self.lib.ukfb_create(self.kind, self.B, self.device, C.byref(h)))
            self.h = h
        h = self.h
        self.n = self.lib.ukfb_dof(h)
        self.MU = self.lib.ukfb_mu_size(h)
        self._inflight = []  # host arrays referenced by enqueued *_async calls

    def close(self):
        if getattr(self, "h", None):
            if self._owned:
                self.lib.ukfb_destroy(self.h)
            self.h = None

    def shard_count(self) -> int:
        return int(self.lib.ukfb_shard_count(self.h))

    def shard(self, i: int):
        """(UkfBatch over shard i's one-device handle -- owned by this object --, first filter, count): the `_dev`
        entry points of a sharded handle live here"""
        sh, first, count = C.c_void_p(), C.c_int64(), C.c_int64()
        self._chk(self.lib.ukfb_shard(self.h, int(i), C.byref(sh), C.byref(first), C.byref(count)))
        return UkfBatch(self.kind, count.value, _borrowed=sh), first.value, count.value

    def _after_torch(self, *tensors):
        """the handle's stream waits for the torch stream that produced these device inputs"""
        st = _torch_stream_of(*tensors)
        if st is not None:
            self._chk(self.lib.ukfb_wait_for_stream(self.h, st))

    def _before_torch(self, *tensors):
        """the torch stream that will read these device outputs waits for the handle's stream"""
        st = _torch_stream_of(*tensors)
        if st is not None:
            self._chk(self.lib.ukfb_stream_wait(self.h, st))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc: int):
        if rc != 0:
            raise UkfbError(rc, (self.lib.ukfb_last_error() or b"").decode())

    # ---- lifecycle -----------------------------------------------------------------
    def initialize(self, mu, sigma):
        mu, pm = _host(mu, np.float64)
        sg, ps = _host(sigma, np.float64)
        if mu.size != self.B * self.MU or sg.size != self.B * self.n * self.n:
            raise ValueError("initialize: mu must be B x MU and sigma B x n x n")
        self._chk(self.lib.ukfb_initialize(self.h, pm, ps))

    def is_initialized(self) -> bool:
        return bool(self.lib.ukfb_is_initialized(self.h))

    def get_state(self, with_sigma: bool = True):
        mu = np.empty((self.B, self.MU))
        sg = np.empty((self.B, self.n, self.n)) if with_sigma else None
        self._chk(self.lib.ukfb_get_state(self.h, mu.ctypes.data_as(C.c_void_p),
                                          sg.ctypes.data_as(C.c_void_p) if with_sigma else None))
        return (mu, sg) if with_sigma else mu

    def get_state_into(self, mu: np.ndarray, sigma: np.ndarray | None = None):
        """getCurrentState into caller-owned (ideally pinned) host arrays."""
        self._chk(self.lib.ukfb_get_state(self.h, mu.ctypes.data_as(C.c_void_p),
                                          sigma.ctypes.data_as(C.c_void_p) if sigma is not None else None))

    def get_state_dev(self, d_mu, d_sigma=None):
        self._after_torch(d_mu, d_sigma)  # torch may still be using the output buffers
        self._chk(self.lib.ukfb_get_state_dev(self.h, _dev(d_mu), _dev(d_sigma)))
        self._before_torch(d_mu, d_sigma)

    def get_mu_range(self, first: int, count: int, out: np.ndarray | None = None):
        """entries [first, first + count) of every filter's state, B x count (PoseUKF pose = (0, 7))"""
        out = np.empty((self.B, count)) if out is None else out
        self._chk(self.lib.ukfb_get_mu_range(self.h, int(first), int(count), out.ctypes.data_as(C.c_void_p)))
        return out

    def get_mu_range_async(self, first: int, count: int, out: np.ndarray):
        self._inflight.append((out,))
        self._chk(self.lib.ukfb_get_mu_range_async(self.h, int(first), int(count), out.ctypes.data_as(C.c_void_p)))

    def get_mu_range_dev(self, first: int, count: int, d_out):
        self._after_torch(d_out)
        self._chk(self.lib.ukfb_get_mu_range_dev(self.h, int(first), int(count), _dev(d_out)))
        self._before_torch(d_out)

    def initialize_from_body_states(self, rbs):
        """BodyStateMeasurement::fromRigidBodyState + initializeFilter; rbs: B x 49 (include/ukf_batch.h)"""
        rbs, pr = _host(rbs, np.float64)
        assert rbs.size == self.B * RBS_DOUBLES
        self._chk(self.lib.ukfb_initialize_from_body_states(self.h, pr))

    def get_body_states(self):
        """getCurrentState + BodyStateMeasurement::toRigidBodyState; B x 49"""
        out = np.empty((self.B, RBS_DOUBLES))
        self._chk(self.lib.ukfb_get_body_states(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def set_process_noise(self, Q):
        Q, pq = _host(Q, np.float64)
        per = 1 if Q.ndim == 3 else 0
        self._chk(self.lib.ukfb_set_process_noise(self.h, pq, per))

    def get_process_noise(self, per_filter: bool = False):
        out = np.empty((self.B, self.n, self.n) if per_filter else (self.n, self.n))
        self._chk(self.lib.ukfb_get_process_noise(self.h, out.ctypes.data_as(C.c_void_p), int(per_filter)))
        return out

    def set_time_bounds(self, min_dt: float, max_dt: float):
        self._chk(self.lib.ukfb_set_time_bounds(self.h, min_dt, max_dt))

    def get_time_bounds(self):
        a, b = C.c_double(), C.c_double()
        self._chk(self.lib.ukfb_get_time_bounds(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_last_time(self, ts):
        ts = np.atleast_1d(np.asarray(ts, np.int64))
        ts, pt = _host(ts, np.int64)
        self._chk(self.lib.ukfb_set_last_time(self.h, pt, int(ts.size == self.B)))

    def get_last_time(self):
        out = np.empty(self.B, np.int64)
        self._chk(self.lib.ukfb_get_last_time(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def set_mahalanobis_gate(self, max_d2: float):
        """accept functor of ukfom update: measurements with innov^T S^-1 innov > max_d2 are not integrated (inf = off)"""
        self._chk(self.lib.ukfb_set_mahalanobis_gate(self.h, float(max_d2)))

    def get_mahalanobis_gate(self) -> float:
        v = C.c_double()
        self._chk(self.lib.ukfb_get_mahalanobis_gate(self.h, C.byref(v)))
        return v.value

    def set_orientation_params(self, tau_g, tau_a, latitude):
        """scalars: one parameter set for all filters; arrays of B values: one per filter"""
        if np.ndim(tau_g) == 0 and np.ndim(tau_a) == 0 and np.ndim(latitude) == 0:
            self._chk(self.lib.ukfb_set_orientation_params(self.h, float(tau_g), float(tau_a), float(latitude)))
            return
        arrs = [np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.B,))) for a in (tau_g, tau_a, latitude)]
        self._chk(self.lib.ukfb_set_orientation_params_per_filter(self.h, *[a.ctypes.data_as(C.c_void_p) for a in arrs]))

    def predict_dt(self, dt):
        dt = np.atleast_1d(np.asarray(dt, np.float64))
        per = int(dt.size == self.B)
        dt, pd = _host(dt, np.float64)
        self._chk(self.lib.ukfb_predict_dt(self.h, pd, per))

    def predict_dt_dev(self, d_dt, per_filter: bool):
        self._after_torch(d_dt)
        self._chk(self.lib.ukfb_predict_dt_dev(self.h, _dev(d_dt), int(per_filter)))

    def predict_time(self, ts):
        ts = np.atleast_1d(np.asarray(ts, np.int64))
        per = int(ts.size == self.B)
        ts, pt = _host(ts, np.int64)
        self._chk(self.lib.ukfb_predict_time(self.h, pt, per))

    def predict_time_dev(self, d_ts, per_filter: bool):
        self._after_torch(d_ts)
        self._chk(self.lib.ukfb_predict_time_dev(self.h, _dev(d_ts), int(per_filter)))

    # ---- measurements -------------------------------------------------------------------------
    def meas_dim(self, kind: int) -> int:
        return self.lib.ukfb_meas_dim(kind)

    def update(self, kind: int, mu, cov, mask=None):
        m = self.meas_dim(kind)
        mu, pm = _host(mu, np.float64)
        cov, pc = _host(cov, np.float64)
        if mu.size != self.B * m:
            raise ValueError(f"update: mu must be B x {m}")
        per = 1 if (cov is not None and cov.ndim == 3) else 0
        mask, pk = _host(mask, np.uint8)
        self._chk(self.lib.ukfb_update(self.h, kind, pm, pc, per, pk))

    def set_measurement_cov(self, kind: int, cov):
        """keep a covariance for `kind` on the device (m x m or B x m x m); update / step / step_async then take cov=None"""
        cov, pc = _host(cov, np.float64)
        self._chk(self.lib.ukfb_set_measurement_cov(self.h, kind, pc, 1 if cov.ndim == 3 else 0))

    def update_dev(self, kind: int, d_mu, d_cov, cov_per_filter: bool, d_mask=None):
        self._after_torch(d_mu, d_cov, d_mask)
        self._chk(self.lib.ukfb_update_dev(self.h, kind, _dev(d_mu), _dev(d_cov), int(cov_per_filter), _dev(d_mask)))

    def update_mixed(self, kinds, mu3, cov33):
        kinds, pk = _host(kinds, np.int8)
        mu3, pm = _host(mu3, np.float64)
        cov33, pc = _host(cov33, np.float64)
        if kinds.size != self.B or mu3.size != self.B * 3 or cov33.size != self.B * 9:
            raise ValueError("update_mixed: kinds B, mu3 B x 3, cov33 B x 3 x 3")
        self._chk(self.lib.ukfb_update_mixed(self.h, pk, pm, pc))

    def update_mixed_dev(self, d_kinds, d_mu3, d_cov33):
        self._after_torch(d_kinds, d_mu3, d_cov33)
        self._chk(self.lib.ukfb_update_mixed_dev(self.h, _dev(d_kinds), _dev(d_mu3), _dev(d_cov33)))

    def set_acceleration(self, mu, cov=None, mask=None):
        mu, pm = _host(mu, np.float64)
        cov, pc = _host(cov, np.float64)
        per = 1 if (cov is not None and cov.ndim == 3) else 0
        mask, pk = _host(mask, np.uint8)
        self._chk(self.lib.ukfb_set_acceleration(self.h, pm, pc, per, pk))

    def set_rotation_rate(self, mu, cov=None, mask=None):
        mu, pm = _host(mu, np.float64)
        cov, pc = _host(cov, np.float64)
        per = 1 if (cov is not None and cov.ndim == 3) else 0
        mask, pk = _host(mask, np.uint8)
        self._chk(self.lib.ukfb_set_rotation_rate(self.h, pm, pc, per, pk))

    def get_rotation_rate(self):
        out = np.empty((self.B, 3))
        self._chk(self.lib.ukfb_get_rotation_rate(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    # ---- fused ------------------------------------------------------------------------------------
    def _step_args(self, dt, kind, mu, cov, mask):
        """(the host arrays, which must outlive the call, and the arguments of ukfb_step after the handle)"""
        dt = np.atleast_1d(np.asarray(dt, np.float64))
        per = int(dt.size == self.B)
        dt, pd = _host(dt, np.float64)
        mu, pm = _host(mu, np.float64)
        cov, pc = _host(cov, np.float64)
        cper = 1 if (cov is not None and cov.ndim == 3) else 0
        mask, pk = _host(mask, np.uint8)
        return (dt, mu, cov, mask), (pd, per, kind, pm, pc, cper, pk)

    def step(self, dt, kind: int, mu=None, cov=None, mask=None):
        arrays, args = self._step_args(dt, kind, mu, cov, mask)
        self._chk(self.lib.ukfb_step(self.h, *args))

    def step_async(self, dt, kind: int, mu=None, cov=None, mask=None):
        """ukfb_step_async: enqueue only.  The arrays passed here are kept alive by this object until synchronize();
        pass pinned, C-contiguous float64 arrays (no conversion copy is made for those) for real overlap."""
        arrays, args = self._step_args(dt, kind, mu, cov, mask)
        self._inflight.append(arrays)
        self._chk(self.lib.ukfb_step_async(self.h, *args))

    def get_state_async(self, mu: np.ndarray, sigma: np.ndarray | None = None):
        """ukfb_get_state_async into caller-owned (pinned) host arrays; valid after synchronize()."""
        self._inflight.append((mu, sigma))
        self._chk(self.lib.ukfb_get_state_async(self.h, mu.ctypes.data_as(C.c_void_p),
                                                sigma.ctypes.data_as(C.c_void_p) if sigma is not None else None))

    def step_dev(self, d_dt, dt_per_filter: bool, kind: int, d_mu=None, d_cov=None, cov_per_filter: bool = False, d_mask=None):
        self._after_torch(d_dt, d_mu, d_cov, d_mask)
        self._chk(self.lib.ukfb_step_dev(self.h, _dev(d_dt), int(dt_per_filter), kind, _dev(d_mu), _dev(d_cov),
                                         int(cov_per_filter), _dev(d_mask)))

    def run_dev(self, K: int, d_dt, dt_per_filter: bool, kinds=None, d_mu3=None, d_cov33=None, cov_per_filter: bool = False,
                d_imu=None):
        kinds_arr, pk = _host(kinds, np.int8)
        if kinds_arr is not None and kinds_arr.size != K:
            raise ValueError("run_dev: kinds must hold K entries")
        self._after_torch(d_dt, d_mu3, d_cov33, d_imu)
        self._chk(self.lib.ukfb_run_dev(self.h, K, _dev(d_dt), int(dt_per_filter), pk, _dev(d_mu3), _dev(d_cov33),
                                        int(cov_per_filter), _dev(d_imu)))

    # ---- status --------------------------------------------------------------------------------------
    def run_events(self, ts, kinds, mu3, cov):
        """K slots of per-filter queued samples (include/ukf_batch.h, "Event streams"): ts, kinds: K x B; mu3: K x B x 3;
        cov: EVENT_KIND_COUNT x 3 x 3 (per-sensor table) or K x B x 3 x 3 (per event)."""
        ts, pt = _host(ts, np.int64)
        kinds, pk = _host(kinds, np.int8)
        mu3, pm = _host(mu3, np.float64)
        cov, pc = _host(cov, np.float64)
        K = ts.shape[0] if ts.ndim == 2 else ts.size // self.B
        assert ts.size == K * self.B and kinds.size == K * self.B and mu3.size == K * self.B * 3
        per_event = cov.shape != (13, 3, 3)  # a (13, 3, 3) array is the per-sensor table
        assert not per_event or cov.size == K * self.B * 9
        self._chk(self.lib.ukfb_run_events(self.h, K, pt, pk, pm, pc, 1 if per_event else 0))

    def run_events_async(self, ts, kinds, mu3, cov):
        """ukfb_run_events_async: enqueue only; pass pinned C-contiguous arrays and keep them unchanged until synchronize()"""
        ts, pt = _host(ts, np.int64)
        kinds, pk = _host(kinds, np.int8)
        mu3, pm = _host(mu3, np.float64)
        cov, pc = _host(cov, np.float64)
        K = ts.size // self.B
        per_event = cov.shape != (13, 3, 3)
        self._inflight.append((ts, kinds, mu3, cov))
        self._chk(self.lib.ukfb_run_events_async(self.h, K, pt, pk, pm, pc, 1 if per_event else 0))

    def run_events_dev(self, K: int, d_ts, d_kinds, d_mu3, d_cov, per_event: bool):
        self._after_torch(d_ts, d_kinds, d_mu3, d_cov)
        self._chk(self.lib.ukfb_run_events_dev(self.h, int(K), _dev(d_ts), _dev(d_kinds), _dev(d_mu3), _dev(d_cov),
                                               1 if per_event else 0))

    def get_status(self):
        out = np.empty(self.B, np.uint32)
        self._chk(self.lib.ukfb_get_status(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def clear_status(self):
        self._chk(self.lib.ukfb_clear_status(self.h))

    def status_summary(self):
        n, bits = C.c_int64(), C.c_uint32()
        self._chk(self.lib.ukfb_status_summary(self.h, C.byref(n), C.byref(bits)))
        return n.value, bits.value

    def get_mean_iter_hist(self):
        out = np.zeros(8, np.uint64)
        self._chk(self.lib.ukfb_get_mean_iter_hist(self.h, out.ctypes.data_as(C.c_void_p)))
        return out

    def clear_mean_iter_hist(self):
        self._chk(self.lib.ukfb_clear_mean_iter_hist(self.h))

    # ---- per-filter access -----------------------------------------------------------------------------
    def get_state_indexed(self, idx, with_sigma: bool = True):
        """getCurrentState of filters idx (global indices, any order, duplicates allowed): (mu n x MU, sigma n x n x n),
        or mu alone with with_sigma=False.  Only those n rows travel."""
        idx, pi = _index_array(idx, "get_state_indexed")
        k = idx.size
        mu = np.empty((k, self.MU))
        sg = np.empty((k, self.n, self.n)) if with_sigma else None
        self._chk(self.lib.ukfb_get_state_indexed(self.h, k, pi, mu.ctypes.data_as(C.c_void_p),
                                                  sg.ctypes.data_as(C.c_void_p) if with_sigma else None))
        return (mu, sg) if with_sigma else mu

    def get_state_indexed_dev(self, d_idx, d_mu, d_sigma=None):
        """the same into device tensors: d_idx int64 (n,), d_mu float64 (n, MU), d_sigma float64 (n, n, n) or None"""
        k = _dev_index(d_idx, "get_state_indexed_dev")
        _dev_rows(d_mu, (k, self.MU), "d_mu")
        if d_sigma is not None:
            _dev_rows(d_sigma, (k, self.n, self.n), "d_sigma")
        self._after_torch(d_idx, d_mu, d_sigma)
        self._chk(self.lib.ukfb_get_state_indexed_dev(self.h, k, _dev(d_idx), _dev(d_mu), _dev(d_sigma)))
        self._before_torch(d_mu, d_sigma)

    def initialize_indexed(self, idx, mu, sigma):
        """initializeFilter of filters idx only (unique global indices): mu n x MU, sigma n x n x n; their t_last = 0.
        Status words are left alone: clear_status_indexed after a recovery."""
        idx, pi = _index_array(idx, "initialize_indexed")
        k = idx.size
        mu = _rows(mu, (k, self.MU), "mu")
        sg = _rows(sigma, (k, self.n, self.n), "sigma")
        self._chk(self.lib.ukfb_initialize_indexed(self.h, k, pi, mu.ctypes.data_as(C.c_void_p), sg.ctypes.data_as(C.c_void_p)))

    def initialize_indexed_dev(self, d_idx, d_mu, d_sigma):
        k = _dev_index(d_idx, "initialize_indexed_dev")
        _dev_rows(d_mu, (k, self.MU), "d_mu")
        _dev_rows(d_sigma, (k, self.n, self.n), "d_sigma")
        self._after_torch(d_idx, d_mu, d_sigma)
        self._chk(self.lib.ukfb_initialize_indexed_dev(self.h, k, _dev(d_idx), _dev(d_mu), _dev(d_sigma)))
        self._before_torch(d_idx, d_mu, d_sigma)  # torch must not overwrite the inputs before the kernel has read them

    def find_status(self, bits: int = 0xFFFFFFFF) -> np.ndarray:
        """ascending indices of every filter whose status word has any of `bits`.  One call returns the count and the
        first FIND_STATUS_FIRST matches (a few failed filters: one round trip); a second one fetches the rest."""
        bits = int(bits) & 0xFFFFFFFF
        n = C.c_int64()
        out = np.empty(min(self.B, FIND_STATUS_FIRST), np.int64)
        self._chk(self.lib.ukfb_find_status(self.h, bits, out.size, out.ctypes.data_as(C.c_void_p), C.byref(n)))
        if n.value > out.size:
            out = np.empty(n.value, np.int64)
            self._chk(self.lib.ukfb_find_status(self.h, bits, n.value, out.ctypes.data_as(C.c_void_p), C.byref(n)))
        return out[: n.value]

    def clear_status_indexed(self, idx):
        idx, pi = _index_array(idx, "clear_status_indexed")
        self._chk(self.lib.ukfb_clear_status_indexed(self.h, idx.size, pi))

    # ---- checkpoint / restore (image format: include/ukf_batch.h) ----------------------------------------
    def checkpoint_size(self) -> int:
        """bytes of this batch's checkpoint image now (Q, orientation-parameter and kept-covariance modes decide it)"""
        n = C.c_uint64()
        self._chk(self.lib.ukfb_checkpoint_size(self.h, C.byref(n)))
        return n.value

    def checkpoint(self, out: np.ndarray | None = None) -> np.ndarray:
        """one image of every filter's full state and the batch's handle-wide values, as a np.uint8 array (into `out`, a
        uint8 array of at least checkpoint_size() bytes -- pinned for speed -- if given).  Writing it to disk is
        `img.tofile(path)`; it restores onto a batch of the same kind and size on any number of devices."""
        size = self.checkpoint_size()
        if out is None:
            out = np.empty(size, np.uint8)
        elif out.dtype != np.uint8 or not out.flags.c_contiguous or out.size < size:
            raise ValueError(f"checkpoint: out must be a contiguous uint8 array of at least {size} bytes")
        self._chk(self.lib.ukfb_checkpoint_save(self.h, out.ctypes.data_as(C.c_void_p), out.size))
        return out[:size]

    def restore(self, buf):
        """replace this batch's whole state by an image of checkpoint(): bytes, bytearray or a uint8 array.  A rejected
        image (other kind or size, bad version, truncated) raises UkfbError and changes nothing."""
        if isinstance(buf, (bytes, bytearray, memoryview)):
            a = np.frombuffer(buf, np.uint8)
        else:
            a = np.asarray(buf)
            if a.dtype != np.uint8:
                raise TypeError(f"restore: the image must be bytes, bytearray or a uint8 array, got {a.dtype}")
            a = np.ascontiguousarray(a.reshape(-1))
        self._chk(self.lib.ukfb_checkpoint_restore(self.h, a.ctypes.data_as(C.c_void_p), a.size))

    def checkpoint_dev(self, out=None):
        """the image into a CUDA torch.uint8 tensor on this batch's device (allocated if None), enqueued on the handle's
        stream and ordered before later work of the torch stream: an in-device snapshot for rollback (restore_dev)"""
        import torch

        size = self.checkpoint_size()
        if out is None:
            out = torch.empty(size, dtype=torch.uint8, device=f"cuda:{self.device}")
        elif out.dtype != torch.uint8 or not out.is_cuda or out.numel() < size or not out.is_contiguous():
            raise ValueError(f"checkpoint_dev: out must be a contiguous CUDA uint8 tensor of at least {size} bytes")
        elif out.device.index != self.device:
            raise ValueError(f"checkpoint_dev: out is on {out.device}, this batch on cuda:{self.device}")
        self._after_torch(out)  # torch may still be using the buffer
        self._chk(self.lib.ukfb_checkpoint_save_dev(self.h, _dev(out), out.numel()))
        self._before_torch(out)
        return out

    def restore_dev(self, t):
        """replace this batch's state by an image in a CUDA torch.uint8 tensor (checkpoint_dev); the header is read back
        to be checked, the payload stays on the device"""
        import torch

        if t.dtype != torch.uint8 or not t.is_cuda:
            raise ValueError("restore_dev: the image must be a CUDA uint8 tensor")
        if t.device.index != self.device:
            raise ValueError(f"restore_dev: the image is on {t.device}, this batch on cuda:{self.device}")
        self._after_torch(t)
        self._chk(self.lib.ukfb_checkpoint_restore_dev(self.h, _dev(t), t.numel()))
        self._before_torch(t)  # torch must not overwrite the image before it has been read

    # ---- stream plumbing ------------------------------------------------------------------------------
    def synchronize(self):
        self._chk(self.lib.ukfb_synchronize(self.h))
        self._inflight.clear()

    def stream(self) -> int:
        return int(self.lib.ukfb_stream(self.h) or 0)

    def event_record(self, slot: int):
        self._chk(self.lib.ukfb_event_record(self.h, slot))

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float()
        self._chk(self.lib.ukfb_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return int(self.lib.ukfb_launch_count(self.h))

    def overlapped_launch_count(self) -> int:
        """how many of those were ordered tile by tile against their predecessor instead of launch by launch"""
        return int(self.lib.ukfb_overlapped_launch_count(self.h))

    def selftest_so3(self, v, x):
        """device exp / log / reciprocal / sqrt of csrc/so3.cuh and simt.cuh on n inputs -> (n, 21), see the header"""
        v, pv = _host(v, np.float64)
        x, px = _host(x, np.float64)
        n = x.size
        assert v.size == 3 * n
        out = np.empty((n, 21))
        self._chk(self.lib.ukfb_selftest_so3(self.h, n, pv, px, out.ctypes.data_as(C.c_void_p)))
        return out

    def measure_fp64_peak(self) -> float:
        v = C.c_double()
        self._chk(self.lib.ukfb_measure_fp64_peak(self.h, C.byref(v)))
        return v.value
