"""ctypes binding of include/ukf_batch.h (lib/libukfb.so).  No compute happens here and
there is no fallback: a missing library raises, and every entry point of the library
itself fails with UKFB_ERR_CUDA on a machine without an sm_100-class GPU."""
from __future__ import annotations

import ctypes as C
import os

from . import _build

P = C.c_void_p
I = C.c_int
L = C.c_int64
D = C.c_double

# name -> (restype, argtypes); one entry per declaration in include/ukf_batch.h
SIGNATURES = {
    "ukfb_last_error": (C.c_char_p, []),
    "ukfb_create": (I, [I, L, I, C.POINTER(P)]),
    "ukfb_destroy": (I, [P]),
    "ukfb_create_sharded": (I, [I, L, P, I, C.POINTER(P)]),
    "ukfb_shard_count": (I, [P]),
    "ukfb_shard": (I, [P, I, C.POINTER(P), C.POINTER(L), C.POINTER(L)]),
    "ukfb_host_alloc": (I, [C.POINTER(P), C.c_uint64]),
    "ukfb_host_free": (I, [P]),
    "ukfb_get_mu_range": (I, [P, I, I, P]),
    "ukfb_get_mu_range_dev": (I, [P, I, I, P]),
    "ukfb_get_mu_range_async": (I, [P, I, I, P]),
    "ukfb_wait_for_stream": (I, [P, P]),
    "ukfb_stream_wait": (I, [P, P]),
    "ukfb_batch": (L, [P]),
    "ukfb_dof": (I, [P]),
    "ukfb_mu_size": (I, [P]),
    "ukfb_device": (I, [P]),
    "ukfb_initialize": (I, [P, P, P]),
    "ukfb_is_initialized": (I, [P]),
    "ukfb_get_state": (I, [P, P, P]),
    "ukfb_get_state_dev": (I, [P, P, P]),
    "ukfb_initialize_from_body_states": (I, [P, P]),
    "ukfb_initialize_from_body_states_dev": (I, [P, P]),
    "ukfb_get_body_states": (I, [P, P]),
    "ukfb_get_body_states_dev": (I, [P, P]),
    "ukfb_set_process_noise": (I, [P, P, I]),
    "ukfb_get_process_noise": (I, [P, P, I]),
    "ukfb_set_time_bounds": (I, [P, D, D]),
    "ukfb_get_time_bounds": (I, [P, C.POINTER(D), C.POINTER(D)]),
    "ukfb_set_last_time": (I, [P, P, I]),
    "ukfb_get_last_time": (I, [P, P]),
    "ukfb_set_orientation_params": (I, [P, D, D, D]),
    "ukfb_set_orientation_params_per_filter": (I, [P, P, P, P]),
    "ukfb_set_mahalanobis_gate": (I, [P, D]),
    "ukfb_get_mahalanobis_gate": (I, [P, C.POINTER(D)]),
    "ukfb_predict_dt": (I, [P, P, I]),
    "ukfb_predict_dt_dev": (I, [P, P, I]),
    "ukfb_predict_time": (I, [P, P, I]),
    "ukfb_predict_time_dev": (I, [P, P, I]),
    "ukfb_update": (I, [P, I, P, P, I, P]),
    "ukfb_update_dev": (I, [P, I, P, P, I, P]),
    "ukfb_set_measurement_cov": (I, [P, I, P, I]),
    "ukfb_meas_dim": (I, [I]),
    "ukfb_update_mixed": (I, [P, P, P, P]),
    "ukfb_update_mixed_dev": (I, [P, P, P, P]),
    "ukfb_set_acceleration": (I, [P, P, P, I, P]),
    "ukfb_set_acceleration_dev": (I, [P, P, P, I, P]),
    "ukfb_set_rotation_rate": (I, [P, P, P, I, P]),
    "ukfb_set_rotation_rate_dev": (I, [P, P, P, I, P]),
    "ukfb_get_rotation_rate": (I, [P, P]),
    "ukfb_step": (I, [P, P, I, I, P, P, I, P]),
    "ukfb_step_dev": (I, [P, P, I, I, P, P, I, P]),
    "ukfb_step_async": (I, [P, P, I, I, P, P, I, P]),
    "ukfb_get_state_async": (I, [P, P, P]),
    "ukfb_run_dev": (I, [P, I, P, I, P, P, P, I, P]),
    "ukfb_run_events_dev": (I, [P, I, P, P, P, P, I]),
    "ukfb_run_events": (I, [P, I, P, P, P, P, I]),
    "ukfb_run_events_async": (I, [P, I, P, P, P, P, I]),
    "ukfb_get_status": (I, [P, P]),
    "ukfb_clear_status": (I, [P]),
    "ukfb_status_summary": (I, [P, C.POINTER(L), C.POINTER(C.c_uint32)]),
    "ukfb_get_mean_iter_hist": (I, [P, P]),
    "ukfb_clear_mean_iter_hist": (I, [P]),
    "ukfb_get_state_indexed": (I, [P, L, P, P, P]),
    "ukfb_get_state_indexed_dev": (I, [P, L, P, P, P]),
    "ukfb_initialize_indexed": (I, [P, L, P, P, P]),
    "ukfb_initialize_indexed_dev": (I, [P, L, P, P, P]),
    "ukfb_find_status": (I, [P, C.c_uint32, L, P, C.POINTER(L)]),
    "ukfb_clear_status_indexed": (I, [P, L, P]),
    "ukfb_synchronize": (I, [P]),
    "ukfb_stream": (P, [P]),
    "ukfb_event_record": (I, [P, I]),
    "ukfb_event_elapsed_ms": (I, [P, I, I, C.POINTER(C.c_float)]),
    "ukfb_launch_count": (L, [P]),
    "ukfb_overlapped_launch_count": (L, [P]),
    "ukfb_measure_fp64_peak": (I, [P, C.POINTER(D)]),
    "ukfb_selftest_so3": (I, [P, L, P, P, P]),
}

_LIB = None


def library_path() -> str:
    return _build.LIB


def load() -> C.CDLL:
    """Load lib/libukfb.so and declare every prototype.  Raises if the library is absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -m slam_pose_estimation_b200._build` "
            "(nvcc, sm_100a).  This engine has no CPU or PyTorch fallback."
        )
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError = a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
