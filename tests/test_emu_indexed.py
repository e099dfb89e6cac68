"""Per-filter access kernels (csrc/ukf_index.cuh) in the host emulation of tests/simt_emu, against NumPy.

Gather (getCurrentState of listed filters), scatter (initializeFilter of listed filters), status compaction and the
indexed status clear, on both record layouts the engine uses: 32-filter entry-major tiles (fast and thread kernels)
and AoS (warp kernel).  tools/run_emu_sanitized.sh runs this file under ASan + UBSan, which is what checks that a
skipped index is never read or written out of bounds.  The host-pointer entry points' refusals are checked here too:
without a GPU they fail with UKFB_ERR_INVALID or UKFB_ERR_CUDA, never crash."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np
import pytest

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "simt_emu")
_SRC = os.path.join(os.path.dirname(_DIR), "..", "slam_pose_estimation_b200", "csrc")
_LIB = None

P = C.c_void_p
LL = C.c_longlong


def _lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    sanitize = os.environ.get("UKFB_EMU_SANITIZE") == "1"
    out = os.path.join(_DIR, "libukfb_emu_index_san.so" if sanitize else "libukfb_emu_index.so")
    srcs = [os.path.join(_DIR, "emu_index.cpp"), os.path.join(_DIR, "simt_emu_rt.hpp")] + [
        os.path.join(_SRC, f) for f in ("ukf_index.cuh", "ukf_thread.cuh", "ukf_device.cuh", "so3.cuh", "simt.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        cmd = ["/usr/bin/g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-I", _DIR, "-o", out, srcs[0]]
        if sanitize:
            cmd[2:3] = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"]
        subprocess.run(cmd, check=True)
    lib = C.CDLL(out)
    lib.emu_get_state_indexed.argtypes = [P, LL, C.c_int, C.c_int, P, LL, P, P]
    lib.emu_initialize_indexed.argtypes = [P, LL, C.c_int, C.c_int, P, LL, P, P, P]
    lib.emu_clear_status_indexed.argtypes = [P, LL, P, LL]
    lib.emu_find_status.argtypes = [P, LL, C.c_uint32, LL, P, P]
    lib.emu_find_status.restype = LL
    _LIB = lib
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Records:
    """B filter records as the engine keeps them on the device, with a logical [filter][entry] view for NumPy"""

    def __init__(self, kind, B, tiled, seed=0):
        self.kind, self.B, self.tiled = kind, B, tiled
        self.n, self.MU = (12, 13) if kind == 0 else (13, 14)
        self.LP = self.n * (self.n + 1) // 2
        self.REC = self.MU + self.LP
        self.Bpad = (B + 31) // 32 * 32
        rng = np.random.default_rng(seed)
        self.logical = rng.standard_normal((self.Bpad, self.REC))
        self.dev = self._to_dev(self.logical)
        self.t_last = rng.integers(1, 1 << 40, B).astype(np.int64)

    def _to_dev(self, logical):
        if self.tiled:
            return np.ascontiguousarray(logical.reshape(-1, 32, self.REC).transpose(0, 2, 1))
        return np.ascontiguousarray(logical)

    def view(self):
        """logical [filter][entry] of the current device image"""
        if self.tiled:
            return self.dev.transpose(0, 2, 1).reshape(self.Bpad, self.REC)
        return self.dev

    def state_of(self, idx):
        lg = self.view()
        mu = lg[idx, : self.MU].copy()
        tl = np.tril_indices(self.n)
        sg = np.zeros((len(idx), self.n, self.n))
        sg[:, tl[0], tl[1]] = lg[idx, self.MU:]
        sg = sg + np.transpose(np.tril(sg, -1), (0, 2, 1))
        return mu, sg

    def get(self, idx, with_sigma=True, fill=-7.0):
        idx = np.ascontiguousarray(idx, np.int64)
        mu = np.full((idx.size, self.MU), fill)
        sg = np.full((idx.size, self.n, self.n), fill) if with_sigma else None
        _lib().emu_get_state_indexed(_p(self.dev), self.B, self.kind, int(self.tiled), _p(idx), idx.size, _p(mu), _p(sg))
        return mu, sg

    def initialize(self, idx, mu, sg):
        idx = np.ascontiguousarray(idx, np.int64)
        mu, sg = np.ascontiguousarray(mu, float), np.ascontiguousarray(sg, float)
        _lib().emu_initialize_indexed(_p(self.dev), self.B, self.kind, int(self.tiled), _p(idx), idx.size, _p(mu), _p(sg),
                                      _p(self.t_last))


LAYOUTS = [(k, t) for k in (0, 1) for t in (True, False)]
SIZES = [1, 31, 33, 203]


def _index_sets(B, rng):
    sets = {"all": np.arange(B), "sorted": np.sort(rng.choice(B, size=max(1, B // 3), replace=False)),
            "unsorted": rng.permutation(B)[: max(1, (2 * B) // 3)]}
    sets["duplicates"] = np.concatenate([sets["unsorted"], sets["unsorted"][::2], [B - 1, 0, B - 1]])
    return sets


@pytest.mark.parametrize("kind,tiled", LAYOUTS)
@pytest.mark.parametrize("B", SIZES)
def test_gather_equals_numpy(kind, tiled, B):
    rng = np.random.default_rng(B)
    r = Records(kind, B, tiled, seed=B + 10 * kind)
    before = r.dev.copy()
    for name, idx in _index_sets(B, rng).items():
        want_mu, want_sg = r.state_of(idx)
        mu, sg = r.get(idx)
        assert np.array_equal(mu, want_mu), name
        assert np.array_equal(sg, want_sg), name
        mu_only, none = r.get(idx, with_sigma=False)
        assert none is None and np.array_equal(mu_only, want_mu), name
    assert np.array_equal(r.dev, before)  # a read changes nothing


@pytest.mark.parametrize("kind,tiled", LAYOUTS)
@pytest.mark.parametrize("B", SIZES)
def test_scatter_replaces_only_the_listed_records(kind, tiled, B):
    rng = np.random.default_rng(100 + B)
    r = Records(kind, B, tiled, seed=B + 20 * kind)
    sets = _index_sets(B, rng)
    for name in ("all", "sorted", "unsorted"):
        idx = sets[name]
        before, t_before = r.view().copy(), r.t_last.copy()
        mu = rng.standard_normal((idx.size, r.MU))
        sg = rng.standard_normal((idx.size, r.n, r.n))  # not symmetric: only the lower triangle may be read
        r.initialize(idx, mu, sg)
        after = r.view()
        tl = np.tril_indices(r.n)
        want = before.copy()
        want[idx, : r.MU] = mu
        want[idx, r.MU:] = sg[:, tl[0], tl[1]]
        assert np.array_equal(after.view(np.uint64), want.view(np.uint64)), name  # byte for byte, padding lanes included
        t_want = t_before.copy()
        t_want[idx] = 0
        assert np.array_equal(r.t_last, t_want), name
        # the gather returns what was written, symmetrised from the lower triangle as ukfb_get_state does
        got_mu, got_sg = r.get(idx)
        low = np.tril(sg)
        assert np.array_equal(got_mu, mu) and np.array_equal(got_sg, low + np.transpose(np.tril(sg, -1), (0, 2, 1)))


@pytest.mark.parametrize("kind,tiled", LAYOUTS)
def test_out_of_range_device_indices_are_skipped(kind, tiled):
    B = 45
    r = Records(kind, B, tiled, seed=3)
    idx = np.array([5, -1, B, 44, -(1 << 40), B + 1000, 0, 1 << 50], np.int64)
    ok = (idx >= 0) & (idx < B)
    mu, sg = r.get(idx)
    want_mu, want_sg = r.state_of(idx[ok])
    assert np.array_equal(mu[ok], want_mu) and np.array_equal(sg[ok], want_sg)
    assert (mu[~ok] == -7.0).all() and (sg[~ok] == -7.0).all()  # rows of skipped indices are not written
    before, t_before = r.view().copy(), r.t_last.copy()
    nmu, nsg = np.full((idx.size, r.MU), 3.0), np.full((idx.size, r.n, r.n), 4.0)
    r.initialize(idx, nmu, nsg)
    after = r.view()
    touched = np.zeros(r.Bpad, bool)
    touched[idx[ok]] = True
    assert np.array_equal(after[~touched], before[~touched])
    assert (after[idx[ok], : r.MU] == 3.0).all() and (after[idx[ok], r.MU:] == 4.0).all()
    assert np.array_equal(r.t_last[~touched[:B]], t_before[~touched[:B]]) and (r.t_last[idx[ok]] == 0).all()


def _find(status, bits, max_n):
    B = status.size
    chunks = (B + 1023) // 1024
    counts = np.full(chunks + 1, -1, np.int64)
    out = np.full(max(1, min(max_n, B)), -1, np.int64)
    count = _lib().emu_find_status(_p(status), B, bits, max_n, _p(counts), _p(out))
    return count, out[: max(0, min(max_n, count))]


@pytest.mark.parametrize("B,density", [(1, 0.2), (31, 0.2), (33, 0.2), (203, 0.2), (1024, 0.2), (1025, 0.2), (5000, 0.2),
                                       (70001, 0.002)])  # 70001: 69 chunks, so scan lanes sum several chunks each
def test_compaction_equals_flatnonzero(B, density):
    rng = np.random.default_rng(B)
    status = np.zeros(B, np.uint32)
    hit = rng.random(B) < density
    status[hit] = rng.choice(np.array([1, 2, 4, 8, 16, 32, 64, 8 | 64], np.uint32), size=int(hit.sum()))
    status[-1] = 8  # the ragged end of the last chunk
    for bits in (0xFFFFFFFF, 8, 1 | 4, 64, 0):
        want = np.flatnonzero(status & np.uint32(bits))
        count, got = _find(status, bits, B + 5)
        assert count == want.size and np.array_equal(got, want), bits
        for max_n in (0, 1, want.size // 2):
            c, g = _find(status, bits, max_n)
            assert c == want.size and np.array_equal(g, want[:max_n]), (bits, max_n)


def test_compaction_all_and_none_flagged():
    for B in (32, 3000):
        for fill, n in ((0, 0), (8, B)):
            status = np.full(B, fill, np.uint32)
            count, got = _find(status, 0xFFFFFFFF, B)
            assert count == n and np.array_equal(got, np.arange(n))


def test_clear_status_indexed_clears_only_listed():
    B = 1000
    rng = np.random.default_rng(5)
    status = rng.integers(0, 128, B).astype(np.uint32)
    idx = np.concatenate([rng.choice(B, 300, replace=False), [7, 7, -1, B, B + 3]]).astype(np.int64)  # dups, skipped
    want = status.copy()
    want[idx[(idx >= 0) & (idx < B)]] = 0
    _lib().emu_clear_status_indexed(_p(status), B, _p(idx), idx.size)
    assert np.array_equal(status, want)


# ---- host-pointer entry points: refusals without a device -------------------------------------------------------------

def test_indexed_entry_points_refuse_without_crashing():
    from slam_pose_estimation_b200 import _build, _capi

    _build.build()
    lib = _capi.load()
    idx = np.array([0, 1], np.int64)
    buf = np.zeros(400)
    n = C.c_int64(-5)
    pi, pb = idx.ctypes.data_as(C.c_void_p), buf.ctypes.data_as(C.c_void_p)
    for rc in (lib.ukfb_get_state_indexed(None, 2, pi, pb, pb), lib.ukfb_get_state_indexed_dev(None, 2, pi, pb, None),
               lib.ukfb_initialize_indexed(None, 2, pi, pb, pb), lib.ukfb_initialize_indexed_dev(None, 2, pi, pb, pb),
               lib.ukfb_find_status(None, 8, 0, None, C.byref(n)), lib.ukfb_clear_status_indexed(None, 2, pi)):
        assert rc == -1  # UKFB_ERR_INVALID: null handle
    assert n.value == -5  # nothing written on refusal
    assert b"null handle" in lib.ukfb_last_error()
    h = C.c_void_p()
    rc = lib.ukfb_create(0, 64, 0, C.byref(h))
    if rc != 0:
        assert rc == -3 and not h.value  # no GPU: UKFB_ERR_CUDA, and there is no handle to misuse
        return
    try:  # a GPU is present: the argument checks of the host-pointer calls
        bad = [np.array([0, 64], np.int64), np.array([-1], np.int64)]
        for b in bad:
            assert lib.ukfb_get_state_indexed(h, b.size, b.ctypes.data_as(C.c_void_p), pb, None) in (-1, -2)
        assert lib.ukfb_get_state_indexed(h, -1, pi, pb, None) == -1
        assert lib.ukfb_clear_status_indexed(h, 2, None) == -1
        assert lib.ukfb_find_status(h, 8, 3, None, C.byref(n)) == -1
        assert lib.ukfb_get_state_indexed(h, 0, None, None, None) == 0  # n = 0: no-op
    finally:
        lib.ukfb_destroy(h)


def test_python_front_end_validates_index_arrays():
    from slam_pose_estimation_b200 import batch

    a, _ = batch._index_array([3, 1, 2], "t")
    assert a.dtype == np.int64 and a.flags.c_contiguous and list(a) == [3, 1, 2]
    with pytest.raises(TypeError):
        batch._index_array(np.array([1.0, 2.0]), "t")
    with pytest.raises(ValueError):
        batch._index_array(np.zeros((2, 2), np.int64), "t")
    with pytest.raises(ValueError):
        batch._rows(np.zeros((3, 13)), (2, 13), "mu")
    with pytest.raises(ValueError):  # the right number of values in the wrong shape is not silently read as rows
        batch._rows(np.zeros((13, 2)), (2, 13), "mu")
    with pytest.raises(ValueError):
        batch._rows(np.zeros((12, 2, 12)), (2, 12, 12), "sigma")
    assert batch._rows(np.zeros(26), (2, 13), "mu").shape == (26,)
