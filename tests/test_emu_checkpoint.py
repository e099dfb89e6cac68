"""Checkpoint record transforms (csrc/ukf_checkpoint.cuh) in the host emulation of tests/simt_emu, against NumPy.

records -> rows (save) and rows -> records (restore), per element and per tile, on both record layouts the engine uses:
32-filter entry-major tiles (fast and thread kernels, tile_index) and AoS (warp kernel).  Grids are smaller than the
work, so every stride loop runs; batch sizes leave ragged last tiles.  The words are random bit patterns with NaN
payloads and -0.0 among them: the transforms must move bits, never values.  tools/run_emu_sanitized.sh runs this file
under ASan + UBSan, which is what checks that rows past B and the padding lanes of a ragged tile are never touched
out of bounds."""
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
    out = os.path.join(_DIR, "libukfb_emu_checkpoint_san.so" if sanitize else "libukfb_emu_checkpoint.so")
    srcs = [os.path.join(_DIR, "emu_checkpoint.cpp"), os.path.join(_DIR, "simt_emu_rt.hpp")] + [
        os.path.join(_SRC, f) for f in ("ukf_checkpoint.cuh", "ukf_index.cuh", "ukf_thread.cuh", "ukf_device.cuh", "so3.cuh",
                                        "simt.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in srcs):
        cmd = ["/usr/bin/g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-I", _DIR, "-o", out, srcs[0]]
        if sanitize:
            cmd[2:3] = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"]
        subprocess.run(cmd, check=True)
    lib = C.CDLL(out)
    lib.emu_checkpoint_transform.argtypes = [C.c_int, C.c_int, P, P, LL, C.c_int, C.c_int, C.c_uint, C.c_uint]
    _LIB = lib
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def rec_words(kind):
    n, mu = (12, 13) if kind == 0 else (13, 14)
    return mu + n * (n + 1) // 2


def tile_index(b, e, REC):
    """ukf_thread.cuh: entry e of filter b in 32-filter entry-major tiles"""
    return (b // 32) * (32 * REC) + e * 32 + (b % 32)


def rec_index(tiled, b, e, REC):
    return tile_index(b, e, REC) if tiled else b * REC + e


def bit_patterns(shape, rng):
    """random 64-bit words, a quarter of them NaNs with payloads (quiet and signalling, both signs), some -0.0 and +0.0"""
    w = rng.integers(0, 1 << 63, size=shape, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=shape, dtype=np.uint64)
    nan = rng.random(shape) < 0.25
    payload = rng.integers(1, 1 << 51, size=shape, dtype=np.uint64)
    sign = rng.integers(0, 2, size=shape, dtype=np.uint64) << np.uint64(63)
    quiet = rng.integers(0, 2, size=shape, dtype=np.uint64) << np.uint64(51)
    w[nan] = (sign | np.uint64(0x7FF0000000000000) | quiet | payload)[nan]
    w[rng.random(shape) < 0.05] = np.uint64(0x8000000000000000)  # -0.0
    w[rng.random(shape) < 0.05] = np.uint64(0)
    return w


def device_image(logical, tiled, REC):
    """records as the engine keeps them: logical [filter][entry] (B rounded up to whole tiles) in the handle's layout"""
    Bpad = logical.shape[0]
    out = np.empty(Bpad * REC, np.uint64)
    b, e = np.meshgrid(np.arange(Bpad), np.arange(REC), indexing="ij")
    out[rec_index(tiled, b, e, REC).reshape(-1)] = logical.reshape(-1)
    return out


def transform(save, variant, rec, rows, B, kind, tiled, grid=3, warps=2):
    _lib().emu_checkpoint_transform(int(save), variant, _p(rec), _p(rows), B, kind, int(tiled), grid, warps)


LAYOUTS = [(k, t) for k in (0, 1) for t in (True, False)]
SIZES = [1, 31, 32, 33, 1007]
VARIANTS = {"elem": 0, "tile": 1}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("kind,tiled", LAYOUTS)
@pytest.mark.parametrize("B", SIZES)
def test_save_gives_canonical_rows(variant, kind, tiled, B):
    REC = rec_words(kind)
    Bpad = (B + 31) // 32 * 32
    rng = np.random.default_rng(B + 7 * kind + 3 * tiled)
    logical = bit_patterns((Bpad, REC), rng)
    rec = device_image(logical, tiled, REC)
    before = rec.copy()
    rows = np.full(B * REC + 64, 0xDEADBEEF, np.uint64)  # 64 guard words past the B rows
    transform(True, VARIANTS[variant], rec, rows, B, kind, tiled)
    assert np.array_equal(rows[: B * REC].reshape(B, REC), logical[:B])  # mu, then tri(r, c): the record's entry order
    assert (rows[B * REC:] == 0xDEADBEEF).all()  # nothing written past row B
    assert np.array_equal(rec, before)  # a save reads only


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("kind,tiled", LAYOUTS)
@pytest.mark.parametrize("B", SIZES)
def test_restore_writes_every_record_and_nothing_else(variant, kind, tiled, B):
    REC = rec_words(kind)
    Bpad = (B + 31) // 32 * 32
    rng = np.random.default_rng(1000 + B + 7 * kind + 3 * tiled)
    old = bit_patterns((Bpad, REC), rng)
    rec = device_image(old, tiled, REC)
    rows = bit_patterns((B, REC), rng)
    transform(False, VARIANTS[variant], rec, rows.reshape(-1).copy(), B, kind, tiled)
    want = old.copy()
    want[:B] = rows  # the padding lanes of a ragged last tile keep what they held
    assert np.array_equal(rec, device_image(want, tiled, REC))


@pytest.mark.parametrize("kind,tiled", LAYOUTS)
@pytest.mark.parametrize("B", SIZES)
def test_round_trip_is_bit_identical_across_variants(kind, tiled, B):
    """save with one variant, restore with the other into cleared records: the same bits come back"""
    REC = rec_words(kind)
    Bpad = (B + 31) // 32 * 32
    rng = np.random.default_rng(2000 + B + kind)
    logical = bit_patterns((Bpad, REC), rng)
    rec = device_image(logical, tiled, REC)
    for save_v, restore_v in ((0, 1), (1, 0), (1, 1)):
        rows = np.zeros(B * REC, np.uint64)
        transform(True, save_v, rec, rows, B, kind, tiled, grid=2, warps=1)
        back = device_image(np.zeros_like(logical), tiled, REC)
        transform(False, restore_v, back, rows, B, kind, tiled, grid=2, warps=3)
        want = np.concatenate([logical[:B], np.zeros((Bpad - B, REC), np.uint64)])
        assert np.array_equal(device_image(want, tiled, REC), back)  # uint64 words: NaN payloads and -0.0 compared as bits


def test_tile_layout_statement_matches_the_engine():
    """the NumPy tile_index above is the engine's: a record image laid out by it reads back through the per-element
    kernel, whose indexing is the engine's own rec_index"""
    B, kind = 70, 0
    REC = rec_words(kind)
    logical = np.arange(96 * REC, dtype=np.uint64).reshape(96, REC)
    rows = np.zeros(B * REC, np.uint64)
    transform(True, 0, device_image(logical, True, REC), rows, B, kind, True, grid=1)
    assert np.array_equal(rows.reshape(B, REC), logical[:B])


# ---- host-pointer entry points: refusals without a device -------------------------------------------------------------

def test_checkpoint_entry_points_refuse_without_crashing():
    from slam_pose_estimation_b200 import _build, _capi

    _build.build()
    lib = _capi.load()
    buf = np.zeros(1024, np.uint8)
    pb = buf.ctypes.data_as(C.c_void_p)
    n = C.c_uint64(7)
    for rc in (lib.ukfb_checkpoint_size(None, C.byref(n)), lib.ukfb_checkpoint_save(None, pb, buf.size),
               lib.ukfb_checkpoint_restore(None, pb, buf.size), lib.ukfb_checkpoint_save_dev(None, pb, buf.size),
               lib.ukfb_checkpoint_restore_dev(None, pb, buf.size)):
        assert rc == -1  # UKFB_ERR_INVALID: null handle
    assert n.value == 7 and not buf.any()  # nothing written on refusal


def test_python_front_end_refuses_other_image_types():
    from slam_pose_estimation_b200 import batch

    class Fake(batch.UkfBatch):
        def __init__(self):  # no handle: the type check comes first
            pass

    with pytest.raises(TypeError):
        Fake().restore(np.zeros(16, np.float64))
