"""What a checkpoint and a restore of a large batch cost (DESIGN.md section 7.6), next to plain copies of the same bytes.

One JSON line per measurement:
  op        save_dev | restore_dev | d2d_copy (cudaMemcpyAsync device -> device of the image's bytes, the HBM reference) |
            save | restore (host-pointer calls) | d2h_copy | h2d_copy (plain copies of the image's bytes, the link reference)
  kind      PoseUKF | OrientationUKF;  B, bytes (of the image)
  variant   tile | elem: the record transform (UKFB_CKPT_TRANSFORM, read once per process: the elem rows come from a
            second process, run by this one with --dev-only)
  host_mem  pinned (ukfb_host_alloc / pinned torch tensors) | pageable, for the host calls and copies
  devices   the handle's devices (one, or all of the box for a sharded handle)
  ms_median, ms_min, ms_max  per call, over `windows` windows of `reps` calls each; GB_s = bytes / ms_median
  dev ops:  CUDA events on the handle's stream around the window (restore_dev includes its synchronous header read);
  host ops: host clock around the window, each call blocking.
usage: python tools/bench_checkpoint.py [--batch 1048576] [--out profiles/r04_checkpoint.jsonl]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(pl.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        power = None
    return name, power


def spread(ms):
    return {"ms_median": statistics.median(ms), "ms_min": min(ms), "ms_max": max(ms)}


def dev_timed(x, fn, reps, windows):
    """per-call device ms of `reps` calls between events on the handle's stream, one value per window"""
    fn()
    x.synchronize()
    out = []
    for _ in range(windows):
        x.event_record(0)
        for _ in range(reps):
            fn()
        x.event_record(1)
        out.append(x.event_elapsed_ms(0, 1) / reps)
    return out


def host_timed(sync, fn, reps, windows):
    fn()
    sync()
    out = []
    for _ in range(windows):
        sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        sync()
        out.append((time.perf_counter() - t0) * 1e3 / reps)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_checkpoint.jsonl"))
    ap.add_argument("--dev-only", action="store_true", help="save_dev / restore_dev only, printed, nothing written")
    a = ap.parse_args()
    variant = "elem" if os.environ.get("UKFB_CKPT_TRANSFORM") == "elem" else "tile"
    import torch

    from slam_pose_estimation_b200 import UkfBatch, synthetic as syn

    if not torch.cuda.is_available():
        sys.exit("bench_checkpoint: no CUDA device -- this measures the engine on the GPU and has no CPU path")
    B = a.batch
    gpu, power = gpu_info()
    rows = []

    def emit(**kw):
        rec = {**kw, "B": B, "gpu": gpu, "power_limit_w": power}
        if "ms_median" in rec:
            rec["GB_s"] = rec["bytes"] / rec["ms_median"] / 1e6
        rows.append(rec)
        print(json.dumps(rec), flush=True)

    def make(kind, **kw):
        x = UkfBatch(kind, B, **kw)
        mu, sg = syn.pose_initial(B) if kind == 0 else syn.orientation_initial(B)
        x.initialize(mu, sg)
        x.predict_dt(syn.DT)
        return x

    for kind, name in ((0, "PoseUKF"), (1, "OrientationUKF")):
        x = make(kind)
        size = x.checkpoint_size()
        lib, h = x.lib, x.h
        base = {"kind": name, "bytes": size, "devices": [0]}
        d_img = torch.empty(size, dtype=torch.uint8, device="cuda")
        d_ref = torch.empty(size, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        p_img = C.c_void_p(d_img.data_ptr())
        save = dev_timed(x, lambda: x._chk(lib.ukfb_checkpoint_save_dev(h, p_img, size)), a.reps, a.windows)
        emit(op="save_dev", variant=variant, **base, **spread(save))
        restore = dev_timed(x, lambda: x._chk(lib.ukfb_checkpoint_restore_dev(h, p_img, size)), a.reps, a.windows)
        emit(op="restore_dev", variant=variant, **base, **spread(restore))
        if a.dev_only:
            x.close()
            del d_img, d_ref
            torch.cuda.empty_cache()
            continue
        stream = torch.cuda.ExternalStream(x.stream())
        with torch.cuda.stream(stream):
            d2d = dev_timed(x, lambda: d_ref.copy_(d_img), a.reps, a.windows)
        emit(op="d2d_copy", **base, **spread(d2d))

        reps = max(1, a.reps // 2)
        pinned = C.c_void_p()
        x._chk(lib.ukfb_host_alloc(C.byref(pinned), size))
        try:
            pageable = np.empty(size, np.uint8)  # referenced until the calls are done
            for mem in ("pinned", "pageable"):
                buf = pinned.value if mem == "pinned" else pageable.ctypes.data
                save = host_timed(x.synchronize, lambda: x._chk(lib.ukfb_checkpoint_save(h, C.c_void_p(buf), size)), reps, a.windows)
                emit(op="save", host_mem=mem, variant="tile", **base, **spread(save))
                restore = host_timed(x.synchronize, lambda: x._chk(lib.ukfb_checkpoint_restore(h, C.c_void_p(buf), size)), reps,
                                     a.windows)
                emit(op="restore", host_mem=mem, variant="tile", **base, **spread(restore))
        finally:
            lib.ukfb_host_free(pinned)
        for mem in ("pinned", "pageable"):
            h_t = torch.empty(size, dtype=torch.uint8, pin_memory=(mem == "pinned"))
            d2h = host_timed(torch.cuda.synchronize, lambda: h_t.copy_(d_img), reps, a.windows)
            emit(op="d2h_copy", host_mem=mem, **base, **spread(d2h))
            h2d = host_timed(torch.cuda.synchronize, lambda: d_ref.copy_(h_t), reps, a.windows)
            emit(op="h2d_copy", host_mem=mem, **base, **spread(h2d))
            del h_t
        img = x.checkpoint()
        del d_img, d_ref
        x.close()
        torch.cuda.empty_cache()

        n = torch.cuda.device_count()
        if n >= 2:  # one handle over every GPU of the box: the shards' copies run concurrently
            devs = list(range(n))
            s = UkfBatch(kind, B, devices=devs)
            s.restore(img)
            pinned = C.c_void_p()
            s._chk(s.lib.ukfb_host_alloc(C.byref(pinned), size))
            try:
                buf = C.c_void_p(pinned.value)
                save = host_timed(s.synchronize, lambda: s._chk(s.lib.ukfb_checkpoint_save(s.h, buf, size)), reps, a.windows)
                emit(op="save", host_mem="pinned", variant="tile", kind=name, bytes=size, devices=devs, **spread(save))
                restore = host_timed(s.synchronize, lambda: s._chk(s.lib.ukfb_checkpoint_restore(s.h, buf, size)), reps, a.windows)
                emit(op="restore", host_mem="pinned", variant="tile", kind=name, bytes=size, devices=devs, **spread(restore))
            finally:
                s.lib.ukfb_host_free(pinned)
            s.close()

    if a.dev_only:
        return
    env = dict(os.environ, UKFB_CKPT_TRANSFORM="elem")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--dev-only", "--batch", str(B), "--reps", str(a.reps),
                        "--windows", str(a.windows)], env=env, capture_output=True, text=True, check=True)
    for line in r.stdout.splitlines():
        if line.startswith("{"):
            rows.append(json.loads(line))
            print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
