"""Per-filter access on a large batch: what reading back or re-initialising a few filters costs, against the whole-batch
calls a caller had before (DESIGN.md section 7.5).

One JSON line per measurement:
  op       get_state_indexed | initialize_indexed | find_status | get_state_dev | get_state | get_mu_range |
           host_workaround (get_state, patch one row, get_last_time, initialize, set_last_time)
  path     host (NumPy arrays, the call copies and synchronises) | dev (torch CUDA tensors, enqueue only)
  n, pattern (contiguous | sorted_random | unsorted_random), sigma (covariances too), flagged (find_status)
  device_ms  CUDA events on the handle's stream around `reps` calls, per call
  wall_ms    host clock around `reps` calls ending in a synchronise, per call (median of 3 such windows)
usage: python tools/bench_indexed.py [--batch 1048576] [--out profiles/r03_indexed_access.jsonl]
"""
from __future__ import annotations

import argparse
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
        power = float(pl)
    except (OSError, ValueError, subprocess.TimeoutExpired):
        power = None
    return name, power


def timed(x, fn, reps):
    """(device ms per call, wall ms per call)"""
    fn()  # warm: staging buffers, module load
    x.synchronize()
    x.event_record(0)
    for _ in range(reps):
        fn()
    x.event_record(1)
    dev = x.event_elapsed_ms(0, 1) / reps
    walls = []
    for _ in range(3):
        x.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        x.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3 / reps)
    return dev, statistics.median(walls)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_indexed_access.jsonl"))
    ap.add_argument("--sharded-batch", type=int, default=None, help="filters of the [0, 0, 0] line (default: --batch)")
    a = ap.parse_args()
    import torch

    from slam_pose_estimation_b200 import UkfBatch, synthetic as syn

    if not torch.cuda.is_available():
        sys.exit("bench_indexed: no CUDA device -- this measures the engine on the GPU and has no CPU path")
    B = a.batch
    gpu, power = gpu_info()
    common = {"B": B, "kind": "PoseUKF", "gpu": gpu, "power_limit_w": power}
    rows = []

    def emit(**kw):
        rec = {**kw, **common}
        rows.append(rec)
        print(json.dumps(rec), flush=True)

    x = UkfBatch(0, B)
    mu0, sg0 = syn.pose_initial(B, perturb=True)
    x.initialize(mu0, sg0)
    del mu0, sg0
    for k in range(1, 4):
        z, R = syn.pose_measurement(8, B, k)
        x.step(syn.DT, 8, z, R)
    rng = np.random.default_rng(1)
    sizes = [n for n in (1, 32, 1024, 32 * 1024, 1 << 20) if n <= B] or [B]

    def patterns(n):
        yield "contiguous", np.arange(B // 2 - n // 2, B // 2 - n // 2 + n) if n < B else np.arange(B)
        if n < B:
            yield "sorted_random", np.sort(rng.choice(B, n, replace=False))
        yield "unsorted_random", rng.permutation(B)[:n]

    # ---- baselines: the whole-batch calls ----
    d_mu_all = torch.empty((B, 13), dtype=torch.float64, device="cuda")
    d_sg_all = torch.empty((B, 12, 12), dtype=torch.float64, device="cuda")
    for sig in (False, True):
        dev, wall = timed(x, lambda: x.get_state_dev(d_mu_all, d_sg_all if sig else None), 10)
        emit(op="get_state_dev", path="dev", n=B, pattern="all", sigma=sig, device_ms=dev, wall_ms=wall)
    h_mu, h_sg = np.empty((B, 13)), np.empty((B, 12, 12))
    for sig in (False, True):
        dev, wall = timed(x, lambda: x.get_state_into(h_mu, h_sg if sig else None), 3)
        emit(op="get_state", path="host", n=B, pattern="all", sigma=sig, device_ms=dev, wall_ms=wall)
    h_pose = np.empty((B, 7))
    dev, wall = timed(x, lambda: x.get_mu_range(0, 7, h_pose), 3)
    emit(op="get_mu_range", path="host", n=B, pattern="all", sigma=False, mu_first=0, mu_count=7, device_ms=dev, wall_ms=wall)

    # ---- the five-step host workaround for ONE filter ----
    def workaround():
        mu, sg = x.get_state()
        mu[12345 % B] = mu[12345 % B]
        t = x.get_last_time()
        x.initialize(mu, sg)
        t[12345 % B] = 0
        x.set_last_time(t)

    dev, wall = timed(x, workaround, 1)
    emit(op="host_workaround", path="host", n=1, pattern="one", sigma=True, device_ms=dev, wall_ms=wall)

    # ---- indexed read-back and re-initialisation ----
    for n in sizes:
        reps = 20 if n <= 32 * 1024 else 5
        for pat, idx in patterns(n):
            idx = np.ascontiguousarray(idx, np.int64)
            d_idx = torch.as_tensor(idx, device="cuda")
            d_mu = torch.empty((n, 13), dtype=torch.float64, device="cuda")
            d_sg = torch.empty((n, 12, 12), dtype=torch.float64, device="cuda")
            for sig in (False, True):
                dev, wall = timed(x, lambda: x.get_state_indexed(idx, with_sigma=sig), reps)
                emit(op="get_state_indexed", path="host", n=n, pattern=pat, sigma=sig, device_ms=dev, wall_ms=wall)
                dev, wall = timed(x, lambda: x.get_state_indexed_dev(d_idx, d_mu, d_sg if sig else None), reps)
                emit(op="get_state_indexed", path="dev", n=n, pattern=pat, sigma=sig, device_ms=dev, wall_ms=wall)
            mu, sg = x.get_state_indexed(idx)  # re-initialised with their own states: the batch stays as it is
            dev, wall = timed(x, lambda: x.initialize_indexed(idx, mu, sg), reps)
            emit(op="initialize_indexed", path="host", n=n, pattern=pat, sigma=True, device_ms=dev, wall_ms=wall)
            d_mu.copy_(torch.as_tensor(mu))
            d_sg.copy_(torch.as_tensor(sg))
            dev, wall = timed(x, lambda: x.initialize_indexed_dev(d_idx, d_mu, d_sg), reps)
            emit(op="initialize_indexed", path="dev", n=n, pattern=pat, sigma=True, device_ms=dev, wall_ms=wall)
            del d_idx, d_mu, d_sg

    # ---- status lookup: 0, 1, 1 % and 100 % of the filters flagged (a time step above max_dt: DT_TOO_LARGE) ----
    for label, count in (("0", 0), ("1", 1), ("1%", B // 100), ("100%", B)):
        x.clear_status()
        if count:
            dt = np.full(B, syn.DT)
            dt[rng.permutation(B)[:count]] = 10.0
            x.set_time_bounds(1e-9, 1.0)
            x.predict_dt(dt)
            x.set_time_bounds(1e-9, np.finfo(float).max)
        found = x.find_status()
        assert found.size == count, (found.size, count)
        dev, wall = timed(x, lambda: x.find_status(), 20)
        emit(op="find_status", path="host", n=count, pattern="flagged", flagged=label, sigma=False, device_ms=dev, wall_ms=wall)
    x.clear_status()
    x.close()
    del h_mu, h_sg, d_mu_all, d_sg_all

    # ---- one sharded [0, 0, 0] handle ----
    Bs = a.sharded_batch or B
    s = UkfBatch(0, Bs, devices=[0, 0, 0])
    mu0, sg0 = syn.pose_initial(Bs, perturb=True)
    s.initialize(mu0, sg0)
    del mu0, sg0
    idx = rng.permutation(Bs)[:1024].astype(np.int64)
    dev, wall = timed(s, lambda: s.get_state_indexed(idx), 20)
    emit(op="get_state_indexed", path="host", n=1024, pattern="unsorted_random", sigma=True, shards=3, sharded_batch=Bs,
         device_ms=dev, wall_ms=wall)
    mu, sg = s.get_state_indexed(idx)
    dev, wall = timed(s, lambda: s.initialize_indexed(idx, mu, sg), 20)
    emit(op="initialize_indexed", path="host", n=1024, pattern="unsorted_random", sigma=True, shards=3, sharded_batch=Bs,
         device_ms=dev, wall_ms=wall)
    s.close()

    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
