#!/usr/bin/env python
"""bench.py -- filter-steps/s of the batched PoseUKF predict+update hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU path (oracle port)
    torchrun ... bench.py --gpus N ...                        # one rank per GPU, filters sharded by index
    python bench.py ... --dump-outputs DIR                    # also write the state the timed steps computed

Workload (BASELINE.json config 4 at one GPU, SURVEY.md section 8(d) "C4"): 1,048,576
PoseUKF instances per GPU, Monte-Carlo initial states, one step = predictionStep(dt = 1 ms)
followed by integrateMeasurement(AngularVelocityMeasurement) (m = 3) for every filter, fused
in one kernel launch.  The filter records (768 B x 1 Mi = 805 MB) are far larger than the
126 MB L2, so every step streams them from HBM (no L2 flush needed).

One JSON line on stdout (rank 0).  `value` is device-timed (CUDA events on the engine's
stream) with inputs resident in HBM; `e2e` goes through the host-pointer C ABI calls with
pinned host buffers: H2D of the step's measurements and D2H of the state estimates inside
the timed region.  The CPU oracle is executed only for `cpu_baseline` / `--impl reference`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "PoseUKF predict+update filter-steps/s"
UNIT = "filter-steps/s"

# Algorithmic work per PoseUKF predict + m=3 update, SURVEY.md section 8(d) / Appendix B
# (contract figures; FMA = 2 flops; specials not counted): 41.7 kflop at k = 3 manifold-mean
# passes per mean, +-1.57 kflop per pass for each of the two state means of a step.
FLOPS_PER_STEP_K3 = 41.7e3
FLOPS_PER_MEAN_PASS = 1.57e3
MEANS_PER_STEP = 2
# state record in and out once (2 x (13 + 144) x 8 B = 2512 B) + dt 8 + z 24 + R 72 (section 8d)
HBM_BYTES_PER_STEP = 2.0 * (13 + 144) * 8 + 8 + 24 + 72


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(float(r[2]) for r in self.rows)}


def bind_to_gpu_numa_node(index: int):
    """Run this rank (and allocate its pinned staging buffers, first touch) on the CPUs NVML reports as closest to its
    GPU, so that the end-to-end copies of the 8 ranks do not all cross one socket's memory controller."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "first": min(cpus), "last": max(cpus)}
    except Exception as e:  # affinity is an optimisation only
        return {"error": str(e)[:80]}
    return None


R_SCALES = (0.25, 1.0, 4.0)  # BASELINE config 4 / SURVEY 8(d) "C4": measurement-covariance scale swept over the filters


def r_scale_of(idx: np.ndarray) -> np.ndarray:
    return np.asarray(R_SCALES)[np.asarray(idx) % len(R_SCALES)]


def make_workload(B: int, first: int, pool: int):
    """initial state (perturbed per filter), `pool` distinct measurement sets and the per-filter measurement covariance
    (sigma_gyro^2 I scaled by 0.25 / 1 / 4 along the sweep) for filters first..first+B"""
    from slam_pose_estimation_b200 import synthetic as syn

    mu, sg = syn.pose_initial(B, perturb=True, first=first)
    zs = np.empty((pool, B, 3))
    for j in range(pool):
        zs[j] = syn.pose_measurement(8, B, j + 1, first=first)[0]
    R = (np.eye(3) * syn.SIGMA_GYRO**2)[None] * r_scale_of(np.arange(first, first + B))[:, None, None]
    return mu, sg, zs, np.ascontiguousarray(R)


def make_workload_of(indices, pool: int):
    """the same as make_workload for an arbitrary list of global filter indices (the parity sample)"""
    parts = [make_workload(1, int(i), pool) for i in indices]
    return (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
            np.concatenate([p[2] for p in parts], axis=1), np.concatenate([p[3] for p in parts]))


def cpu_arm():
    """which CPU implementation the baseline legs time: oracle/_ref (the reference's own PoseUKF.cpp /
    UnscentedKalmanFilter.hpp compiled unmodified against oracle/ref_shim, over the restated ukfom / MTK engine) when it
    was built in the build container, else the oracle port.  Returns (variant, kind, description)."""
    from oracle import oracle_lib as O

    if os.path.exists(O.REF_LIB):
        return "ref", "reference", ("oracle/_ref: the reference's own wrapper sources (PoseUKF.cpp, UnscentedKalmanFilter.hpp) compiled "
                                    "unmodified; ukfom / MTK / Eigen underneath are the oracle's restatement (slam/mtk is not vendored)")
    return "left", "port", "oracle port (the reference could not be compiled here)"


def time_oracle(B: int, steps: int, warmup: int, threads: int | None = None):
    """the reference's CPU path (cpu_arm) on the same workload, OpenMP over filters; returns steps/s, threads, seconds"""
    from oracle.oracle_lib import OracleBatch
    from slam_pose_estimation_b200 import synthetic as syn

    mu, sg, zs, R = make_workload(B, 0, 4)
    o = OracleBatch(0, B, variant=cpu_arm()[0], threads=threads)
    o.initialize(mu, sg)
    for k in range(warmup):
        o.step(syn.DT, 8, zs[k % 4], R)
    t0 = time.perf_counter()
    for k in range(steps):
        o.step(syn.DT, 8, zs[k % 4], R)
    dt = time.perf_counter() - t0
    return B * steps / dt, o.max_threads(), dt


def parity_sample(applied, indices, mu_gpu, sg_gpu, pool: int):
    """replays the steps the engine has applied (`applied`: the measurement-set index of every step so far) on the CPU
    oracle for the sampled filters and returns the parity figures of tests/parity.py"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import parity as P
    from oracle.oracle_lib import OracleBatch
    from slam_pose_estimation_b200 import synthetic as syn

    mu0, sg0, zs, R = make_workload_of(indices, pool)
    o = OracleBatch(0, len(indices))
    o.initialize(mu0, sg0)
    for j in applied:
        o.step(syn.DT, 8, zs[j], R)
    mu_ref, sg_ref = o.get_state()
    return {"filters": len(indices), "steps_replayed": len(applied), "checker": "CPU oracle (oracle/), same inputs",
            "max_mu_err": float(P.mu_error(0, mu_gpu, mu_ref).max()), "max_sigma_err": float(P.sigma_error(sg_gpu, sg_ref).max()),
            "tolerance": 1e-9}


DUMP_FILTERS = 32768  # mu + sigma of this many filters: 41 MB of float64


def dump_outputs(out_dir, f, dev):
    """--dump-outputs: the state estimates (ukfb_get_state) of a fixed sample of DUMP_FILTERS filters (seeded, in index
    order; every filter when there are fewer) as DIR/mu.npy (S x 13) and DIR/sigma.npy (S x 12 x 12), float64.  The
    inputs depend on the arguments only, so two builds of the engine can be compared output for output."""
    import torch

    B = f.B
    idx = np.arange(B) if B <= DUMP_FILTERS else np.sort(np.random.default_rng(0).choice(B, DUMP_FILTERS, replace=False))
    d_mu = torch.empty((B, f.MU), dtype=torch.float64, device=dev)
    d_sg = torch.empty((B, f.n, f.n), dtype=torch.float64, device=dev)
    f.get_state_dev(d_mu, d_sg)
    d_idx = torch.from_numpy(idx).to(dev)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "mu.npy"), d_mu[d_idx].cpu().numpy())
    np.save(os.path.join(out_dir, "sigma.npy"), d_sg[d_idx].cpu().numpy())


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (cpu_arm: oracle/_ref, else the oracle port), OpenMP over filters on
    all host cores.  Rank 0 only."""
    if rank != 0:
        return
    B = args.ref_filters
    per_step_s = None
    # every host thread this process may use, whatever OMP_NUM_THREADS says (torchrun sets it to 1 per rank)
    ncpu = len(os.sched_getaffinity(0))
    value, threads, _ = time_oracle(B, 2, 1, threads=ncpu)  # calibrate
    per_step_s = B / value
    # bound the whole run to ~ 2 minutes
    budget = 120.0
    total_steps = args.steps + args.warmup
    while B > 256 and per_step_s * total_steps > budget:
        B //= 2
        per_step_s /= 2
    value, threads, dt = time_oracle(B, args.steps, args.warmup, threads=ncpu)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C4: PoseUKF Monte-Carlo sweep sharded by filter index; step = predictionStep(1 ms) + "
                               "AngularVelocityMeasurement update (m=3)",
                   "sample": f"{B} filters of the sweep per step on the host cores ({cpu_arm()[2]}; OpenMP over filters)",
                   "filters": B},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": cpu_arm()[1],
                         "sample": f"{B} filters x {args.steps} steps, OpenMP over filters; {cpu_arm()[2]}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def timed_steps(f, step, steps, warmup, barrier, max_over_ranks):
    """`warmup` untimed then `steps` timed calls of step(k) on handle f: device-timed with CUDA events on the engine's
    stream, barrier + synchronize on both sides, max over ranks.  Returns ms for the `steps` calls."""
    for k in range(warmup):
        step(k)
    barrier()
    f.event_record(0)
    for k in range(steps):
        step(warmup + k)
    f.event_record(1)
    barrier()
    return max_over_ranks(f.event_elapsed_ms(0, 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--filters", type=int, default=1 << 20, help="filters per GPU")
    ap.add_argument("--ref-filters", type=int, default=4096)
    ap.add_argument("--pool", type=int, default=4, help="distinct measurement sets cycled through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-literal", action="store_true", help="skip the secondary measurement of the literal kernel")
    ap.add_argument("--no-orientation", action="store_true", help="skip the secondary OrientationUKF (C2) figure")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (1 Mi filters in total) at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state after the last timed step (a fixed sample of "
                                                          "rank 0's filters) to DIR/mu.npy and DIR/sigma.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the engine has no CPU path"}), flush=True)
        return 2
    torch.cuda.set_device(local)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from slam_pose_estimation_b200 import _build, synthetic as syn
    from slam_pose_estimation_b200.batch import UkfBatch
    from slam_pose_estimation_b200.shard import gather_estimates

    if not os.path.exists(_build.LIB):
        raise RuntimeError("lib/libukfb.so missing -- run __graft_entry__.build()")

    B = args.filters
    pool = args.pool
    first = rank * B  # contiguous shard [rank*B, (rank+1)*B) of a world*B Monte-Carlo sweep
    mu0, sg0, zs, R = make_workload(B, first, pool)
    f = UkfBatch(0, B, device=local)
    f.initialize(mu0, sg0)
    f.set_measurement_cov(8, R)  # the sensor covariances stay on the device: a streaming caller sends z only
    dev = torch.device("cuda", local)
    d_dt = torch.full((1,), syn.DT, dtype=torch.float64, device=dev)
    d_R = torch.from_numpy(R).to(dev)
    d_z = [torch.from_numpy(zs[j]).to(dev) for j in range(pool)]
    torch.cuda.synchronize()
    applied = []  # measurement-set index of every step handle f has taken (the parity sample replays them)

    def barrier():
        f.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-timed: inputs resident in HBM --------------------------------------------------
    def dev_step(k):
        applied.append(k % pool)
        f.step_dev(d_dt, False, 8, d_z[k % pool], d_R, True)

    for k in range(args.warmup):
        dev_step(k)
    f.clear_mean_iter_hist()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = f.launch_count()
    f.event_record(0)
    for k in range(args.steps):
        dev_step(args.warmup + k)
    f.event_record(1)
    barrier()
    ms = max_over_ranks(f.event_elapsed_ms(0, 1))
    launches = f.launch_count() - launches0
    hist = f.get_mean_iter_hist()
    n_flag, bits = f.status_summary()
    if args.dump_outputs and rank == 0:  # before the end-to-end legs below take further steps on f
        dump_outputs(args.dump_outputs, f, dev)

    # ---- end to end through the host-pointer C ABI ----------------------------------------------
    # Every step: H2D of that step's measurements from pinned host memory, the fused kernel, D2H of the estimates into
    # pinned host memory.  `e2e` uses the streaming calls (ukfb_step_async / ukfb_get_state_async: copy-in, compute and
    # copy-out streams, two staging slots each, so step k+1's input copy and kernel overlap step k's output copy) and
    # reads back the whole B x 13 mean; `pose_only` reads back position + orientation (7 of the 13 entries, what a
    # consumer of BodyStateMeasurement's pose needs); `blocking` uses the blocking calls.
    e2e = None
    if not args.no_e2e:
        z_pin = [torch.from_numpy(zs[j]).pin_memory() for j in range(pool)]
        z_np = [t.numpy() for t in z_pin]
        dt_pin = torch.full((1,), syn.DT, dtype=torch.float64).pin_memory()
        mu_pin = [torch.empty((B, 13), dtype=torch.float64).pin_memory() for _ in range(2)]
        mu_np = [t.numpy() for t in mu_pin]
        pose_np = [torch.empty((B, 7), dtype=torch.float64).pin_memory().numpy() for _ in range(2)]

        def e2e_loop(step, read, n):
            for k in range(n):
                applied.append(k % pool)
                step(k)
                read(k)
            f.synchronize()

        blk = (lambda k: f.step(syn.DT, 8, z_np[k % pool], None), lambda k: f.get_state_into(mu_np[0]))
        full = (lambda k: f.step_async(dt_pin.numpy(), 8, z_np[k % pool], None), lambda k: f.get_state_async(mu_np[k & 1]))
        pose = (lambda k: f.step_async(dt_pin.numpy(), 8, z_np[k % pool], None), lambda k: f.get_mu_range_async(0, 7, pose_np[k & 1]))
        res = {}
        for name, (step, read) in (("blocking", blk), ("full", full), ("pose_only", pose)):
            e2e_loop(step, read, 3)
            barrier()
            t0 = time.perf_counter()
            e2e_loop(step, read, args.steps)
            res[name] = max_over_ranks(time.perf_counter() - t0)
            barrier()
        e2e_s = res["full"]
        e2e = {"value": world * B * args.steps / e2e_s, "unit": UNIT,
               "h2d_bytes_per_step": int(B * 3 * 8 + 8), "d2h_bytes_per_step": int(B * 13 * 8),
               "ms_per_step": e2e_s / args.steps * 1e3,
               "api": "ukfb_step_async(host z; per-filter R kept on the device by ukfb_set_measurement_cov) + "
                      "ukfb_get_state_async(host mu) per step, pinned host buffers, one ukfb_synchronize at the end; copies "
                      "of step k overlap the kernel of step k+1",
               "pose_only": {"value": world * B * args.steps / res["pose_only"], "ms_per_step": res["pose_only"] / args.steps * 1e3,
                             "d2h_bytes_per_step": int(B * 7 * 8),
                             "api": "the same with ukfb_get_mu_range_async(0, 7): position + orientation only"},
               "blocking": {"value": world * B * args.steps / res["blocking"], "ms_per_step": res["blocking"] / args.steps * 1e3,
                            "api": "ukfb_step + ukfb_get_state, each returning after its own copies"}}
        assert np.isfinite(mu_np[0]).all() and np.isfinite(mu_np[1]).all()
        assert np.array_equal(pose_np[(args.steps - 1) & 1], f.get_mu_range(0, 7))
    sampler.stop()
    clocks = sampler.summary()

    # ---- the final gather of the estimates and a parity sample against the CPU oracle ----------------------------------
    # N > 1: every rank's B x 13 means travel to rank 0 (one torch.distributed gather over NCCL, then one D2H): the only
    # cross-GPU traffic of the job.  The sample: S filters per rank at a stride through the shard, mean AND covariance,
    # compared with the oracle replaying the very steps applied above.
    S = 8
    loc = (np.arange(S) * (B // S)).astype(np.int64)
    d_mu = torch.empty((B, 13), dtype=torch.float64, device=dev)
    d_sg = torch.empty((B, 12, 12), dtype=torch.float64, device=dev)
    if world > 1:  # NCCL sets its channels up on first use, and for a message of this size: not part of the transfer being timed
        gather_estimates(torch.zeros((world, 13), dtype=torch.float64, device=dev)[rank:rank + 1], world)
        gather_estimates(d_mu, world * B)  # same shapes as the timed one (contents: whatever the allocation held)
    # the host side of the gather: page-locked, allocated before the clock starts (a pageable destination is what a first
    # version of this leg timed: 0.4 s for 0.87 GB, none of it the transfer)
    host_mu = torch.empty((world * B if rank == 0 else 1, 13), dtype=torch.float64).pin_memory()
    barrier()
    t0 = time.perf_counter()
    f.get_state_dev(d_mu, d_sg)
    f.synchronize()
    gathered = None
    if world > 1:
        gathered = gather_estimates(d_mu, world * B)
        if rank == 0:
            gathered = host_mu.copy_(gathered, non_blocking=True)
    else:
        gathered = host_mu.copy_(d_mu, non_blocking=True)
    torch.cuda.synchronize()
    gather_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    smp_mu, smp_sg = d_mu[torch.from_numpy(loc).to(dev)], d_sg[torch.from_numpy(loc).to(dev)]
    if world > 1:
        mus = [torch.empty_like(smp_mu) for _ in range(world)]
        sgs = [torch.empty_like(smp_sg) for _ in range(world)]
        dist.all_gather(mus, smp_mu)
        dist.all_gather(sgs, smp_sg)
        smp_mu, smp_sg = torch.cat(mus), torch.cat(sgs)
    del d_sg
    gather = None
    if rank == 0:
        gidx = np.concatenate([r * B + loc for r in range(world)])
        assert np.array_equal(gathered.numpy()[gidx], smp_mu.cpu().numpy())  # the gathered buffer is in filter order
        gather = {"ms": gather_ms, "bytes": int(world * B * 13 * 8),
                  "api": "ukfb_get_state_dev per rank + one torch.distributed.gather (NCCL) + D2H on rank 0" if world > 1
                         else "ukfb_get_state_dev + D2H",
                  "parity_sample": parity_sample(applied, gidx, smp_mu.cpu().numpy(), smp_sg.cpu().numpy(), pool)}
    del gathered, d_mu, host_mu

    # ---- strong scaling: BASELINE config 4 proper, ONE batch of 1 Mi filters sharded over the N GPUs ---------------------
    strong = None
    if world > 1 and not args.no_strong:
        total = 1 << 20
        Bs = total // world
        mu_s, sg_s, zs_s, R_s = make_workload(Bs, rank * Bs, pool)
        fs = UkfBatch(0, Bs, device=local)
        fs.initialize(mu_s, sg_s)
        fs.set_measurement_cov(8, R_s)
        ds_R = torch.from_numpy(R_s).to(dev)
        ds_z = [torch.from_numpy(zs_s[j]).to(dev) for j in range(pool)]
        torch.cuda.synchronize()

        def sbarrier():
            fs.synchronize()
            torch.cuda.synchronize()
            dist.barrier()

        reps = max(args.steps, 20) * 4  # short launches: more of them for a stable figure
        s_ms = timed_steps(fs, lambda k: fs.step_dev(d_dt, False, 8, ds_z[k % pool], ds_R, True), reps, args.warmup, sbarrier, max_over_ranks)
        per_step = s_ms / reps
        tiles = (Bs + 31) // 32
        resident = 148 * 8
        strong = {"filters_total": total, "filters_per_gpu": Bs, "value": total / (per_step * 1e-3), "unit": UNIT,
                  "ms_per_step": per_step, "steps": reps,
                  "efficiency_vs_one_gpu_launch": (ms / args.steps) / (world * per_step),
                  "note": "efficiency = time of the 1 Mi-filter launch on one GPU (the weak leg above, same kernel) / (N x this "
                          "leg's time per step)",
                  "warps_per_gpu": tiles, "resident_warps_per_gpu": resident, "waves": tiles / resident}
        if not args.no_e2e:
            zs_pin = [torch.from_numpy(zs_s[j]).pin_memory().numpy() for j in range(pool)]
            dts_pin = torch.full((1,), syn.DT, dtype=torch.float64).pin_memory().numpy()
            mus_pin = [torch.empty((Bs, 13), dtype=torch.float64).pin_memory().numpy() for _ in range(2)]
            for k in range(3):
                fs.step_async(dts_pin, 8, zs_pin[k % pool], None)
                fs.get_state_async(mus_pin[k & 1])
            sbarrier()
            t0 = time.perf_counter()
            for k in range(reps):
                fs.step_async(dts_pin, 8, zs_pin[k % pool], None)
                fs.get_state_async(mus_pin[k & 1])
            fs.synchronize()
            se = max_over_ranks(time.perf_counter() - t0)
            sbarrier()
            strong["e2e"] = {"value": total * reps / se, "ms_per_step": se / reps * 1e3,
                             "h2d_bytes_per_step": int(Bs * 3 * 8 + 8), "d2h_bytes_per_step": int(Bs * 13 * 8)}
        fs.close()

    # ---- the literal kernel on the same workload (secondary figure) -----------------------------------
    # UKFB_KERNEL=thread selects ukf_thread.cuh at ukfb_create: every sigma point of every pass is pushed through
    # boxplus / model / boxminus exactly in the reference's sequence.  The default kernel (ukf_pose_fast.cuh) computes
    # the same estimator with the closed forms its header lists.
    literal = None
    if not args.no_literal:
        f.close()
        os.environ["UKFB_KERNEL"] = "thread"
        g = UkfBatch(0, B, device=local)
        os.environ.pop("UKFB_KERNEL")
        g.initialize(mu0, sg0)

        def gbarrier():
            g.synchronize()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()

        lit_ms = timed_steps(g, lambda k: g.step_dev(d_dt, False, 8, d_z[k % pool], d_R, True), args.steps, args.warmup, gbarrier, max_over_ranks)
        literal = {"kernel": "ukf_thread_kernel<PoseF>", "value": world * B * args.steps / (lit_ms * 1e-3), "unit": UNIT,
                   "ms_per_step": lit_ms / args.steps}
        fp64_peak = g.measure_fp64_peak() if rank == 0 else 0.0
        g.close()
    else:
        fp64_peak = f.measure_fp64_peak() if rank == 0 else 0.0

    # ---- BASELINE.json config 2 (secondary figure): 65,536 OrientationUKF on a 1 kHz IMU stream ----------------------
    # 100 ticks per launch (ukfb_run_dev: IMU sample stored + predict every tick, one body-velocity update on the last
    # tick), state on chip between ticks; ukf_ori_fast_kernel.  Contract flops: SURVEY.md 8(d) 22.7 kflop per predict at
    # k = 3 mean passes, -1.747 kflop per pass; 27.8 kflop per update likewise.
    orientation = None
    if not args.no_orientation and world == 1:
        Bo, Ko = 65536, 100
        mu_o, sg_o = syn.orientation_initial(Bo)
        g = UkfBatch(1, Bo, device=local)
        g.set_orientation_params(syn.ORI_TAU, syn.ORI_TAU, syn.LATITUDE_BREMEN)
        g.initialize(mu_o, sg_o)
        g.set_process_noise(syn.ORI_Q)
        imu = np.empty((4, Bo, 6))
        for j in range(4):
            imu[j, :, :3], imu[j, :, 3:] = syn.orientation_imu(Bo, j + 1)
        d_imu = torch.from_numpy(imu).to(dev)[torch.arange(Ko, device=dev) % 4].contiguous()
        kinds_o = np.full(Ko, -1, np.int8)
        kinds_o[Ko - 1] = 9
        d_zo = torch.from_numpy(syn.orientation_velocity(Bo, 1)[0]).to(dev)[None].expand(Ko, Bo, 3).contiguous()
        d_Ro = torch.from_numpy(np.tile(np.eye(3) * syn.SIGMA_DVL**2, (Ko, 1, 1))).to(dev)
        d_dto = torch.full((Ko,), syn.DT, dtype=torch.float64, device=dev)
        torch.cuda.synchronize()  # the inputs above were produced on torch's stream (run_dev also orders itself after it)
        for _ in range(2):
            g.run_dev(Ko, d_dto, False, kinds_o, d_zo, d_Ro, False, d_imu)
        g.synchronize()
        g.clear_mean_iter_hist()
        reps = 5
        g.event_record(0)
        for _ in range(reps):
            g.run_dev(Ko, d_dto, False, kinds_o, d_zo, d_Ro, False, d_imu)
        g.event_record(1)
        g.synchronize()
        o_ms = g.event_elapsed_ms(0, 1) / reps
        oh = g.get_mean_iter_hist()
        o_passes = float((oh * np.arange(8)).sum() / max(1, oh.sum()))
        o_flops = Ko * (22.7e3 + (o_passes - 3.0) * 1.747e3) + (27.8e3 + (o_passes - 3.0) * 1.747e3)
        orientation = {"workload": "C2: 65,536 OrientationUKF, 1 kHz IMU stream, 100 ticks per launch (store IMU + predict), "
                                   "velocity update on the last tick", "kernel": "ukf_ori_fast_kernel",
                       "value": Bo * Ko / (o_ms * 1e-3), "unit": "filter-ticks/s", "launch_ms": o_ms, "mean_passes_avg": o_passes,
                       "flops_per_launch_per_filter": o_flops, "achieved_tflops": o_flops * Bo / (o_ms * 1e-3) / 1e12,
                       "status_flagged": int(g.status_summary()[0])}
        g.close()

    # ---- roofline -------------------------------------------------------------------------------
    passes = float((hist * np.arange(8)).sum() / max(1, hist.sum()))
    flops_step = FLOPS_PER_STEP_K3 + (passes - 3.0) * MEANS_PER_STEP * FLOPS_PER_MEAN_PASS
    launch_s = ms * 1e-3 / args.steps
    achieved_flops = flops_step * B / launch_s
    achieved_gbs = HBM_BYTES_PER_STEP * B / launch_s / 1e9
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # ncu figures of the dominant kernel (one `ncu --set full` capture, profiles/): only reported when the capture was
    # taken from the kernel sources this library is built from
    prof = {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    prof_current = bool(prof) and prof.get("source_sha16") == _build.source_hash()
    traffic = prof.get("dram_bytes_per_launch") if (prof_current and B == (1 << 20)) else None
    executed = None
    if prof_current and prof.get("executed_fp64_flops_per_step") and fp64_peak:
        ex = float(prof["executed_fp64_flops_per_step"]) * B / launch_s
        executed = {"flops_per_step": prof["executed_fp64_flops_per_step"], "achieved": ex / 1e12, "frac": ex / fp64_peak,
                    "fp64_pipe_active_pct_ncu": prof.get("fp64_pipe_active_pct"),
                    "source": "ncu op counts of this kernel on this workload (profiles/traffic.json, same source hash as the "
                              "loaded library) / this run's launch time"}
    if orientation and fp64_peak:
        orientation["roofline_frac"] = orientation["achieved_tflops"] * 1e12 / fp64_peak
    if literal and fp64_peak:
        literal["roofline_frac"] = flops_step * B / (literal["ms_per_step"] * 1e-3) / fp64_peak

    value = world * B * args.steps / (ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C4: PoseUKF Monte-Carlo sweep (initial states drawn per filter, measurement covariance scaled "
                               "x0.25 / x1 / x4 along the sweep) sharded by filter index; step = predictionStep(1 ms) + "
                               "AngularVelocityMeasurement update (m=3), one fused launch",
                   "filters_per_gpu": B, "filters_total": world * B, "parallelism": f"filter-shard x{world}, no collective on the step path",
                   "l2": "state records 805 MB per GPU >> 126 MB L2 (inputs larger than L2)" if B * 768 > 3 * 126e6 else "inputs smaller than L2",
                   "mean_passes_avg": passes, "status_flagged": int(n_flag), "rank0_cpu_affinity": numa,
                   "kernel_source_sha16": _build.source_hash()},
        "clocks": clocks,
        "gpu_launches": int(launches),
        "roofline": {"bound": "fp64", "achieved": achieved_flops / 1e12, "peak": fp64_peak / 1e12, "unit": "TFLOP/s",
                     "frac": (achieved_flops / fp64_peak) if fp64_peak else None, "traffic": traffic,
                     "traffic_note": None if prof_current else "profiles/traffic.json was captured from other kernel sources: not reported",
                     "peak_source": "measured in this run: independent-DFMA microkernel (MEASURED_PEAKS.json holds no FP64 figure)",
                     "flops_per_step": flops_step, "flops_per_step_contract_k3": FLOPS_PER_STEP_K3,
                     "flops_basis": "SURVEY.md 8(d): algorithmic flops of the reference's sigma-point sequence per step; the "
                                    "kernel reaches the same result with fewer executed operations, see `executed`",
                     "executed": executed, "literal_kernel": literal,
                     "kernel": "ukf_pose_fast_kernel", "launch_ms": launch_s * 1e3,
                     "hbm": {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                             "bytes_per_step": HBM_BYTES_PER_STEP,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"}},
    }
    if e2e:
        line["e2e"] = e2e
    if gather:
        line["gather"] = gather
    if strong:
        line["strong_1M"] = strong
    if orientation:
        line["orientation_c2"] = orientation
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        os.sched_setaffinity(0, all_cpus)  # the CPU baseline gets every host core
        v, threads, dt = time_oracle(args.ref_filters, 2, 1, threads=len(all_cpus))  # calibrate, then ~10 s of CPU work
        nsteps = int(min(20000, max(4, 12.0 / (dt / 2))))  # about 12 s of CPU work
        v, threads, dt = time_oracle(args.ref_filters, nsteps, 1, threads=len(all_cpus))
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": cpu_arm()[1],
                                "sample": f"{args.ref_filters} filters x {nsteps} steps of the same workload, OpenMP over filters, "
                                          f"{dt:.1f} s; {cpu_arm()[2]}"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
