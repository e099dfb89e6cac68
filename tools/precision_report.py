#!/usr/bin/env python
"""tools/precision_report.py -- the per-block accuracy table of tests/precision.py as JSON lines.

Runs every scenario of tests/precision.py through the FP64 oracle and through the step kernels `fast`, `thread` and
`warp`, in the SIMT emulator (--impl emu, no GPU) or on the GPU through UkfBatch (--impl gpu), and prints one line per
scenario, implementation, block and quantity (mean or covariance): the error in standard deviations of the long-double
oracle's state, the FP64 oracle's error, their ratio and whether the acceptance rule holds.  The first line names the
machine: for --impl gpu the device and its power limit.

    python tools/precision_report.py --impl emu > profiles/r05_precision_emu.jsonl
    python tools/precision_report.py --impl gpu > profiles/r05_precision_b200.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import platform
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

KERNELS = ("fast", "thread", "warp")


def _gpu_factory(kernel: str):
    from slam_pose_estimation_b200.batch import UkfBatch

    def make(kind, B):
        os.environ["UKFB_KERNEL"] = kernel  # read by ukfb_create
        return UkfBatch(kind, B)

    return make


def _emu_factory(kernel: str):
    from emu_lib import EmuBatch

    return lambda kind, B: EmuBatch(kind, B, kernel=kernel)


def _machine(impl: str) -> dict:
    head = {"impl": impl, "cpu": platform.processor() or platform.machine()}
    if impl == "gpu":
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True).stdout.splitlines()[0]
        head["gpu"], head["power_limit"] = (s.strip() for s in q.split(","))
    return head


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--impl", choices=("emu", "gpu"), required=True)
    ap.add_argument("--scenarios", default=None, help="comma-separated ids (default: all)")
    args = ap.parse_args()

    import numpy as np

    import precision as PR

    print(json.dumps(_machine(args.impl)), flush=True)
    factory = _gpu_factory if args.impl == "gpu" else _emu_factory
    names = args.scenarios.split(",") if args.scenarios else [n for n in PR.SCENARIOS if n not in PR.TICK_SCENARIOS]
    for name in names:
        kind, fn = PR.SCENARIOS[name]
        ld, d = PR.oracle_runs(name)
        ref, fp64 = ld.get_state(), d.get_state()
        same = bool(np.array_equal(ld.get_status(), d.get_status())
                    and np.array_equal(ld.get_mean_iter_hist(), d.get_mean_iter_hist()))
        impls = [("oracle_fp64", d)] + [(f"{args.impl}_{k}", fn(factory(k))) for k in KERNELS]
        for label, x in impls:
            branches = bool(np.array_equal(x.get_status(), d.get_status())
                            and np.array_equal(x.get_mean_iter_hist(), d.get_mean_iter_hist()))
            for blk, what, err, e64 in PR.judge(kind, x.get_state(), fp64, ref):
                print(json.dumps({"scenario": name, "impl": label, "block": blk, "kind": what, "err": err,
                                  "err_fp64_oracle": e64, "ratio": err / e64 if e64 > 0 else None,
                                  "pass": not PR.failures([(blk, what, err, e64)]),
                                  "branches_match_oracle": branches, "ld_fp64_branches_match": same}), flush=True)


if __name__ == "__main__":
    main()
