"""The scenarios of tests/precision.py through the SIMT emulator's step kernels, judged block by block against the
long-double oracle (see tests/precision.py for the metric and the acceptance rule).

`fast` and `thread` run every scenario.  The emulated warp-per-group kernel costs about 0.1 s a launch (one host thread
per CUDA thread and a host barrier per __syncwarp), about 9 minutes over all nine scenarios, so here it runs the two
shortest: P4 (the nearly singular Cholesky) and O3 (the any-angle orientation).  tests/test_gpu_precision.py runs
all three kernels on every scenario, and profiles/r05_precision_emu.jsonl records the emulated warp kernel on all nine.
"""
from __future__ import annotations

import pytest

import precision as PR
from emu_lib import EmuBatch

CASES = [(name, kernel) for name in PR.SCENARIOS if name not in PR.TICK_SCENARIOS for kernel in ("fast", "thread")]
CASES += [("P4", "warp"), ("O3", "warp")]


@pytest.mark.parametrize("name,kernel", CASES)
def test_emulated_kernel_per_block_precision(name, kernel):
    _, fn = PR.SCENARIOS[name]
    PR.check(name, fn(lambda kind, B: EmuBatch(kind, B, kernel=kernel)), what=f"emu {kernel}")
