#!/usr/bin/env python
"""Per-phase SM-cycle breakdown of predict_var_i8_kernel (predict_i8.cu) at cfg3 (bench.make_problem, 2^20 queries,
mean + variance + BAPE utility) from the -DAPGP_PROF build.  Run as

    APGP_LIB=approxposterior_b200/libapgp_prof.so APGP_PROF_PRINT=1 python tools/profile_var_i8_phases.py [label]

The library prints one '[i8prof]' line per profiled CTA (the first four of the grid, ranks 0-3 of group 0) per call
to stderr; this script captures them for one call after a warm-up and prints, per CTA, cycles per tile of each phase
and its share of the kernel's cycles (see the slot list at the top of predict_i8.cu)."""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from approxposterior_b200 import GP, kernels  # noqa: E402
import bench  # noqa: E402

NAMES = ["phase1_panel", "group_barrier_wait", "finaliser", "mma_wait_full", "mma_wait_accempty", "mma_issue",
         "mma_wait_last_epilogue", "phase2_wall", "kernel_total"]


def main():
    label = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("APGP_LIB", "default")
    X, y, logM, mean = bench.make_problem()
    d = X.shape[1]
    gp = GP(kernel=kernels.ExpSquaredKernel(np.exp(logM), ndim=d), fit_mean=True, mean=mean, white_noise=-12.0)
    gp.compute(X, y=y)
    gp.set_var_engine("i8")
    g = torch.Generator(device="cuda:0"); g.manual_seed(1)
    q = -5.0 + 10.0 * torch.rand((1 << 20, d), dtype=torch.float64, device="cuda:0", generator=g)
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            gp._predict_raw(q, True, utility="bape")        # warm-up (operand pack)
            torch.cuda.synchronize()
            tmp.write("#measured\n"); tmp.flush()
            gp._predict_raw(q, True, utility="bape")
            torch.cuda.synchronize()
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        text = tmp.read()
    lines = [ln for ln in text.split("#measured", 1)[-1].splitlines() if ln.startswith("[i8prof]")]
    if not lines:
        raise SystemExit("no [i8prof] lines: run with the -DAPGP_PROF library and APGP_PROF_PRINT=1")
    print(f"# {label}: cfg3 N={X.shape[0]} Q={q.shape[0]}  device {torch.cuda.get_device_name(0)}")
    for ln in lines:
        head, vals = ln.split("cycles:")
        v = [int(t) for t in vals.split()]
        tiles = max(v[9], 1)
        tot = v[8]
        parts = "  ".join(f"{n}={v[i] / tiles:.0f} ({100.0 * v[i] / tot:.1f}%)" for i, n in enumerate(NAMES))
        print(f"{head.strip()} tiles={v[9]}  per tile: {parts}")
        if len(v) > 11 and v[10] and v[11]:
            # the group planner's c1: one panel block's cost in phase-2 units (one 64-wide k-stage of a block-row)
            p1 = v[0] / v[10]
            p2 = v[7] / v[11]
            print(f"    panel blocks/tile {v[10] / tiles:.2f}, phase-2 units/tile {v[11] / tiles:.2f}: "
                  f"{p1:.0f} cycles per panel block, {p2:.0f} cycles per phase-2 unit -> c1 = {p1 / p2:.3f} units")


if __name__ == "__main__":
    main()
