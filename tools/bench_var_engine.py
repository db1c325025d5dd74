#!/usr/bin/env python
"""int8 (predict_i8.cu) vs DMMA variance engine: the cfg3 problem (bench.make_problem) and a cfg5 sweep (d = 5),
both engines alternating, CUDA events around each predict call.  Also reads the card's name and power limit and
measures the int8 peak of the same run (torch._int_mm at 8192^3, best of several).  One JSON line per point, also
appended to profiles/r03_var_engine.jsonl (or the path given as the first argument).

    python tools/bench_var_engine.py [out.jsonl]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from approxposterior_b200 import GP, kernels  # noqa: E402
import bench  # noqa: E402

REPEATS = 3
dev = torch.device("cuda", 0)
out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_var_engine.jsonl")


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    with open(out_path, "a") as f:
        f.write(line + "\n")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        name, plim = [s.strip() for s in r.stdout.strip().split(",")]
        return name, plim
    except Exception:
        return torch.cuda.get_device_name(0), "not read"


def int8_peak():
    if not hasattr(torch, "_int_mm"):
        return None
    try:
        a = torch.randint(-128, 127, (8192, 8192), dtype=torch.int8, device=dev)
        b = torch.randint(-128, 127, (8192, 8192), dtype=torch.int8, device=dev)
        for _ in range(3):
            torch._int_mm(a, b)
        best = float("inf")
        for _ in range(10):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12         # TOPS (two ops per MAC)
    except RuntimeError:
        return None


def time_engines(gp, q, N):
    Npad = (N + 63) // 64 * 64
    nblk = Npad // 64
    macs_i8 = 34 * sum((ib + 1) * 64 * 64 for ib in range(nblk))     # executed int8 MACs per query
    flop64 = float(N) * N                                              # algorithmic FP64 flop per query (triangle)
    ts = {"dmma": [], "i8": []}
    for eng in ts:                                                     # warm-up (the i8 pack happens here)
        gp.set_var_engine(eng)
        gp._predict_raw(q, True, utility="bape")
    torch.cuda.synchronize()
    for _ in range(REPEATS):
        for eng in ts:
            gp.set_var_engine(eng)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); gp._predict_raw(q, True, utility="bape"); e1.record(); torch.cuda.synchronize()
            ts[eng].append(e0.elapsed_time(e1))
    gp.set_var_engine("i8")
    Q = q.shape[0]
    rec = {"N": N, "Q": Q}
    for eng, v in ts.items():
        rec[eng + "_ms"] = float(np.median(v))
        rec[eng + "_spread_ms"] = float(max(v) - min(v))
        rec[eng + "_fp64_equiv_tflops"] = flop64 * Q / (np.median(v) * 1e-3) / 1e12
    rec["i8_int8_tops_executed"] = 2.0 * macs_i8 * Q / (rec["i8_ms"] * 1e-3) / 1e12
    rec["speedup"] = rec["dmma_ms"] / rec["i8_ms"]
    return rec


def main():
    name, plim = card()
    peak = int8_peak()
    emit({"card": name, "power_limit": plim,
          "int8_peak_tops_int_mm_8192": peak if peak is not None else "not measured"})
    X, y, logM, mean = bench.make_problem()
    d = X.shape[1]
    gp = GP(kernel=kernels.ExpSquaredKernel(np.exp(logM), ndim=d), fit_mean=True, mean=mean, white_noise=-12.0)
    gp.compute(X, y=y)
    g = torch.Generator(device=dev); g.manual_seed(1)
    q = -5.0 + 10.0 * torch.rand((1 << 20, d), dtype=torch.float64, device=dev, generator=g)
    rec = time_engines(gp, q, X.shape[0])
    rec.update(config="cfg3", card=name, power_limit=plim)
    if peak:
        rec["i8_share_of_int_mm_peak"] = rec["i8_int8_tops_executed"] / peak
    emit(rec)
    del gp, q
    for N in (256, 512, 1024, 2048, 4096, 8192):
        rng = np.random.default_rng(N + d)
        X = rng.uniform(-5, 5, size=(N, d)); y = rng.standard_normal(N)
        gp = GP(kernel=kernels.ExpSquaredKernel(np.full(d, float(d)), ndim=d), fit_mean=True, mean=0.0,
                white_noise=-12.0)
        gp.compute(X, y=y)
        q = -5.0 + 10.0 * torch.rand((1 << (20 if N <= 4096 else 18), d), dtype=torch.float64, device=dev, generator=g)
        rec = time_engines(gp, q, N)
        rec.update(config="cfg5", d=d, card=name, power_limit=plim)
        if peak:
            rec["i8_share_of_int_mm_peak"] = rec["i8_int8_tops_executed"] / peak
        emit(rec)
        del gp, q
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
