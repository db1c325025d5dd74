#!/usr/bin/env python
"""cfg4-shaped batched log-likelihood WITH gradients (R restarts, d = 10, P = 12) beyond the one-CTA class: the cluster
kernel with gradients (apgp_loglik_batch path 4) against the same call value-only (path 2) and against the per-vector
fallback (value kernel + one full factorisation and gradient per vector, forced with APGP_LOGLIK_PATH=group); plus
optimizeGP(method="l-bfgs-b") wall time on both routes.  One JSON object per line; the first names the card and its power
limit.  Usage: python tools/bench_loglik_grad.py [N ...]

Algorithmic flop count of one gradient evaluation:
  F_llg = F_ll + 2 N^3 / 3 + P N^2
  F_ll  = N^3 / 3 + 2 N^2 + (3 d + 1) N^2 / 2     (SURVEY 8(d): covariance build, Cholesky, forward substitution)
  + N^3 / 3 for the triangular inverse W = L^{-1}, + N^3 / 3 for the lower triangle of W^T W, + P N^2 for the trace products.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from approxposterior_b200 import GP, _lib, gpUtils, kernels  # noqa: E402
import ctypes  # noqa: E402

DEV = torch.device("cuda", 0)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    name, power, clock = [v.strip() for v in q.split(",")]
    return dict(gpu=name, power_limit=power, sm_clock_max=clock)


def dgemm_peak():
    a = torch.randn(8192, 8192, dtype=torch.float64, device=DEV); b = torch.randn_like(a)
    torch.matmul(a, b); torch.cuda.synchronize()
    best = 1e9
    for _ in range(4):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2 * 8192 ** 3 / best * 1e-9


def branin(u, v):
    return (v - 5.1 / (4 * np.pi ** 2) * u ** 2 + 5 / np.pi * u - 6) ** 2 + 10 * (1 - 1 / (8 * np.pi)) * np.cos(u) + 10


def path_of(gp):
    p = ctypes.c_int(-1)
    _lib.check(_lib.load().apgp_debug_last_loglik_path(gp._h, ctypes.byref(p)), "apgp_debug_last_loglik_path")
    return p.value


def timed(fn, min_s=0.3, max_reps=50):
    fn()                                                          # warm-up of this shape
    reps, t0 = 0, time.perf_counter()
    while True:
        fn()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_s or reps >= max_reps:
            return dt / reps


def setenv(path):
    if path is None:
        os.environ.pop("APGP_LOGLIK_PATH", None)
    else:
        os.environ["APGP_LOGLIK_PATH"] = path


info = card()
PEAK = dgemm_peak()
print(json.dumps(dict(config="card", dgemm_tflops=PEAK, **info)), flush=True)
rng = np.random.default_rng(64)
d, P_ = 10, 12
which = [int(v) for v in sys.argv[1:]] or [256, 512, 1024, 2048]
for N in which:
    X = rng.uniform(-5, 5, size=(N, d))
    U = (X + 5) / 10
    y = -sum(branin(15 * U[:, 2 * i] - 5, 15 * U[:, 2 * i + 1]) for i in range(5)) / 100.0
    gp = GP(kernel=float(np.var(y)) * kernels.ExpSquaredKernel(np.ones(d), ndim=d), fit_mean=True,
            mean=float(np.median(y)), white_noise=-12.0)
    gp.compute(X, y=y)
    F_ll = N ** 3 / 3.0 + 2.0 * N * N + (3 * d + 1) * N * N / 2.0
    F_llg = F_ll + 2.0 * N ** 3 / 3.0 + P_ * N * N
    for R in (1, 8, 64):
        P = np.column_stack([np.full(R, np.median(y)), rng.standard_normal((R, P_ - 1))])
        row = dict(config="cfg4-loglik-grad", N=N, d=d, R=R, **info)
        setenv(None)
        t_grad = timed(lambda: gp.log_likelihood_batch(P, y, return_grad=True))
        assert path_of(gp) == 4
        ll, g = gp.log_likelihood_batch(P, y, return_grad=True)
        setenv("group")
        t_val = timed(lambda: gp.log_likelihood_batch(P, y))
        assert path_of(gp) == 2
        t_fb = timed(lambda: gp.log_likelihood_batch(P, y, return_grad=True), min_s=0.5, max_reps=5)
        ll_f, g_f = gp.log_likelihood_batch(P, y, return_grad=True)
        setenv(None)
        fin = np.isfinite(ll)
        row.update(ms_grad_path4=t_grad * 1e3, ms_value_path2=t_val * 1e3, ms_fallback_per_vector=t_fb * 1e3,
                   speedup_over_fallback=t_fb / t_grad, grad_over_value=t_grad / t_val,
                   tflops_llg=R * F_llg / t_grad * 1e-12, frac_of_dgemm_llg=R * F_llg / t_grad * 1e-12 / PEAK,
                   tflops_ll_value=R * F_ll / t_val * 1e-12, frac_of_dgemm_ll_value=R * F_ll / t_val * 1e-12 / PEAK,
                   finite=int(fin.sum()),
                   max_rel_ll_diff_vs_fallback=float(np.max(np.abs(ll[fin] - ll_f[fin]) / np.abs(ll_f[fin]))) if fin.any() else None,
                   max_grad_diff_vs_fallback_over_max=float(np.max(np.abs(g[fin] - g_f[fin])) / np.max(np.abs(g_f[fin]))) if fin.any() else None,
                   note="wall time of one gp.log_likelihood_batch call (staging copies, launch, synchronise included)")
        print(json.dumps(row), flush=True)
    if N <= 1024:
        for route, forced in (("path4", None), ("fallback", "group")):
            setenv(forced)
            keep = gp.get_parameter_vector()
            np.random.seed(64)
            t0 = time.perf_counter()
            gpUtils.optimizeGP(gp, X, y, nGPRestarts=64, method="l-bfgs-b", options={"maxiter": 20})
            dt = time.perf_counter() - t0
            setenv(None)
            print(json.dumps(dict(config="cfg4-optGP-lbfgsb", N=N, restarts=64, route=route, seconds=dt,
                                  stats=gpUtils.optimizeGP.last_stats, best_ll=float(gp.log_likelihood(y)),
                                  note="L-BFGS-B capped at maxiter=20 per restart", **info)), flush=True)
            gp.set_parameter_vector(keep); gp.recompute()
