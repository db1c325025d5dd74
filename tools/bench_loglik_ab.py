"""A/B timing of two builds of libapgp.so on the batched log-likelihood and the device optimisers of the hyper-parameters,
alternating the builds round by round (each round is a fresh process with APGP_LIB set).  Per case it prints the median
call time of each build and whether their outputs were bit-identical.

    python tools/bench_loglik_ab.py --lib-a path/to/parent/libapgp.so --lib-b approxposterior_b200/libapgp.so [--rounds 3]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOGLIK = [(N, R) for N in (50, 100, 200, 230, 512, 1024) for R in (1, 8, 64)]
MINIMIZE = [(70, "powell"), (70, "nelder-mead"), (200, "powell"), (300, "powell"), (300, "nelder-mead")]


def _problem(N, d=3, seed=0):
    import numpy as np
    from approxposterior_b200 import GP, kernels
    rng = np.random.default_rng(seed)
    X = rng.uniform(-5, 5, size=(N, d))
    y = np.sin(X).sum(axis=1) + 0.1 * rng.standard_normal(N)
    gp = GP(kernel=2.0 * kernels.ExpSquaredKernel(np.full(d, 4.0), ndim=d), fit_mean=True, mean=float(np.median(y)),
            white_noise=-12.0)
    gp._x, gp._y = X, y
    gp._upload_training()
    return gp, y


def _timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)            # every call ends in a device synchronise (results on the host)
    ts.sort()
    return ts[len(ts) // 2], out


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(a.tobytes())
    return h.hexdigest()[:16]


def worker():
    import ctypes
    import numpy as np
    sys.path.insert(0, ROOT)
    from approxposterior_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in [n for n in _lib._SIGNATURES if not hasattr(lib, n)]:      # a build older than some debug entry point
        del _lib._SIGNATURES[name]
    res = {}
    for N, R in LOGLIK:
        gp, y = _problem(N)
        P = gp.get_parameter_vector()[None, :] + 0.5 * np.random.default_rng(R).standard_normal((R, len(gp)))
        t, ll = _timed(lambda: gp.log_likelihood_batch(P, y), 20)
        res["loglik N=%d R=%d" % (N, R)] = (t, _digest(ll))
    for N, method in MINIMIZE:
        gp, y = _problem(N, seed=1)
        P = gp.get_parameter_vector()[None, :] + 0.5 * np.random.default_rng(2).standard_normal((64, len(gp)))
        t, (p, f, nfev) = _timed(lambda: gp.minimize_nll(P, y, method=method, options={"maxfev": 300}), 3)
        res["minimize_nll N=%d %s R=64" % (N, method)] = (t, _digest(p, f, nfev))
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib-a", required=True)
    ap.add_argument("--lib-b", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--worker", action="store_true")
    a = ap.parse_args()
    if a.worker:
        worker()
        return
    runs = {"a": [], "b": []}
    for _ in range(a.rounds):
        for key, lib in (("a", a.lib_a), ("b", a.lib_b)):
            env = dict(os.environ, APGP_LIB=os.path.abspath(lib))
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", "--lib-a", a.lib_a, "--lib-b",
                                  a.lib_b], env=env, cwd=ROOT, capture_output=True, text=True, check=True).stdout
            runs[key].append(json.loads(out.strip().split("\n")[-1]))
    for case in runs["a"][0]:
        ta = sorted(r[case][0] for r in runs["a"])
        tb = sorted(r[case][0] for r in runs["b"])
        same = len({r[case][1] for r in runs["a"] + runs["b"]}) == 1
        print(json.dumps({"case": case, "a_ms": [round(1e3 * t, 4) for t in ta], "b_ms": [round(1e3 * t, 4) for t in tb],
                          "b_over_a": round(tb[len(tb) // 2] / ta[len(ta) // 2], 4), "identical": same}))


if __name__ == "__main__":
    main()
