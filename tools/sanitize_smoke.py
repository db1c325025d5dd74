"""Small end-to-end pass over every kernel for compute-sanitizer (memcheck / racecheck / synccheck)."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from approxposterior_b200 import GP, kernels

rng = np.random.default_rng(0)
for N, d, amp in ((70, 2, None), (200, 3, 2.0), (300, 5, None)):
    X = rng.uniform(-5, 5, size=(N, d)); y = np.sin(X).sum(axis=1)
    k = kernels.ExpSquaredKernel(np.full(d, 3.0), ndim=d)
    if amp:
        k = amp * k
    gp = GP(kernel=k, fit_mean=True, mean=0.0, white_noise=-12.0)
    gp.compute(X, y=y)
    q = rng.uniform(-5, 5, size=(700, d))
    gp.predict(y, q, return_cov=False, return_var=True)
    gp.predict(y, q, return_cov=False, return_var=False)
    gp.predict_utility(y, q, "jones", bounds=[(-5, 5)] * d)
    gp.predict(y, q[:1], return_cov=False, return_var=True)          # few-query kernel (S CTAs per query, arrival counter)
    gp.predict_utility(y, q[:7], "bape", bounds=[(-5, 5)] * d)
    P = np.vstack([gp.get_parameter_vector() + 0.1 * i for i in range(5)])
    gp.log_likelihood_batch(P, y)
    if N > 224:                                                       # fused cluster log-likelihood at every cluster size
        for C in ("1", "2", "4"):
            os.environ["APGP_CHOL_CLUSTER"] = C
            gp.log_likelihood_batch(P, y)
        del os.environ["APGP_CHOL_CLUSTER"]
    gp.log_likelihood_batch(P, y, return_grad=(N <= 224))
    gp.grad_log_likelihood(y)
    gp.append_point(rng.uniform(-5, 5, size=d), 0.3)
    y2 = np.concatenate([y, [0.3]])
    gp.predict(y2, q[:100], return_cov=False, return_var=True)
    p0 = rng.uniform(-5, 5, size=(2 * 4 * d, d))
    gp.run_ensembles(y2, p0, 20, [(-5, 5)] * d, nens=2, seed=3)
    # device-resident optimisers (one CTA per start) and their evaluate-only entry
    starts = rng.uniform(-4, 4, size=(3, d))
    for kind in ("bape", "negmean"):
        gp.minimize_utility(y2, starts, kind, bounds=[(-5, 5)] * d, evaluate_only=True)
        gp.minimize_utility(y2, starts, kind, bounds=[(-5, 5)] * d, options={"adaptive": True, "maxfev": 40})
        gp.minimize_utility(y2, starts, kind, bounds=[(-5, 5)] * d, method="powell", options={"maxfev": 40})
    if gp.can_minimize_nll():
        gp.minimize_nll(P[:3], y2, evaluate_only=True)
        gp.minimize_nll(P[:3], y2, method="powell", options={"maxfev": 25})
        gp.minimize_nll(P[:3], y2, method="nelder-mead", options={"maxfev": 25})
    os.environ["APGP_LOGLIK_PATH"] = "tiled"
    gp.log_likelihood_batch(P, y2)
    del os.environ["APGP_LOGLIK_PATH"]
# grouped variance kernel (G CTAs per query tile, cooperative launch): N >= 1024 selects it automatically
N, d = 1100, 3
X = rng.uniform(-5, 5, size=(N, d)); y = np.sin(X).sum(axis=1)
gp = GP(kernel=kernels.ExpSquaredKernel(np.full(d, 3.0), ndim=d), fit_mean=True, mean=0.0, white_noise=-12.0)
gp.compute(X, y=y)
q = rng.uniform(-5, 5, size=(3000, d))
gp.predict_utility(y, q, "bape", bounds=[(-5, 5)] * d)
gp.set_group(4)
gp.predict_utility(y, q[:300], "agp", bounds=[(-5, 5)] * d)
# latency regime of the grouped kernel (few tiles -> many CTAs per tile) and the sampler as a thread-block cluster
gp.set_group(-1)
gp.predict_utility(y, q[:5], "bape", bounds=[(-5, 5)] * d)
os.environ["APGP_SAMPLER_CLUSTER"] = "4"
p0 = rng.uniform(-5, 5, size=(64, d))
gp.run_ensembles(y, p0, 30, [(-5, 5)] * d, nens=1, seed=3, thin=2)
del os.environ["APGP_SAMPLER_CLUSTER"]
print("sanitize_smoke ok")
