"""Device-resident optimisers (csrc/optimize.cu, apgp_minimize_utility / apgp_minimize_nll) against

  * the host restatements of SciPy's Nelder-Mead / Powell (approxposterior_b200/_optimizers.py, themselves
    checked point-for-point against scipy.optimize.minimize in tests/test_host_logic.py) driven by the very
    objective function the device minimises (evaluate_only=True): same iterates => same optimum, bit for bit;
  * the batched predict / log-likelihood kernels and the CPU oracle for the objective values themselves;
  * the reference's own known answers through gpUtils.optimizeGP / utility.minimizeObjective.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _gp(N=60, d=2, seed=3, amp=None, fit_y=True):
    from approxposterior_b200 import GP, kernels
    rng = np.random.default_rng(seed)
    X = rng.uniform(-5, 5, size=(N, d))
    y = -0.5 * np.sum((X / 2.0) ** 2, axis=1) + 0.1 * rng.standard_normal(N) if fit_y else rng.standard_normal(N)
    k = kernels.ExpSquaredKernel(np.full(d, 4.0), ndim=d)
    if amp is not None:
        k = amp * k
    gp = GP(kernel=k, fit_mean=True, mean=float(np.median(y)), white_noise=-12.0)
    gp.compute(X, y=y)
    return gp, X, y


def _run_host(gen_factory, starts, batch_fn):
    from approxposterior_b200 import _optimizers as opt
    out, rounds, evals = opt.run_generators([gen_factory(t0) for t0 in starts], batch_fn)
    return np.array([o[0] for o in out]), np.array([o[1] for o in out]), evals


@pytest.mark.parametrize("kind", ["bape", "agp", "jones", "negmean"])
def test_utility_point_objective_matches_batched_predict(kind):
    """evaluate_only: the single-point objective of the device optimiser == fused predict kernel == oracle formula."""
    gp, X, y = _gp(N=90, d=3, seed=5)
    rng = np.random.default_rng(0)
    T = rng.uniform(-5.5, 5.5, size=(200, 3))
    bounds = [(-5.0, 5.0)] * 3
    _, f, _ = gp.minimize_utility(y, T, kind, bounds=bounds, evaluate_only=True)
    inside = np.all((T >= -5) & (T <= 5), axis=1)
    assert np.all(np.isposinf(f[~inside]))
    if kind == "negmean":
        ref = -np.asarray(gp.predict(y, T[inside], return_cov=False))
        assert np.allclose(f[inside], ref, rtol=1e-10, atol=1e-10 * np.max(np.abs(y)))
    else:
        mu, var, u = gp.predict_utility(y, T[inside], kind, bounds=bounds)
        fin = np.isfinite(u)
        # the utilities amplify the rounding of var = A - sum W^2 (an O(A) cancellation): compare like the variance test
        tol = 1e-9 * (1.0 + np.abs(u[fin])) / np.minimum(1.0, np.abs(var[fin]))
        assert np.all(np.abs(f[inside][fin] - u[fin]) <= tol)
        assert np.array_equal(np.isnan(f[inside]), np.isnan(u))


@pytest.mark.parametrize("amp", [None, 7.5])
def test_nll_point_objective_matches_loglik_batch_and_oracle(amp):
    from oracle import GPOracle
    gp, X, y = _gp(N=70, d=2, seed=11, amp=amp)
    rng = np.random.default_rng(1)
    P = gp.get_parameter_vector()[None, :] + 0.5 * rng.standard_normal((16, len(gp)))
    P[3, 1] = 25.0                      # rejected by defaultHyperPrior
    P[5, -1] = np.nan
    _, f, _ = gp.minimize_nll(P, y, evaluate_only=True)
    assert np.isposinf(f[3]) and np.isposinf(f[5])
    ll = gp.log_likelihood_batch(P, y)
    ok = np.ones(16, bool); ok[[3, 5]] = False
    assert np.array_equal(f[ok], -ll[ok])            # one evaluator (loglik.cuh): the same bits
    for r in (0, 7):
        p = P[r]
        a = 2 * np.exp(p[1]) if amp is not None else None
        orc = GPOracle(2, np.exp(p[-2:]), mean=p[0], white_noise=-12.0, amp=a)
        orc.compute(X)
        assert abs(f[r] + orc.log_likelihood(y)) <= 1e-9 * abs(f[r])


@pytest.mark.parametrize("method,options", [
    ("nelder-mead", {"adaptive": True}),
    ("nelder-mead", None),
    ("powell", None),
    ("nelder-mead", {"adaptive": True, "maxfev": 37}),
    ("powell", {"maxfev": 23}),
    ("powell", {"xtol": 1e-6, "ftol": 1e-8, "maxiter": 3}),
])
@pytest.mark.parametrize("kind", ["bape", "negmean"])
def test_device_minimize_utility_is_the_scipy_iteration(method, options, kind):
    """One CTA per start on the device visits exactly the points the host restatement of SciPy visits."""
    from approxposterior_b200 import _optimizers as opt
    gp, X, y = _gp(N=60, d=2, seed=3)
    bounds = [(-5.0, 5.0)] * 2
    rng = np.random.default_rng(7)
    starts = rng.uniform(-5, 5, size=(6, 2))
    starts[4] = [4.99, -4.99]            # hugs the prior edge: +inf objective values, ties in the simplex
    starts[5] = [0.0, 1.0]               # a zero coordinate (SciPy's zdelt branch)
    xd, fd, nd = gp.minimize_utility(y, starts, kind, bounds=bounds, method=method, options=options)
    o = dict(options or {})
    if method == "nelder-mead":
        make = lambda t0: opt.nelder_mead_gen(t0, _stable=True, **o)
    else:
        make = lambda t0: opt.powell_gen(t0, **o)
    xh, fh, evals = _run_host(make, starts, lambda P: gp.minimize_utility(y, np.array(P), kind, bounds=bounds,
                                                                        evaluate_only=True)[1])
    assert np.array_equal(xd, xh), (xd, xh)
    assert np.array_equal(fd, fh)
    assert int(np.sum(nd)) == evals


@pytest.mark.parametrize("method,options", [("powell", None), ("nelder-mead", None), ("powell", {"maxfev": 60})])
@pytest.mark.parametrize("amp", [None, 3.0])
def test_device_minimize_nll_is_the_scipy_iteration(method, options, amp):
    from approxposterior_b200 import _optimizers as opt
    gp, X, y = _gp(N=50, d=2, seed=21, amp=amp)
    np.random.seed(5)
    P = len(gp)
    x0s = np.array([[np.median(y)] + [np.random.randn() for _ in range(P - 1)] for _ in range(4)])
    pd_, fd, nd = gp.minimize_nll(x0s, y, method=method, options=options)
    o = dict(options or {})
    make = (lambda t0: opt.powell_gen(t0, **o)) if method == "powell" else (lambda t0: opt.nelder_mead_gen(t0, _stable=True, **o))
    ph, fh, evals = _run_host(make, x0s, lambda Q: gp.minimize_nll(np.array(Q), y, evaluate_only=True)[1])
    assert np.array_equal(pd_, ph), (pd_, ph)
    assert np.array_equal(fd, fh)
    assert int(np.sum(nd)) == evals
    # and the GP itself was left alone
    assert gp.computed


def test_device_and_lockstep_engines_agree_on_optimizeGP():
    """Same starts, same algorithm; objective values differ in the last bits between the two kernels, so the
    optima agree to optimiser tolerance rather than bit for bit."""
    from approxposterior_b200 import gpUtils, likelihood as lh
    res = {}
    for engine in ("device", "lockstep"):
        np.random.seed(57)
        theta = np.array(lh.rosenbrockSample(50))
        y = np.array([lh.rosenbrockLnlike(t) + lh.rosenbrockLnprior(t) for t in theta])
        gp = gpUtils.defaultGP(theta, y, fitAmp=False)
        gp = gpUtils.optimizeGP(gp, theta, y, nGPRestarts=5, method="powell", engine=engine)
        res[engine] = (gp.get_parameter_vector(), gp.log_likelihood(y), dict(gpUtils.optimizeGP.last_stats))
    assert res["device"][2]["scheduler"] == "device" and res["device"][2]["batches"] == 1
    assert res["lockstep"][2]["scheduler"] == "generators"
    assert np.allclose(res["device"][0], res["lockstep"][0], rtol=1e-3, atol=1e-3)
    assert abs(res["device"][1] - res["lockstep"][1]) <= 1e-6 * abs(res["lockstep"][1])


def test_device_minimize_objective_retries_and_matches_lockstep():
    from approxposterior_b200 import utility as ut, likelihood as lh
    gp, X, y = _gp(N=80, d=2, seed=9)
    prior = lh.BoxPrior([(-5, 5), (-5, 5)])
    out = {}
    for engine in ("device", "lockstep"):
        np.random.seed(3)
        out[engine] = ut.minimizeObjective(ut.BAPEUtility, y, gp, sampleFn=prior.sample, priorFn=prior, nRestarts=5,
                                           args=(y, gp, prior), engine=engine)
        st = dict(ut.minimizeObjective.last_stats)
        assert st["scheduler"] == ("device" if engine == "device" else "generators")
    assert np.allclose(out["device"][0], out["lockstep"][0], atol=5e-4)
    assert abs(out["device"][1] - out["lockstep"][1]) <= 1e-6 * (1 + abs(out["lockstep"][1]))


def test_device_optimizer_large_training_set_reads_linv_from_global():
    """N = 400: the packed L^-1 (642 KB) no longer fits in shared memory; rows stream from L2 instead."""
    from approxposterior_b200 import _optimizers as opt
    gp, X, y = _gp(N=400, d=3, seed=4)
    bounds = [(-5.0, 5.0)] * 3
    starts = np.random.default_rng(2).uniform(-4, 4, size=(3, 3))
    xd, fd, _ = gp.minimize_utility(y, starts, "agp", bounds=bounds, options={"adaptive": True})
    xh, fh, _ = _run_host(lambda t0: opt.nelder_mead_gen(t0, adaptive=True, _stable=True), starts,
                          lambda P: gp.minimize_utility(y, np.array(P), "agp", bounds=bounds, evaluate_only=True)[1])
    assert np.array_equal(xd, xh) and np.array_equal(fd, fh)
    # N = 400 is beyond the one-CTA shared-memory nll objective: the cluster-per-restart objective takes over
    # (tests/test_gpu_chol_group.py); only training sets beyond 4096 points are refused
    assert gp.can_minimize_nll()
    p, f, nfev = gp.minimize_nll(gp.get_parameter_vector()[None, :], y, options={"maxiter": 1})
    assert np.isfinite(f[0]) and nfev[0] > 3


def test_find_map_on_device():
    """reference tests/test_MAP.py shape: sphere function, MAP of the GP mean near the origin."""
    from approxposterior_b200 import approx, gpUtils, likelihood as lh, utility as ut
    np.random.seed(42)
    bounds = [(-2, 2), (-2, 2)]
    theta = lh.sphereSample(40)
    y = np.array([lh.sphereLnlike(t) for t in theta])
    gp = gpUtils.defaultGP(theta, y, fitAmp=True)
    prior = lh.BoxPrior(bounds)
    ap = approx.ApproxPosterior(theta=theta, y=y, gp=gp, lnprior=prior, lnlike=lh.sphereLnlike,
                                priorSample=lh.sphereSample, bounds=bounds, algorithm="jones")
    ap.optGP(seed=42, method="powell", nGPRestarts=3)
    MAP, val = ap.findMAP(nRestarts=8)
    assert ut.minimizeObjective.last_stats["scheduler"] == "device"
    assert np.allclose(MAP, [0.0, 0.0], atol=5e-2) and abs(val) < 5e-2


@pytest.mark.parametrize("method,options", [("nelder-mead", {"adaptive": True}), ("powell", None),
                                            ("nelder-mead", {"maxfev": 1}), ("powell", {"maxfev": 2})])
def test_device_optimisers_one_dimensional(method, options):
    """ndim = 1 (the reference's 1-D Bayesian-optimisation example): simplex of two points, one Powell direction."""
    from approxposterior_b200 import _optimizers as opt
    gp, X, y = _gp(N=30, d=1, seed=8)
    bounds = [(-5.0, 5.0)]
    starts = np.array([[-3.0], [0.0], [4.5], [5.5]])          # the last start is outside the prior: +inf everywhere
    xd, fd, nd = gp.minimize_utility(y, starts, "jones", bounds=bounds, method=method, options=options)
    o = dict(options or {})
    make = (lambda t0: opt.nelder_mead_gen(t0, _stable=True, **o)) if method == "nelder-mead" else (lambda t0: opt.powell_gen(t0, **o))
    xh, fh, evals = _run_host(make, starts, lambda P: gp.minimize_utility(y, np.array(P), "jones", bounds=bounds,
                                                                        evaluate_only=True)[1])
    assert np.array_equal(xd, xh, equal_nan=True) and np.array_equal(fd, fh, equal_nan=True)
    assert int(np.sum(nd)) == evals
    P0 = np.array([[np.median(y), 0.3], [np.median(y), -1.0]])
    pd_, fnd, nn = gp.minimize_nll(P0, y, method=method, options=options)
    ph, fnh, ev2 = _run_host(make, P0, lambda Q: gp.minimize_nll(np.array(Q), y, evaluate_only=True)[1])
    assert np.array_equal(pd_, ph, equal_nan=True) and np.array_equal(fnd, fnh, equal_nan=True) and int(np.sum(nn)) == ev2
