"""GPU parity: CUDA path (through the C-ABI) vs the CPU oracle on identical inputs.

Tolerances (fp64): north_star asks for 1e-9 relative on mean, variance, utility and
log-likelihood.  The variance is a difference of O(A) terms, so its parity is stated as
|dvar| <= 1e-9 * A + 1e-9 * |var| (SURVEY 7 "variance cancellation"); everything else is rtol 1e-9
with an atol tied to the problem scale.
"""
import numpy as np
import pytest

from conftest import extended_truth, rosenbrock_training, synthetic_gp_problem, utility_error_bound

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def make_pair(X, y, logM, amp=None, mean=None, wn=-12.0):
    from approxposterior_b200 import GP, kernels
    from oracle import GPOracle
    d = X.shape[1]
    mean = float(np.median(y)) if mean is None else mean
    k = kernels.ExpSquaredKernel(metric=np.exp(logM), ndim=d)
    if amp is not None:
        k = amp * k
    gp = GP(kernel=k, fit_mean=True, mean=mean, white_noise=wn, fit_white_noise=False)
    gp.compute(X, y=y)
    orc = GPOracle(d, np.exp(logM), amp=amp, mean=mean, white_noise=wn)
    orc.compute(X)
    return gp, orc


def check_mean(mu, mu_o, orc, y, Xq):
    """Mean parity at north_star's 1e-9 (relative, with 1e-9 of the data scale as the absolute floor).  Where an entry
    misses that strict bound -- cond(K) reaches 1e6-1e8 on the d = 1, 2 problems and BOTH fp64 implementations carry
    forward errors of order cond(K) eps in alpha -- the disagreement is arbitrated against extended-precision truth
    (conftest.extended_truth): the engine may be at most 4x as far from the truth as the LAPACK oracle is.
    Measured max errors vs truth are in profiles/r02_parity_errors.txt (current library and the pre-9d0af3d diagonal
    kernel, next to the oracle's own)."""
    scale = max(np.max(np.abs(y)), 1.0)
    strict = np.abs(mu - mu_o) <= RTOL * np.abs(mu_o) + RTOL * scale
    if np.all(strict):
        return 0.0
    mu_t, _ = extended_truth(orc._x, y, orc.log_M, Xq, amp=(orc.amplitude if orc.fit_amp else None), mean=orc.mean,
                             wn=orc.white_noise)
    err_g, err_o = np.max(np.abs(mu - mu_t)), np.max(np.abs(mu_o - mu_t))
    assert err_g <= 4.0 * err_o, (err_g, err_o, int(np.sum(~strict)))
    return float(np.max(np.abs(mu - mu_o)))        # conditioning-limited disagreement both implementations share


def check_predict(gp, orc, y, Xq, amp_scale):
    mu, var = gp.predict(y, Xq, return_cov=False, return_var=True)
    mu_o, var_o = orc.predict(y, Xq, return_var=True)
    check_mean(mu, mu_o, orc, y, Xq)
    assert np.all(np.abs(var - var_o) <= 1e-9 * amp_scale + 1e-9 * np.abs(var_o))
    mu1 = gp.predict(y, Xq, return_cov=False, return_var=False)
    check_mean(mu1, mu_o, orc, y, Xq)
    return mu, var


@pytest.mark.parametrize("N,d", [(20, 2), (64, 1), (100, 3), (256, 2), (300, 5), (700, 5), (2100, 20)])
def test_factor_and_predict_vs_oracle(N, d):
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + d)
    gp, orc = make_pair(X, y, logM)
    L = gp._chol()
    np.testing.assert_allclose(L, orc._L, rtol=1e-9, atol=1e-10 * np.max(np.abs(orc._L)))
    Linv = gp._linv()
    assert np.max(np.abs(Linv @ orc._L - np.eye(N))) < 1e-9
    alpha = gp._alpha()
    alpha_o = orc._compute_alpha(y)
    np.testing.assert_allclose(alpha, alpha_o, rtol=1e-8, atol=1e-9 * np.max(np.abs(alpha_o)))
    assert abs(gp.log_likelihood(y) - orc.log_likelihood(y)) <= 1e-9 * abs(orc.log_likelihood(y))
    assert abs(gp.log_determinant - orc.log_determinant) <= 1e-9 * max(1.0, abs(orc.log_determinant))
    rng = np.random.default_rng(1)
    Xq = rng.uniform(-5, 5, size=(777, d))
    Xq[:5] = X[:5]                      # on top of training points: var ~ 0 (cancellation case)
    check_predict(gp, orc, y, Xq, 1.0)


@pytest.mark.parametrize("N,d", [(256, 2), (256, 20), (8192, 2), (8192, 20)])
def test_cfg5_corners_end_to_end_utility(N, d):
    """BASELINE configs[4] corners: mean / variance / utility of the fused kernel against the oracle END TO END (oracle
    utilities from the oracle's own mu, var) at the bound the 1e-9 (mu, var) parity implies
    (conftest.utility_error_bound); oracle on a 400-query subsample of a 50 000-query call."""
    from oracle import UTILITY_BY_NAME
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=5)
    gp, orc = make_pair(X, y, logM)
    rng = np.random.default_rng(N + d)
    Xq = rng.uniform(-5, 5, size=(50000, d))
    idx = rng.choice(len(Xq), size=400, replace=False)
    bounds = [(-5.0, 5.0)] * d
    mu_o, var_o = orc.predict(y, Xq[idx], return_var=True)
    scale = max(1.0, float(np.max(np.abs(y))))
    for kind in ("agp", "bape", "jones"):
        mu, var, u = gp.predict_utility(y, Xq, kind, bounds=bounds)
        slack = check_mean(mu[idx], mu_o, orc, y, Xq[idx])
        assert np.all(np.abs(var[idx] - var_o) <= 1e-9 + 1e-9 * np.abs(var_o))
        fn = UTILITY_BY_NAME[kind]
        ref = fn(mu_o, var_o, float(np.max(y))) if kind == "jones" else fn(mu_o, var_o)
        bound, resolved = utility_error_bound(kind, mu_o, var_o, 1.0, scale, ybest=float(np.max(y)))
        good = np.isfinite(ref) & resolved
        assert np.sum(good) > 0.5 * len(idx)
        tol = bound[good] + 2.0 * slack + 1e-9 * np.abs(ref[good])
        assert np.all(np.abs(u[idx][good] - ref[good]) <= tol), (kind, np.max(np.abs(u[idx][good] - ref[good]) / tol))


@pytest.mark.parametrize("fitAmp", [False, True])
def test_reference_kat_utilities(fitAmp):
    """Reference KATs tests/test_GPUtil.py:50,56,62,101,107,113 reproduced by the CUDA path."""
    from approxposterior_b200 import gpUtils
    theta, y = rosenbrock_training(20)
    np.random.seed(57)
    rosenbrock_training(20)            # replays the RNG consumption of the reference test
    gp = gpUtils.defaultGP(theta, y, fitAmp=fitAmp)
    t = np.array([[-2.3573, 4.673]])
    bounds = [(-5, 5), (-5, 5)]
    gold = (31.92055252, -114623.57332731, -77.37826545) if fitAmp else (37.41585067, 76.15271103, 0.0)
    for kind, g in zip(("agp", "bape", "jones"), gold):
        _, _, u = gp.predict_utility(y, t, kind, bounds=bounds)
        assert np.allclose(u[0], g, rtol=1.0e-4), (kind, u[0], g)


@pytest.mark.parametrize("amp", [None, 57000.0])
def test_utilities_vs_oracle(amp):
    from oracle import agp_utility, bape_utility, jones_utility
    theta, y = rosenbrock_training(50)
    logM = np.array([-1.0552327, -1.16092752])
    gp, orc = make_pair(theta, y, logM, amp=amp)
    rng = np.random.default_rng(3)
    Xq = rng.uniform(-6, 6, size=(1000, 2))     # some outside the +-5 box
    bounds = [(-5, 5), (-5, 5)]
    ok = np.all(np.abs(Xq) <= 5, axis=1)
    mu_o, var_o = orc.predict(y, Xq, return_var=True)
    A = amp if amp is not None else 1.0
    for kind, fn in (("agp", agp_utility), ("bape", bape_utility)):
        mu, var, u = gp.predict_utility(y, Xq, kind, bounds=bounds)
        # compare the epilogue on identical (mu,var): isolates the utility formula
        ref_same = fn(mu, var, ok)
        fin = np.isfinite(ref_same)
        assert np.array_equal(np.isinf(u) & (u > 0), ~ok)
        np.testing.assert_allclose(u[fin], ref_same[fin], rtol=1e-9, atol=1e-9)
        assert np.array_equal(np.isnan(u), np.isnan(ref_same))
        assert np.all(np.abs(var - var_o) <= 1e-9 * A + 1e-9 * np.abs(var_o))
    mu, var, u = gp.predict_utility(y, Xq, "jones", bounds=bounds)
    ref_same = jones_utility(mu, var, y.max(), 0.01, ok)
    fin = np.isfinite(ref_same)
    np.testing.assert_allclose(u[fin], ref_same[fin], rtol=1e-9, atol=1e-12 * A)


@pytest.mark.parametrize("fit_amp", [False, True])
def test_loglik_batch_and_grad(fit_amp):
    N, d = 90, 2
    theta, y = rosenbrock_training(N)
    amp = float(np.var(y)) if fit_amp else None
    gp, orc = make_pair(theta, y, np.zeros(d), amp=amp)
    rng = np.random.default_rng(11)
    R = 37
    P = np.column_stack([np.full(R, np.median(y))] + [rng.standard_normal(R) for _ in range(len(gp) - 1)])
    P[3, -1] = 25.0           # still factorises (prior gating is the host's job)
    P[5, 1] = np.nan          # non-finite hyper-parameter -> -inf
    ll = gp.log_likelihood_batch(P, y)
    for r in range(R):
        if not np.all(np.isfinite(P[r])):
            assert ll[r] == -np.inf
            continue
        orc.set_parameter_vector(P[r])
        ref = orc.log_likelihood(y, quiet=True)
        if np.isfinite(ref):
            assert abs(ll[r] - ref) <= 1e-9 * abs(ref), (r, ll[r], ref)
        else:
            assert ll[r] == -np.inf
    # single-GP path and gradient
    p = P[0]
    gp.set_parameter_vector(p)
    orc.set_parameter_vector(p)
    assert abs(gp.log_likelihood(y, quiet=True) - orc.log_likelihood(y, quiet=True)) <= 1e-9 * abs(orc.log_likelihood(y))
    g = gp.grad_log_likelihood(y, quiet=True)
    g_o = orc.grad_log_likelihood(y, quiet=True)
    np.testing.assert_allclose(g, g_o, rtol=1e-8, atol=1e-8 * np.max(np.abs(g_o)))


@pytest.mark.parametrize("N,fit_amp", [(40, True), (150, False), (224, True), (300, True)])
def test_loglik_batch_gradients(N, fit_amp):
    """Batched gradients: fused shared-memory kernel up to N ~ 224, per-vector path beyond; both vs the oracle."""
    theta, y = rosenbrock_training(N)
    gp, orc = make_pair(theta, y, np.zeros(2), amp=float(np.var(y)) if fit_amp else None)
    rng = np.random.default_rng(N)
    R = 9
    P = np.column_stack([np.full(R, np.median(y))] + [0.7 * rng.standard_normal(R) for _ in range(len(gp) - 1)])
    P[4, -1] = np.nan
    keep = gp.get_parameter_vector().copy()
    ll, g = gp.log_likelihood_batch(P, y, return_grad=True)
    assert np.array_equal(gp.get_parameter_vector(), keep)
    for r in range(R):
        if not np.all(np.isfinite(P[r])):
            assert ll[r] == -np.inf and np.all(g[r] == 0)
            continue
        orc.set_parameter_vector(P[r])
        ref_ll = orc.log_likelihood(y, quiet=True)
        ref_g = orc.grad_log_likelihood(y, quiet=True)
        assert abs(ll[r] - ref_ll) <= 1e-9 * abs(ref_ll)
        np.testing.assert_allclose(g[r], ref_g, rtol=1e-7, atol=1e-8 * np.max(np.abs(ref_g)))


def test_loglik_batch_fused_and_tiled_paths_agree(monkeypatch):
    """N small enough for the one-restart-per-CTA shared-memory kernel: it must agree with the tiled
    multi-launch path (forced with APGP_LOGLIK_PATH=tiled) and with the oracle."""
    theta, y = rosenbrock_training(150)
    gp, orc = make_pair(theta, y, np.zeros(2), amp=float(np.var(y)))
    rng = np.random.default_rng(5)
    P = np.column_stack([np.full(20, np.median(y)), rng.standard_normal((20, 3))])
    ll_small = gp.log_likelihood_batch(P, y)
    monkeypatch.setenv("APGP_LOGLIK_PATH", "tiled")
    ll_tiled = gp.log_likelihood_batch(P, y)
    np.testing.assert_allclose(ll_small, ll_tiled, rtol=1e-10)
    for r in range(0, 20, 5):
        orc.set_parameter_vector(P[r])
        assert abs(ll_small[r] - orc.log_likelihood(y, quiet=True)) <= 1e-9 * abs(ll_small[r])


def test_not_positive_definite_is_reported():
    from approxposterior_b200 import GP, kernels
    X = np.array([[0.0, 0.0], [0.0, 0.0], [1.0, 1.0]])      # duplicate point, no noise to speak of
    y = np.array([1.0, 2.0, 3.0])
    gp = GP(kernel=kernels.ExpSquaredKernel([1.0, 1.0], ndim=2), fit_mean=True, mean=0.0, white_noise=-80.0)
    with pytest.raises(np.linalg.LinAlgError):
        gp.compute(X, y=y)
    assert not gp.computed
    assert gp.log_likelihood(y, quiet=True) == -np.inf
    assert np.all(gp.grad_log_likelihood(y, quiet=True) == 0.0)


def test_sampler_replay_matches_oracle():
    from oracle import stretch_move_oracle
    from oracle.sampler_oracle import gpll_batch
    theta, y = rosenbrock_training(50)
    logM = np.array([0.5, 1.2])
    gp, orc = make_pair(theta, y, logM)
    lo, hi = np.array([-5.0, -5.0]), np.array([5.0, 5.0])
    nw, nsteps = 20, 200
    rng = np.random.RandomState(42)
    p0 = rng.uniform(-5, 5, size=(nw, 2))
    ref = stretch_move_oracle(lambda q: gpll_batch(orc, y, q, lo, hi), p0, nsteps, rng=rng, record=True)
    replay = {k: ref[k][None] for k in ("inds", "zz", "rint", "logu")}
    out = gp.run_ensembles(y, p0, nsteps, bounds=list(zip(lo, hi)), nens=1, replay=replay)
    np.testing.assert_allclose(out["chain"], ref["chain"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(out["log_prob"], ref["log_prob"], rtol=1e-9, atol=1e-9)
    assert np.array_equal(out["naccepted"], ref["naccepted"])
    assert np.array_equal(np.isnan(out["blobs"]), np.isnan(ref["blobs"]))


def _thinned(chain, discard, c=3.0):
    """Samples thinned by c x the integrated autocorrelation time (emcee's estimator), flattened: close enough to
    independent for a two-sample Kolmogorov-Smirnov test to hold its nominal level."""
    from approxposterior_b200.sampler import integrated_time
    ch = chain[discard:]
    tau = integrated_time(ch, tol=0, quiet=True)
    step = max(int(np.ceil(c * np.nanmax(tau))), 1)
    return ch[::step].reshape(-1, ch.shape[-1]), tau


def _assert_same_posterior(a, b, alpha=0.01):
    """Two-sample KS at level alpha on every marginal (Bonferroni over the dimensions) plus first/second moments at
    4 standard errors.  A sampler that over- or under-disperses by 10 % fails this with a few thousand samples."""
    from scipy import stats
    d = a.shape[1]
    for c in range(d):
        res = stats.ks_2samp(a[:, c], b[:, c])
        assert res.pvalue > alpha / d, (c, res.statistic, res.pvalue, len(a), len(b))
        se = np.sqrt(a[:, c].var() / len(a) + b[:, c].var() / len(b))
        assert abs(a[:, c].mean() - b[:, c].mean()) < 4.0 * se, (c, a[:, c].mean(), b[:, c].mean(), se)
        # std ratio: se of a sample std ~ std / sqrt(2 n) for near-Gaussian marginals; heavy tails -> 6 "sigma"
        ratio = a[:, c].std() / b[:, c].std()
        assert abs(ratio - 1.0) < 6.0 * np.sqrt(0.5 / len(a) + 0.5 / len(b)) + 0.02, (c, ratio)


def test_sampler_philox_statistics():
    """Philox-driven device sampler vs the oracle's emcee restatement on the same surrogate: thinned-by-tau samples,
    two-sample KS at alpha = 0.01 per marginal, moments at 4 standard errors (north_star: "posterior moments and KS
    tests agree")."""
    from oracle import stretch_move_oracle
    from oracle.sampler_oracle import gpll_batch
    theta, _ = rosenbrock_training(50)
    # a unimodal target (the Rosenbrock surrogate at these hyper-parameters is multi-modal with tau > 100: two CPU
    # oracle runs with different seeds already disagree at this chain length, which is why the first version of this
    # test could only afford a KS statistic < 0.2)
    y = -0.5 * ((theta[:, 0] - 1.0) ** 2 / 1.5 ** 2 + (theta[:, 1] + 0.5) ** 2 / 0.8 ** 2)
    logM = np.array([0.5, 1.2])
    gp, orc = make_pair(theta, y, logM)
    lo, hi = np.array([-5.0, -5.0]), np.array([5.0, 5.0])
    nw, nsteps, nens = 20, 4000, 16
    rng = np.random.RandomState(7)
    p0 = rng.uniform(-5, 5, size=(nens * nw, 2))
    out = gp.run_ensembles(y, p0, nsteps, bounds=list(zip(lo, hi)), nens=nens, seed=123)
    assert np.all(out["naccepted"] > 0)
    acc = out["naccepted"].mean() / nsteps
    assert 0.1 < acc < 0.9
    yo = y.copy(); yo.setflags(write=False)
    ref = stretch_move_oracle(lambda q: gpll_batch(orc, yo, q, lo, hi), p0[:nw], 30000, rng=rng)
    # each ensemble is its own chain: thin per ensemble with the pooled tau
    b, tau_b = _thinned(ref["chain"], 1000)
    a, tau_a = _thinned(out["chain"], 1000)
    assert np.all(np.abs(tau_a / tau_b - 1.0) < 0.35), (tau_a, tau_b)
    assert len(a) > 2000 and len(b) > 1000
    _assert_same_posterior(a, b)
    assert np.all(a >= -5) and np.all(a <= 5)
    # the test can fail: a sampler whose proposals ignored the (d-1) log z Jacobian over-disperses -- emulate by
    # inflating one marginal by 10 %
    with pytest.raises(AssertionError):
        _assert_same_posterior(a * np.array([1.1, 1.0]), b)


def test_posterior_cfg1_engine_vs_oracle_driver():
    """BASELINE configs[0] (README Rosenbrock BAPE run): the engine's device chain on the FINAL surrogate of a real
    ApproxPosterior.run against emcee's restatement driven on the CPU oracle built from the same training set and
    hyper-parameters (20 walkers, as the README): KS alpha = 0.01 per marginal on thinned samples."""
    from approxposterior_b200 import approx, gpUtils, likelihood as lh
    from oracle import GPOracle, stretch_move_oracle
    from oracle.sampler_oracle import gpll_batch
    np.random.seed(57)
    theta = lh.rosenbrockSample(50)
    y = np.array([lh.rosenbrockLnlike(t) + lh.rosenbrockLnprior(t) for t in theta])
    gp = gpUtils.defaultGP(theta, y, white_noise=-12)
    ap = approx.ApproxPosterior(theta=theta, y=y, gp=gp, lnprior=lh.rosenbrockLnprior, lnlike=lh.rosenbrockLnlike,
                                priorSample=lh.rosenbrockSample, bounds=[(-5, 5), (-5, 5)], algorithm="bape")
    ap.run(m=20, nmax=2, estBurnin=True, nGPRestarts=3, mcmcKwargs={"iterations": int(2.0e4)}, cache=False,
           samplerKwargs={"nwalkers": 20}, verbose=False, thinChains=False, onlyLastMCMC=True)
    assert ap.theta.shape == (90, 2)
    eng = ap.sampler.get_chain()                                   # (20000, 20, 2) from the device (Philox) engine
    p = ap.gp.get_parameter_vector()
    orc = GPOracle(2, np.exp(p[1:]), mean=p[0], white_noise=-12.0)
    orc.compute(ap.theta)
    lo, hi = np.full(2, -5.0), np.full(2, 5.0)
    rs = np.random.RandomState(1)
    yo = ap.y.copy(); yo.setflags(write=False)                     # read-only: the oracle caches alpha for it
    ref = stretch_move_oracle(lambda q: gpll_batch(orc, yo, q, lo, hi), lh.rosenbrockSample(20), 40000, rng=rs)
    a, tau_a = _thinned(eng, 1000)
    b, tau_b = _thinned(ref["chain"], 1000)
    assert np.all(np.abs(tau_a / tau_b - 1.0) < 0.4), (tau_a, tau_b)
    _assert_same_posterior(a, b)


def test_posterior_cfg2_many_ensembles_vs_single_ensemble():
    """BASELINE configs[1] shape (Rosenbrock 2-D surrogate on N = 1024 training points, many independent ensembles of
    32 walkers): the pooled short chains of 512 ensembles against ONE long 32-walker chain on the device and against
    the CPU oracle's emcee restatement -- KS alpha = 0.01 on thinned samples."""
    from oracle import stretch_move_oracle
    from oracle.sampler_oracle import gpll_batch
    theta, y = rosenbrock_training(1024)
    logM = np.array([1.0, 2.5])
    gp, orc = make_pair(theta, y, logM)
    lo, hi = np.full(2, -5.0), np.full(2, 5.0)
    bounds = list(zip(lo, hi))
    rng = np.random.RandomState(11)
    nw, nens = 32, 512
    many = gp.run_ensembles(y, rng.uniform(-5, 5, size=(nens * nw, 2)), 3000, bounds, nens=nens, seed=2, thin=10)
    one = gp.run_ensembles(y, rng.uniform(-5, 5, size=(nw, 2)), 150000, bounds, nens=1, seed=3, thin=5)
    yo = y.copy(); yo.setflags(write=False)                        # read-only: the oracle caches alpha for it
    cpu = stretch_move_oracle(lambda q: gpll_batch(orc, yo, q, lo, hi), rng.uniform(-5, 5, size=(nw, 2)), 25000, rng=rng)
    # many short chains (tau ~ 50-130 steps on this banana-shaped surrogate): burn-in 1500 of 3000 steps (> 10 tau),
    # then every 500th step of every walker
    tau = _thinned(one["chain"], 400)[1] * 5
    assert np.all(tau < 250), tau
    a = many["chain"][150::50].reshape(-1, 2)
    b, _ = _thinned(one["chain"], 400)
    c, _ = _thinned(cpu["chain"], 1000)
    _assert_same_posterior(a, b)
    _assert_same_posterior(b, c)
    _assert_same_posterior(a, c)


@pytest.mark.parametrize("entry", ["apgp_debug_exp_neg", "apgp_debug_exp_neg256"])
def test_kernel_exp_matches_libm(entry):
    """The table+polynomial exp(-s) used inside the kernels (64-entry table + degree 5 in the fused predict kernel,
    256-entry table + degree 4 in the sampler and the mean-only predict): <= 2 ulp against numpy."""
    import ctypes as C
    from approxposterior_b200 import GP, kernels, _lib
    gp = GP(kernel=kernels.ExpSquaredKernel([1.0], ndim=1))
    rng = np.random.default_rng(0)
    s = np.concatenate([rng.uniform(0, 700, 200000), rng.uniform(0, 3, 200000), [0.0, 1e-300, 1e-12, 699.999, 700.0, 750.0, 1e6, np.inf]])
    out = np.empty_like(s)
    fn = getattr(gp._lib, entry)
    _lib.check(fn(gp._h, _lib.ptr(s), s.size, _lib.ptr(out)), entry)
    ref = np.exp(-s)
    live = s < 700.0
    rel = np.abs(out[live] - ref[live]) / ref[live]
    assert rel.max() < 4.5e-16, rel.max()
    assert np.all(out[~live] == 0.0)
    nan_out = np.empty(1)
    _lib.check(fn(gp._h, _lib.ptr(np.array([np.nan])), 1, _lib.ptr(nan_out)), entry)
    assert np.isnan(nan_out[0])            # NaN queries must stay NaN (approx.py:185 maps them to -inf)


@pytest.mark.parametrize("N,d", [(1, 1), (2, 2), (65, 31), (130, 32), (96, 20)])
def test_edge_shapes(N, d):
    """Smallest training sets and the largest supported dimensionalities (d = 32 switches the variance
    kernel to its 128x128 tiling because the 256x64 one cannot stage 32 x 256 scaled queries)."""
    rng = np.random.default_rng(N * 100 + d)
    X = rng.uniform(-2, 2, size=(N, d))
    y = rng.standard_normal(N)
    logM = np.full(d, np.log(4.0 * d))
    gp, orc = make_pair(X, y, logM, amp=1.7)
    Xq = rng.uniform(-2, 2, size=(300, d))
    check_predict(gp, orc, y, Xq, 1.7)
    assert abs(gp.log_likelihood(y) - orc.log_likelihood(y)) <= 1e-9 * max(1.0, abs(orc.log_likelihood(y)))
    P = np.vstack([gp.get_parameter_vector(), gp.get_parameter_vector() - 0.2])
    ll = gp.log_likelihood_batch(P, y)
    for p, v in zip(P, ll):
        orc.set_parameter_vector(p)
        assert abs(v - orc.log_likelihood(y, quiet=True)) <= 1e-9 * max(1.0, abs(v))


def test_dimension_limits_are_reported():
    from approxposterior_b200 import GP, kernels, _lib
    gp = GP(kernel=kernels.ExpSquaredKernel(np.ones(33), ndim=33))
    with pytest.raises(_lib.ApgpError):
        gp.compute(np.zeros((4, 33)), y=np.zeros(4))


def test_sampler_replay_large_training_set_global_path():
    """(d+1) x N too large for shared memory: the sampler reads the training set through L2 instead."""
    from oracle import stretch_move_oracle
    from oracle.sampler_oracle import gpll_batch
    N, d = 1300, 20
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=9)
    gp, orc = make_pair(X, y, logM)
    lo, hi = np.full(d, -5.0), np.full(d, 5.0)
    nw, nsteps = 44, 15
    rng = np.random.RandomState(4)
    p0 = rng.uniform(-1, 1, size=(nw, d))
    ref = stretch_move_oracle(lambda q: gpll_batch(orc, y, q, lo, hi), p0, nsteps, rng=rng, record=True)
    out = gp.run_ensembles(y, p0, nsteps, bounds=list(zip(lo, hi)), nens=1,
                           replay={k: ref[k][None] for k in ("inds", "zz", "rint", "logu")})
    np.testing.assert_allclose(out["chain"], ref["chain"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(out["log_prob"], ref["log_prob"], rtol=1e-9, atol=1e-9)
    assert np.array_equal(out["naccepted"], ref["naccepted"])


@pytest.mark.parametrize("N0,nadd", [(50, 30), (120, 10), (255, 3)])
def test_append_point_matches_full_compute(N0, nadd):
    """Bordered O(N^2) append (reference approx.py:693-717 refactors from scratch) vs a fresh factorisation:
    alpha, L^-1, log-likelihood and predictions must agree; crossing a 64-row padding boundary falls back."""
    rng = np.random.default_rng(N0)
    d = 3
    X = rng.uniform(-5, 5, size=(N0 + nadd, d))
    y = np.sin(X).sum(axis=1)
    logM = np.log(np.full(d, 3.0))
    gp, _ = make_pair(X[:N0], y[:N0], logM, amp=2.0, mean=0.1)
    fast = 0
    for k in range(N0, N0 + nadd):
        fast += bool(gp.append_point(X[k], y[k]))
    ref, orc = make_pair(X, y, logM, amp=2.0, mean=0.1)
    assert fast >= nadd - 1 - nadd // 64        # only padding-boundary crossings refactor
    assert gp._x.shape == (N0 + nadd, d) and np.array_equal(gp._y, y)
    np.testing.assert_allclose(gp._alpha(), ref._alpha(), rtol=1e-8, atol=1e-10 * np.max(np.abs(ref._alpha())))
    assert np.max(np.abs(gp._linv() @ orc._L - np.eye(N0 + nadd))) < 1e-9
    assert abs(gp.log_likelihood(y) - orc.log_likelihood(y)) <= 1e-9 * abs(orc.log_likelihood(y))
    assert abs(gp.log_determinant - orc.log_determinant) <= 1e-9 * max(1.0, abs(orc.log_determinant))
    Xq = rng.uniform(-5, 5, size=(400, d))
    check_predict(gp, orc, y, Xq, 2.0)
    # a duplicated point makes the bordered pivot vanish only up to the white noise: still positive definite
    assert gp.append_point(X[0], y[0]) in (True, False) and gp.computed


def test_ill_conditioned_against_multiprecision_truth():
    """cond(K) ~ 1e10 (huge amplitude, very long length scale -- the regime optimizeGP's amplitude fits end in,
    reference tests/test_OptimizeGP.py:50).  Neither fp64 implementation can agree with the other to 1e-9
    there; what must hold is that the CUDA path is as close to the 60-digit truth as the oracle is."""
    import mpmath as mp
    mp.mp.dps = 60
    N, amp, logM, wn = 40, 5.7e4, np.array([4.2, 10.8]), -12.0
    theta, y = rosenbrock_training(N)
    mean = float(np.median(y))
    gp, orc = make_pair(theta, y, logM, amp=amp, mean=mean, wn=wn)
    Xq = np.random.default_rng(2).uniform(-5, 5, size=(12, 2))
    mu_g, var_g = gp.predict(y, Xq, return_cov=False, return_var=True)
    mu_o, var_o = orc.predict(y, Xq, return_var=True)
    # multiprecision reference
    w = [mp.e ** (-mp.mpf(float(v))) for v in logM]
    A = mp.mpf(orc.amplitude)
    def k(a, b):
        return A * mp.e ** (-mp.mpf("0.5") * sum(w[i] * (mp.mpf(float(a[i])) - mp.mpf(float(b[i]))) ** 2 for i in range(2)))
    K = mp.matrix(N, N)
    for i in range(N):
        for j in range(N):
            K[i, j] = k(theta[i], theta[j])
        K[i, i] += mp.e ** mp.mpf(wn) + mp.mpf("1.25e-12") ** 2
    r = mp.matrix([mp.mpf(float(v)) - mp.mpf(mean) for v in y])
    alpha = mp.lu_solve(K, r)
    err_g = err_o = verr_g = verr_o = 0.0
    for qi, q in enumerate(Xq):
        ks = mp.matrix([k(q, theta[j]) for j in range(N)])
        mu_t = mp.mpf(mean) + sum(ks[j] * alpha[j] for j in range(N))
        v_t = A - sum(ks[j] * s for j, s in enumerate(mp.lu_solve(K, ks)))
        err_g = max(err_g, abs(float(mp.mpf(float(mu_g[qi])) - mu_t)))
        err_o = max(err_o, abs(float(mp.mpf(float(mu_o[qi])) - mu_t)))
        verr_g = max(verr_g, abs(float(mp.mpf(float(var_g[qi])) - v_t)))
        verr_o = max(verr_o, abs(float(mp.mpf(float(var_o[qi])) - v_t)))
    scale = float(np.max(np.abs(y)))
    assert err_g <= 20 * max(err_o, 1e-12 * scale), (err_g, err_o)
    assert verr_g <= 20 * max(verr_o, 1e-12 * amp), (verr_g, verr_o)


def test_sampler_argument_errors_are_reported():
    from approxposterior_b200 import _lib
    theta, y = rosenbrock_training(30)
    gp, _ = make_pair(theta, y, np.zeros(2))
    b = [(-5, 5), (-5, 5)]
    with pytest.raises(_lib.ApgpError):
        gp.run_ensembles(y, np.zeros((7, 2)), 10, b)            # odd number of walkers
    with pytest.raises(_lib.ApgpError):
        gp.run_ensembles(y, np.zeros((4, 2)), 0, b)             # no steps
    with pytest.raises(ValueError):
        gp.run_ensembles(y, np.zeros((10, 2)), 10, b, nens=3)   # rows not a multiple of nens


@pytest.mark.parametrize("N,d,Q,group", [(1024, 2, 40000, -1), (2048, 5, 70001, 16), (2048, 5, 70001, 8),
                                         (1100, 3, 30011, 6), (1100, 3, 700, 4), (4096, 2, 20000, -1),
                                         (2048, 5, 5, -1), (512, 2, 300, -1), (300, 3, 1, -1)])
def test_grouped_variance_kernel_matches_one_tile_per_cta(N, d, Q, group):
    """G CTAs sharing one query tile (L2-resident K* panels) must reproduce the one-tile-per-CTA kernel.  The variance
    agrees to ~1e-15; the mean adds the same per-column terms in a different order, so it agrees to the rounding of a
    length-N sum of terms bounded by max|alpha| (alpha reaches 6e5 with cancellation on these problems)."""
    import torch
    from approxposterior_b200 import GP, kernels
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + d)
    gp = GP(kernel=kernels.ExpSquaredKernel(np.exp(logM), ndim=d), fit_mean=True, mean=0.1, white_noise=-12.0)
    gp.compute(X, y=y)
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    q = -5.5 + 11.0 * torch.rand((Q, d), dtype=torch.float64, device="cuda", generator=g)
    bounds = [(-5.0, 5.0)] * d
    gp.set_group(0)
    mu0, var0, u0 = gp._predict_raw(q, True, utility="agp", bounds=bounds)
    gp.set_group(group)
    mu_tol = 2.3e-16 * N * float(np.abs(gp._alpha()).max())
    for rep in range(2):                                   # twice: the barrier counters are reset per launch
        mu1, var1, u1 = gp._predict_raw(q, True, utility="agp", bounds=bounds)
        assert float((mu1 - mu0).abs().max()) <= mu_tol
        assert torch.allclose(var1, var0, rtol=0, atol=1e-12)
        fin = torch.isfinite(u0)
        assert torch.equal(fin, torch.isfinite(u1))
        assert float((u1[fin] - u0[fin]).abs().max()) <= mu_tol + 1e-9
    gp.set_group(0)


@pytest.mark.parametrize("cluster", [2, 4, 8])
def test_sampler_cluster_replicas_give_the_same_chain(cluster, monkeypatch):
    """A thread-block cluster per ensemble (state replicated in every CTA's shared memory, accepted moves written to
    all replicas through DSMEM, one cluster barrier per half-step) must reproduce the single-CTA chain bit for bit,
    with Philox draws and with replayed draws."""
    from oracle.sampler_oracle import gpll_batch, stretch_move_oracle
    X, y, logM, _ = synthetic_gp_problem(300, 3, seed=12)
    gp, orc = make_pair(X, y, logM)
    bounds = [(-5.0, 5.0)] * 3
    rng = np.random.default_rng(4)
    p0 = rng.uniform(-3, 3, size=(2 * 60, 3))                 # two ensembles of 60 walkers
    monkeypatch.setenv("APGP_SAMPLER_CLUSTER", "1")
    a = gp.run_ensembles(y, p0, 120, bounds, nens=2, seed=5, thin=3)
    monkeypatch.setenv("APGP_SAMPLER_CLUSTER", str(cluster))
    b = gp.run_ensembles(y, p0, 120, bounds, nens=2, seed=5, thin=3)
    for k in ("chain", "log_prob", "blobs", "naccepted"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    rs = np.random.RandomState(3)
    q0 = rs.uniform(-2, 2, size=(24, 3))
    lo, hi = np.full(3, -5.0), np.full(3, 5.0)
    ref = stretch_move_oracle(lambda q: gpll_batch(orc, y, q, lo, hi), q0, 40, rng=rs, record=True)
    out = gp.run_ensembles(y, q0, 40, bounds, nens=1, replay={k: ref[k][None] for k in ("inds", "zz", "rint", "logu")})
    np.testing.assert_allclose(out["chain"], ref["chain"], rtol=1e-9, atol=1e-9)
    assert np.array_equal(out["naccepted"], ref["naccepted"])


@pytest.mark.parametrize("nens,nw,nsteps,thin", [(3, 40, 125, 4), (1, 120, 61, 1), (300, 32, 200, 2)])
def test_sampler_in_pieces_is_the_same_chain(nens, nw, nsteps, thin, monkeypatch):
    """apgp_sampler_run(on_host=1) runs long chains as several launches so that one piece's rows cross PCIe while the
    next piece samples: the kernel resumes from the previous piece's last stored row, the counter-based draws are
    indexed by the chain's global step and the acceptance counts keep counting.  Any number of pieces -- including the
    automatic choice for results of more than 4 MB (third case) -- must give the single-launch chain bit for bit
    (steps left over after the last stored row included: they still count in naccepted), as must the device-resident
    call, which is never cut."""
    import torch
    X, y, logM, _ = synthetic_gp_problem(300, 3, seed=21)
    gp, _ = make_pair(X, y, logM)
    bounds = [(-5.0, 5.0)] * 3
    rng = np.random.default_rng(8)
    p0 = rng.uniform(-3, 3, size=(nens * nw, 3))
    p0[1] = [7.0, 0.0, 0.0]                                    # a walker outside the prior box: -inf / nan until it moves
    monkeypatch.setenv("APGP_SAMPLER_PIECES", "1")
    ref = gp.run_ensembles(y, p0, nsteps, bounds, nens=nens, seed=77, thin=thin)
    for pieces in ("2", "5", "1000", None):
        if pieces is None:
            monkeypatch.delenv("APGP_SAMPLER_PIECES")
        else:
            monkeypatch.setenv("APGP_SAMPLER_PIECES", pieces)
        l0 = gp.launch_count
        out = gp.run_ensembles(y, p0, nsteps, bounds, nens=nens, seed=77, thin=thin)
        launches = gp.launch_count - l0
        if pieces is not None:
            assert launches == min(int(pieces), nsteps // thin)
        elif (nsteps // thin) * nens * nw * 5 * 8 >= 4 << 20:
            assert launches == 8                                 # the automatic choice cut this one
        for k in ("chain", "log_prob", "blobs", "naccepted"):
            assert np.array_equal(ref[k], out[k], equal_nan=True), (pieces, k)
    dev = gp.run_ensembles(y, p0, nsteps, bounds, nens=nens, seed=77, thin=thin, device_out=True)
    for k in ("chain", "log_prob", "blobs", "naccepted"):
        assert np.array_equal(ref[k], dev[k].cpu().numpy(), equal_nan=True), k


@pytest.mark.parametrize("N,d,Q,kind", [(300, 3, 200000, "bape"), (1100, 5, 170001, None), (256, 2, 600000, "agp")])
def test_pipelined_host_predict_equals_device_resident(N, d, Q, kind, monkeypatch):
    """apgp_predict(on_host=1) cuts large calls into slices whose H2D copy, kernel and D2H copies overlap on three
    streams (double-buffered staging).  Results must be bit-identical to the device-resident call and to the serial
    host path, for pageable and for pinned host buffers, mean-only and fused utility alike."""
    import torch
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + 1)
    gp, _ = make_pair(X, y, logM)
    g = torch.Generator(device="cuda"); g.manual_seed(N)
    q = -5.5 + 11.0 * torch.rand((Q, d), dtype=torch.float64, device="cuda", generator=g)
    bounds = [(-5.0, 5.0)] * d
    ref = gp._predict_raw(q, True, utility=kind, bounds=bounds)
    qh = q.cpu().numpy()
    pinned_q = torch.empty((Q, d), dtype=torch.float64).pin_memory(); pinned_q.copy_(q.cpu())
    for host_q in (qh, pinned_q.numpy()):
        for serial in (False, True):
            if serial:
                monkeypatch.setenv("APGP_NO_PIPELINE", "1")
            else:
                monkeypatch.delenv("APGP_NO_PIPELINE", raising=False)
            out = gp._predict_raw(host_q, True, utility=kind, bounds=bounds)
            for a, b in zip(out, ref):
                if b is None:
                    assert a is None
                else:
                    assert np.array_equal(a, b.cpu().numpy(), equal_nan=True)
    monkeypatch.delenv("APGP_NO_PIPELINE", raising=False)
    m_only = gp._predict_raw(qh, False)[0]
    assert np.array_equal(m_only, gp._predict_raw(q, False)[0].cpu().numpy(), equal_nan=True)


@pytest.mark.parametrize("N,d,nw,nens", [(2000, 10, 60, 1), (1300, 20, 44, 3), (3000, 5, 24, 2)])
def test_sampler_training_set_partitioned_over_the_cluster(N, d, nw, nens, monkeypatch):
    """Training sets too large for one CTA's shared memory are partitioned over the cluster (every CTA keeps a slice
    resident, partial means meet through distributed shared memory and are added in rank order).  Against the
    stream-from-L2 path (APGP_SAMPLER_NO_SPLIT) the log-probabilities differ by summation order only, so short chains
    agree to rounding and accept the same moves; every slice count gives a valid, deterministic chain; and the replayed
    oracle draws are reproduced to 1e-9."""
    from oracle import stretch_move_oracle
    from oracle.sampler_oracle import gpll_batch
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + d)
    gp, orc = make_pair(X, y, logM)
    lo, hi = np.full(d, -5.0), np.full(d, 5.0)
    bounds = list(zip(lo, hi))
    rng = np.random.default_rng(3)
    p0 = rng.uniform(-1, 1, size=(nens * nw, d))
    monkeypatch.setenv("APGP_SAMPLER_NO_SPLIT", "1")
    ref = gp.run_ensembles(y, p0, 12, bounds, nens=nens, seed=4)
    monkeypatch.delenv("APGP_SAMPLER_NO_SPLIT")
    outs = []
    for slices in (None, "2", "4", "8"):
        if slices is None:
            monkeypatch.delenv("APGP_SAMPLER_SPLIT", raising=False)
        else:
            monkeypatch.setenv("APGP_SAMPLER_SPLIT", slices)
        a = gp.run_ensembles(y, p0, 12, bounds, nens=nens, seed=4)
        b = gp.run_ensembles(y, p0, 12, bounds, nens=nens, seed=4)
        assert np.array_equal(a["chain"], b["chain"]) and np.array_equal(a["naccepted"], b["naccepted"])
        np.testing.assert_allclose(a["log_prob"], ref["log_prob"], rtol=1e-10, atol=1e-10)
        np.testing.assert_allclose(a["chain"], ref["chain"], rtol=1e-10, atol=1e-12)
        assert np.array_equal(a["naccepted"], ref["naccepted"])
        outs.append(a)
    monkeypatch.delenv("APGP_SAMPLER_SPLIT", raising=False)
    rs = np.random.RandomState(4)
    q0 = rs.uniform(-1, 1, size=(nw, d))
    yo = y.copy(); yo.setflags(write=False)
    orc_run = stretch_move_oracle(lambda q: gpll_batch(orc, yo, q, lo, hi), q0, 10, rng=rs, record=True)
    out = gp.run_ensembles(y, q0, 10, bounds, nens=1, replay={k: orc_run[k][None] for k in ("inds", "zz", "rint", "logu")})
    np.testing.assert_allclose(out["chain"], orc_run["chain"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(out["log_prob"], orc_run["log_prob"], rtol=1e-9, atol=1e-9)
    assert np.array_equal(out["naccepted"], orc_run["naccepted"])


@pytest.mark.parametrize("N,d,amp", [(70, 2, None), (300, 5, 2.5), (1100, 3, None), (2048, 5, 4.0)])
def test_few_query_predict_kernel(N, d, amp):
    """Calls of at most 16 queries (the reference's one-point-per-call loops, utility.py:131,178,224) run
    predict_few_kernel -- several CTAs per query against the explicit inverse, partial sums added in split order --
    instead of a 256-query DMMA tile: same mean / variance / utility as the oracle (1e-9) and as the tiled kernels."""
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + d)
    gp, orc = make_pair(X, y, logM, amp=amp)
    rng = np.random.default_rng(5)
    A = amp if amp is not None else 1.0
    bounds = [(-3.0, 3.0)] * d
    for Q in (1, 7, 16):
        q = rng.uniform(-2.5, 2.5, size=(Q, d))
        q[-1] = X[3]                                          # a training input: variance ~ noise level
        if Q > 1:
            q[0, 0] = 3.5                                     # outside the box: utility +inf
        outs = {}
        for few in (True, False):
            gp.set_predict_few(few)
            n0 = gp.launch_count
            outs[few] = [np.array(v) for v in gp.predict_utility(y, q, "bape", bounds=bounds)]
            assert gp.launch_count == n0 + 1
        gp.set_predict_few(True)
        mu_o, var_o = orc.predict(y, q, return_var=True)
        for mu, var, util in outs.values():
            check_mean(mu, mu_o, orc, y, q)
            assert np.all(np.abs(var - var_o) <= 1e-9 * A + 1e-9 * np.abs(var_o))
        (mu1, var1, u1), (mu0, var0, u0) = outs[True], outs[False]
        assert np.all(np.abs(mu1 - mu0) <= 1e-10 * np.abs(mu0) + 1e-10 * np.max(np.abs(y)))
        assert np.all(np.abs(var1 - var0) <= 1e-10 * A)
        assert np.array_equal(np.isinf(u1), np.isinf(u0)) and (Q == 1 or np.isposinf(u1[0]))
    # repeated calls re-arm the arrival counters: identical bits
    q = rng.uniform(-2.5, 2.5, size=(5, d))
    a = [np.array(v) for v in gp.predict(y, q, return_var=True)]
    b = [np.array(v) for v in gp.predict(y, q, return_var=True)]
    assert all(np.array_equal(u, v) for u, v in zip(a, b))
