"""CPU tests of the host-side logic: kernels/parameter bookkeeping, lock-step optimiser batching,
the emcee-flow sampler + autocorrelation, MCSE, and that the C-ABI library loads and exports every
symbol include/apgp.h declares (no compute calls: there is no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, rosenbrock_training


def test_library_exports_every_declared_symbol():
    from approxposterior_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "build libapgp.so first (__graft_entry__.build())"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    header = open(os.path.join(ROOT, "include", "apgp.h")).read()
    declared = set(re.findall(r"\b(apgp_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    lib.apgp_version.restype = ctypes.c_int
    assert lib.apgp_version() >= 100


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from approxposterior_b200 import GP, kernels, _lib
    with pytest.raises(_lib.ApgpError):
        GP(kernel=kernels.ExpSquaredKernel([1.0], ndim=1))


def test_product_path_does_not_import_oracle():
    pkg = os.path.join(ROOT, "approxposterior_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), fn


def test_kernel_parameter_layout():
    from approxposterior_b200 import kernels
    k = kernels.ExpSquaredKernel(metric=[2.0, 3.0], ndim=2)
    assert np.allclose(k.get_parameter_vector(), np.log([2.0, 3.0]))
    assert k.get_parameter_names() == ("metric:log_M_0_0", "metric:log_M_1_1")
    kp = 8.0 * k
    assert np.allclose(kp.get_parameter_vector(), [np.log(8.0 / 2), np.log(2.0), np.log(3.0)])
    assert kp.get_parameter_names() == ("k1:log_constant", "k2:metric:log_M_0_0", "k2:metric:log_M_1_1")
    assert np.isclose(kp.amplitude, 8.0) and kp.fit_amp and not k.fit_amp
    kp.set_parameter_vector([0.0, 1.0, 2.0])
    assert np.isclose(kp.amplitude, 2.0) and np.allclose(kp.log_M, [1.0, 2.0])
    with pytest.raises(NotImplementedError):
        k + k
    with pytest.raises(NotImplementedError):
        kernels.LinearKernel(log_gamma2=1.0, order=1, ndim=2)


def test_default_hyper_prior():
    from approxposterior_b200.gpUtils import defaultHyperPrior
    assert defaultHyperPrior([1e6, 19.9, -19.9]) == 0.0
    assert defaultHyperPrior([0.0, 20.1, 0.0]) == -np.inf
    assert defaultHyperPrior([0.0, 0.0, -20.1]) == -np.inf


def test_lockstep_matches_sequential_powell():
    """Lock-step batching must leave each restart's optimiser path untouched."""
    from scipy.optimize import minimize
    from approxposterior_b200._lockstep import run_lockstep
    f = lambda x: float(np.sum((np.asarray(x) - 1.5) ** 2) + np.sin(3 * x[0]))
    x0s = [np.array([0.1 * i, -0.3 * i]) for i in range(1, 7)]
    seq = [minimize(f, x0, method="powell")["x"] for x0 in x0s]
    calls = []

    def batch(xs):
        calls.append(len(xs))
        return [f(x) for x in xs]

    out, ev = run_lockstep(len(x0s), batch, lambda w, g: minimize(g, x0s[w], method="powell")["x"])
    for a, b in zip(seq, out):
        assert np.array_equal(a, b)
    assert max(calls) == len(x0s) and ev.nevals == sum(calls) and ev.nbatches < ev.nevals


def test_lockstep_propagates_errors():
    from approxposterior_b200._lockstep import run_lockstep

    def batch(xs):
        raise ValueError("boom")

    with pytest.raises(ValueError):
        run_lockstep(3, batch, lambda w, g: g(np.zeros(2)))


def test_optimizeGP_lockstep_equals_sequential_on_oracle():
    from oracle import default_gp_oracle
    from approxposterior_b200 import gpUtils

    class BatchedOracle(object):
        """Oracle GP + a log_likelihood_batch so the lock-step branch of optimizeGP is exercised."""
        def __init__(self, gp):
            self.__dict__["gp"] = gp

        def __getattr__(self, k):
            return getattr(self.gp, k)

        def log_likelihood_batch(self, P, y):
            p0 = self.gp.get_parameter_vector()
            out = []
            for p in np.atleast_2d(P):
                self.gp.set_parameter_vector(p)
                out.append(self.gp.log_likelihood(y, quiet=True))
            self.gp.set_parameter_vector(p0)
            return np.array(out)

    res = []
    for batched in (False, True):
        theta, y = rosenbrock_training(30)
        gp = default_gp_oracle(theta, y, fitAmp=False)
        g = BatchedOracle(gp) if batched else gp
        g = gpUtils.optimizeGP(g, theta, y, nGPRestarts=3, method="powell", batched=batched)
        res.append(g.get_parameter_vector())
    assert np.allclose(res[0], res[1], rtol=1e-12, atol=0)


def test_emcee_flow_sampler_burnin_kat():
    """reference tests/test_Burnin.py:17-91: seed 42 line fit, 32 walkers x 5000 -> [iburn, ithin] = [67, 15]
    (rtol 1e-1).  Hitting it requires the restated emcee 3.0.x RNG flow *and* autocorrelation estimator."""
    from approxposterior_b200 import mcmcUtils
    from approxposterior_b200.sampler import EnsembleSampler
    np.random.seed(42)
    N = 50
    x = np.sort(10 * np.random.rand(N))
    obserr = 0.5
    obs = -0.9594 * x + 4.294
    obs += obserr * np.random.randn(N)

    def log_prob(T):
        T = np.atleast_2d(T)
        m, b = T[:, 0], T[:, 1]
        ok = (m > -5.0) & (m < 0.5) & (b > 0.0) & (b < 10.0)
        ll = -0.5 * np.sum((obs[None, :] - (m[:, None] * x[None, :] + b[:, None])) ** 2 / obserr ** 2, axis=1)
        return np.where(ok, ll, -np.inf), np.zeros(len(m))

    p0 = np.random.randn(32, 2)
    sampler = EnsembleSampler(32, 2, log_prob, engine="host-rng")
    with np.errstate(invalid="ignore"):
        sampler.run_mcmc(p0, 5000)
    iburn, ithin = mcmcUtils.estimateBurnin(sampler, estBurnin=True, thinChains=True)
    assert np.allclose([67, 15], [iburn, ithin], rtol=1.0e-1), (iburn, ithin)
    assert sampler.get_chain().shape == (5000, 32, 2)
    assert sampler.get_chain(discard=100, thin=10, flat=True).shape == (490 * 32, 2)
    assert 0.2 < sampler.acceptance_fraction.mean() < 0.9


def test_host_sampler_equals_oracle_sampler():
    from oracle import stretch_move_oracle
    from approxposterior_b200.sampler import EnsembleSampler
    lp = lambda q: (-0.5 * np.sum(np.atleast_2d(q) ** 2, axis=1), np.zeros(len(np.atleast_2d(q))))
    p0 = np.random.RandomState(3).randn(10, 3)
    np.random.seed(11)
    s = EnsembleSampler(10, 3, lp, engine="host-rng")
    s.run_mcmc(p0, 50)
    ref = stretch_move_oracle(lp, p0, 50, rng=np.random.RandomState(11))
    assert np.array_equal(s.get_chain(), ref["chain"])
    assert np.array_equal(s.naccepted, ref["naccepted"])


def test_mcse_kat():
    """reference tests/test_MCSE.py:16-36: AR(1)-like chain MCSE ~ 0.00494 (atol 2.5e-3)."""
    from approxposterior_b200 import mcmcUtils
    np.random.seed(42)
    samples = np.random.randn(10000) * 0.5
    got = mcmcUtils.batchMeansMCSE(samples)
    assert got > 0 and abs(got - 0.5 / np.sqrt(10000)) < 2.5e-3


def test_utilities_scalar_forms_on_oracle_gp():
    """Scalar utility wrappers reproduce the reference KATs when driven with any george-like GP."""
    from oracle import default_gp_oracle
    from approxposterior_b200 import likelihood as lh, utility as ut
    theta, y = rosenbrock_training(20)
    gp = default_gp_oracle(theta, y, fitAmp=False)
    t = np.array([-2.3573, 4.673])
    assert np.allclose(ut.AGPUtility(t, y, gp, lh.rosenbrockLnprior), 37.41585067, rtol=1e-4)
    assert np.allclose(ut.BAPEUtility(t, y, gp, lh.rosenbrockLnprior), 76.15271103, rtol=1e-4)
    assert np.allclose(ut.JonesUtility(t, y, gp, lh.rosenbrockLnprior), 0.0, rtol=1e-4)
    assert ut.BAPEUtility(np.array([6.0, 0.0]), y, gp, lh.rosenbrockLnprior) == np.inf
    assert ut.logsubexp(1.0, 2.0) == -np.inf
    assert np.isclose(ut.logsubexp(2.0, 0.0), np.log(np.exp(2.0) - 1.0))


def test_box_prior_and_fixtures():
    from approxposterior_b200 import likelihood as lh
    p = lh.BoxPrior([(-5, 5), (-5, 5)])
    assert p([0, 0]) == 0.0 and p([5.0, -5.0]) == 0.0 and p([5.01, 0]) == -np.inf and p([np.nan, 0]) == -np.inf
    assert lh.rosenbrockLnlike(np.array([1.0, 1.0])) == 0.0
    assert lh.rosenbrockLnprob(np.array([6.0, 1.0])) == -np.inf
    assert np.isclose(lh.sphereLnlike(np.array([1.0, 2.0])), -5.0)
    assert lh.testBOFnLnPrior(2.5) == -np.inf and lh.testBOFnLnPrior(0.0) == 0.0


def test_shard_bounds_cover_exactly():
    from approxposterior_b200.dist import shard_bounds
    for n in (0, 1, 7, 1000003):
        for ws in (1, 2, 3, 8):
            blocks = [shard_bounds(n, r, ws) for r in range(ws)]
            assert blocks[0][0] == 0 and blocks[-1][1] == n
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(ws - 1))
            sizes = [b - a for a, b in blocks]
            assert max(sizes) - min(sizes) <= 1


class _OracleGP(object):
    """Factory for an oracle GP with george's constructor signature (oracle.refshim.GP) carrying the batched entry
    points, so the whole ApproxPosterior driver (lock-step restarts, design-point loop with the reference's
    rebuild-per-point, host-rng MCMC) runs on CPU."""

    @staticmethod
    def make(ndim, metric, mean, white_noise=-12.0):
        from oracle import UTILITY_BY_NAME, refshim

        class G(refshim.GP):
            def predict_utility(self, y, t, kind, bounds=None, zeta=0.01):
                mu, var = self.predict(y, t, return_var=True)
                fn = UTILITY_BY_NAME[kind]
                return mu, var, (fn(mu, var, np.max(y), zeta, True) if kind == "jones" else fn(mu, var, True))

            def log_likelihood_batch(self, P, y):
                p0 = self.get_parameter_vector()
                out = []
                for p in np.atleast_2d(P):
                    self.set_parameter_vector(p)
                    out.append(self.log_likelihood(y, quiet=True))
                self.set_parameter_vector(p0)
                self.recompute(quiet=True)
                return np.array(out)

        return G(kernel=refshim._ExpSquared(metric, ndim), fit_mean=True, mean=mean, white_noise=white_noise)


def test_approx_posterior_driver_on_oracle_gp(tmp_path):
    """Host logic of ApproxPosterior.run (reference approx.py:229-524) end to end on the CPU oracle."""
    from approxposterior_b200 import approx, likelihood as lh
    np.random.seed(57)
    bounds = [(-5, 5), (-5, 5)]
    theta = lh.rosenbrockSample(30)
    y = np.array([lh.rosenbrockLnlike(t) + lh.rosenbrockLnprior(t) for t in theta])
    gp = _OracleGP.make(2, np.fabs(np.random.randn(2)), float(np.median(y)))
    gp.compute(theta)
    ap = approx.ApproxPosterior(theta=theta, y=y, gp=gp, lnprior=lh.rosenbrockLnprior, lnlike=lh.rosenbrockLnlike,
                                priorSample=lh.rosenbrockSample, bounds=bounds, algorithm="alternate")
    ap.run(m=3, nmax=2, estBurnin=True, nGPRestarts=2, mcmcKwargs={"iterations": 300},
           samplerKwargs={"nwalkers": 10, "engine": "host-rng"}, cache=True, runName=str(tmp_path / "ap"),
           verbose=False, thinChains=True, timing=True, seed=3, convergenceCheck=True, nMinObjRestarts=3)
    assert ap.theta.shape == (36, 2) and ap.y.shape == (36,)
    assert len(ap.trainingTime) == 2 and len(ap.mcmcTime) == 2 and len(ap.iburns) == 2
    assert len(ap.marginalMeans) == 2
    chain = ap.sampler.get_chain()
    assert chain.shape == (300, 10, 2) and np.all(np.abs(chain) <= 5)
    for f in ("apAPFModelCache.npz", "apAPGP.npz", "apAPTiming.npz", "apConvergenceCache.npz", "ap1.npz", "ap0.h5", "ap1.h5"):
        assert (tmp_path / f).exists(), f
    # the chain cache of the last iteration, in emcee's HDFBackend layout (reference approx.py:829-833)
    from approxposterior_b200 import hdf5min
    assert ap.backends == [str(tmp_path / "ap0.h5"), str(tmp_path / "ap1.h5")]
    h5 = hdf5min.read_emcee_backend(str(tmp_path / "ap1.h5"))
    assert np.array_equal(h5["chain"], chain) and np.array_equal(h5["log_prob"], ap.sampler.get_log_prob())
    assert int(h5["attrs"]["iteration"]) == 300 and int(h5["attrs"]["nwalkers"]) == 10 and int(h5["attrs"]["ndim"]) == 2
    cache = np.load(tmp_path / "apAPFModelCache.npz")
    assert np.array_equal(cache["theta"], ap.theta) and np.array_equal(cache["y"], ap.y)
    # _gpll conventions (approx.py:167-188)
    assert ap._gpll(np.array([np.nan, np.nan])) == (-np.inf, np.nan) or np.isnan(ap._gpll(np.array([np.nan, np.nan]))[1])
    assert ap._gpll(np.array([6.0, 0.0]))[0] == -np.inf
    mu, lp = ap._gpll(np.array([0.5, 0.5]))
    assert np.isfinite(mu) and lp == 0.0
    lpb, blob = ap._gpll_batch(np.array([[0.5, 0.5], [6.0, 0.0], [np.nan, 1.0]]))
    assert np.isclose(lpb[0], float(np.ravel(mu)[0])) and lpb[1] == -np.inf and lpb[2] == -np.inf and np.isnan(blob[1])
    # MAP and a short Bayesian-optimisation loop run through the same drivers
    m, v = ap.findMAP(nRestarts=3)
    assert np.all(np.isfinite(m)) and np.isfinite(v)
    soln = ap.bayesOpt(nmax=2, verbose=False, cache=False, nGPRestarts=1, nMinObjRestarts=2, findMAP=False, seed=5)
    assert soln["nev"] == 2 and len(ap.y) == 38


def test_approx_posterior_argument_validation():
    from approxposterior_b200 import approx, likelihood as lh
    theta = np.zeros((4, 2)); y = np.zeros(4)
    with pytest.raises(ValueError):
        approx.ApproxPosterior(None, y, lh.rosenbrockLnprior, lh.rosenbrockLnlike, lh.rosenbrockSample, [(-5, 5)] * 2, gp=1)
    with pytest.raises(ValueError):
        approx.ApproxPosterior(theta, y, lh.rosenbrockLnprior, lh.rosenbrockLnlike, lh.rosenbrockSample, [(-5, 5)], gp=1)
    with pytest.raises(ValueError):
        approx.ApproxPosterior(theta, y, lh.rosenbrockLnprior, lh.rosenbrockLnlike, lh.rosenbrockSample, [(-5, 5)] * 2,
                               gp=1, algorithm="naive")
    bad = theta.copy(); bad[0, 0] = np.inf
    with pytest.raises(ValueError):
        approx.ApproxPosterior(bad, y, lh.rosenbrockLnprior, lh.rosenbrockLnlike, lh.rosenbrockSample, [(-5, 5)] * 2, gp=1)


def test_generator_optimisers_match_scipy():
    """The coroutine restatements of SciPy's Nelder-Mead / Powell must evaluate exactly the points SciPy
    evaluates (same order, bit-identical) and return the same optimum -- including through inf regions."""
    import warnings
    from scipy.optimize import minimize, rosen
    from approxposterior_b200._optimizers import nelder_mead_gen, powell_gen, run_generators, supported
    funcs = {
        "rosen3": (rosen, 3),
        "quad+sin": (lambda x: float(np.sum((x - 1.5) ** 2) + np.sin(3 * x[0])), 2),
        "walled": (lambda x: float(np.sum(np.abs(x)) + (np.inf if x[0] > 3 else 0)), 3),
        "log": (lambda x: float(np.log(x[0]) + x[0] ** 2 + x[1] ** 2) if x[0] > 0 else np.inf, 2),
        "flat": (lambda x: 1.0, 2),
    }
    rng = np.random.default_rng(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for name, (f, n) in funcs.items():
            for trial in range(3):
                x0 = np.abs(rng.standard_normal(n)) * 2 + 0.1
                for method, gen, opts in (("nelder-mead", nelder_mead_gen, {"adaptive": True}),
                                          ("nelder-mead", nelder_mead_gen, {"maxfev": 37}),
                                          ("powell", powell_gen, {}), ("powell", powell_gen, {"maxfev": 29})):
                    assert supported(method, opts)
                    rec, rec2 = [], []
                    res = minimize(lambda x: (rec.append(np.array(x, copy=True)), f(np.asarray(x)))[1], x0,
                                   method=method, options=opts or None)
                    (out,), rounds, evals = run_generators(
                        [gen(x0, **opts)], lambda xs: (rec2.extend(np.array(x, copy=True) for x in xs),
                                                       [f(x) for x in xs])[1])
                    assert len(rec) == len(rec2) == evals, (name, method, opts, len(rec), len(rec2))
                    assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(rec, rec2)), (name, method)
                    assert np.array_equal(res.x, out[0], equal_nan=True)
    assert not supported("powell", {"direc": np.eye(2)}) and not supported("l-bfgs-b", None)
    assert not supported("nelder-mead", {"adaptive": True}, bounds=[(0, 1)])


def test_generator_lockstep_batches_restarts():
    from approxposterior_b200._optimizers import nelder_mead_gen, run_generators
    f = lambda x: float(np.sum((np.asarray(x) - 1.5) ** 2))
    x0s = [np.array([0.1 * i, -0.3 * i, 0.2]) for i in range(1, 8)]
    sizes = []
    out, rounds, evals = run_generators([nelder_mead_gen(x0, adaptive=True) for x0 in x0s],
                                        lambda xs: (sizes.append(len(xs)), [f(x) for x in xs])[1])
    assert max(sizes) == len(x0s) and rounds == len(sizes) and evals == sum(sizes) and rounds < evals
    for (x, fx) in out:
        assert np.allclose(x, 1.5, atol=1e-3) and fx < 1e-6


# ---------------------------------------------------------------- device-optimiser host protocol (no GPU: fake GP)
class _FakeDeviceGP(object):
    """Stands in for approxposterior_b200.GP on the CPU: ``minimize_utility`` / ``minimize_nll`` run the host
    restatements of SciPy's algorithms on an analytic objective, recording how they were called."""
    computed = True

    def __init__(self, fail_first=0):
        self.calls = []
        self.fail_first = fail_first

    def minimize_utility(self, y, x0, utility, bounds=None, method="nelder-mead", options=None, zeta=0.01,
                         evaluate_only=False):
        from approxposterior_b200 import _optimizers as opt
        x0 = np.atleast_2d(x0)
        self.calls.append(dict(kind=utility, R=len(x0), bounds=bounds, method=method, options=options))
        fn = lambda P: [float(np.sum((np.asarray(p) - 1.0) ** 2)) for p in P]
        out, _, evals = opt.run_generators([opt.nelder_mead_gen(t, **(options or {})) for t in x0], fn)
        xs = np.array([o[0] for o in out]); fs = np.array([o[1] for o in out])
        if len(self.calls) <= self.fail_first:
            xs[0] = np.nan                                   # a restart that must be redrawn and re-run
        return xs, fs, np.full(len(x0), evals // len(x0))


def test_minimize_objective_device_engine_protocol():
    from approxposterior_b200 import utility as ut, likelihood as lh
    prior = lh.BoxPrior([(-5, 5), (-5, 5)])
    gp = _FakeDeviceGP(fail_first=1)
    np.random.seed(11)
    y = np.zeros(4)
    x, f = ut.minimizeObjective(ut.BAPEUtility, y, gp, sampleFn=prior.sample, priorFn=prior, nRestarts=4,
                                args=(y, gp, prior))
    assert np.allclose(x, [1.0, 1.0], atol=1e-3) and f < 1e-6
    assert ut.minimizeObjective.last_stats["scheduler"] == "device"
    # first launch carried all 4 restarts with the reference's default options; the failed one was redrawn alone
    assert [c["R"] for c in gp.calls] == [4, 1]
    assert gp.calls[0]["kind"] == "bape" and gp.calls[0]["options"] == {"adaptive": True}
    assert gp.calls[0]["bounds"] == prior.bounds
    # a Python prior without .bounds, or engine="lockstep", never takes the device path
    gp2 = _FakeDeviceGP()
    with pytest.raises(AttributeError):                      # falls through to the lock-step path -> predict_utility
        ut.minimizeObjective(ut.BAPEUtility, y, gp2, sampleFn=prior.sample, priorFn=prior, nRestarts=2,
                             args=(y, gp2, prior), engine="lockstep")
    assert gp2.calls == []


def test_device_optimizer_option_mapping():
    from approxposterior_b200 import _lib
    from approxposterior_b200.gp import GP
    o = GP._opt_opts("nelder-mead", {"adaptive": True, "xatol": 1e-6, "maxfev": 77})
    assert (o.method, o.adaptive, o.xtol, o.ftol, o.maxiter, o.maxfev) == (0, 1, 1e-6, 1e-4, -1, 77)
    o = GP._opt_opts("Powell", {"ftol": 1e-8, "maxiter": np.inf})
    assert (o.method, o.adaptive, o.xtol, o.ftol, o.maxiter, o.maxfev) == (1, 0, 1e-4, 1e-8, _lib.OPT_INF, -1)
    with pytest.raises(KeyError):
        GP._opt_opts("l-bfgs-b", None)


# ---------------------------------------------------------------- grouped variance kernel: host-side work split
def _group_plan(N, Q, requested=-1, sms=148, d=5):
    from approxposterior_b200 import _lib
    lib = _lib.load()
    G = ctypes.c_int()
    tab = np.zeros(512, dtype=np.int32)
    assert lib.apgp_debug_group_plan(N, sms, d, Q, requested, ctypes.byref(G), tab.ctypes.data) == 0
    return G.value, tab


@pytest.mark.parametrize("N,G_expected", [(256, 1), (512, 1), (1024, 4), (1536, 6), (2048, 8), (3000, 12), (4096, 16),
                                          (8192, 32)])
def test_group_plan_throughput_regime(N, G_expected):
    """2^20 queries: group size by L2 footprint and balance; every block-row / column block owned by exactly one rank
    of the group; load (block-row ib costs ib + 1, a column block (2d+12)/64) within 1 % of the mean."""
    G, tab = _group_plan(N, 1 << 20)
    assert G == G_expected
    if G == 1:
        return
    nblk = (N + 63) // 64
    tail = 148 % G
    for base, gs in ((0, G), (256, tail if tail > 0 else G)):
        own2, own1 = tab[base:base + nblk], tab[base + 128:base + 128 + nblk]
        assert own2.min() >= 0 and own2.max() < gs and own1.min() >= 0 and own1.max() < gs
        if 2 * gs > nblk:
            continue                                         # a tiny last group may be unbalanced; it is weighted in
        load = np.zeros(gs)
        for ib in range(nblk):
            load[own2[ib]] += ib + 1
        for cb in range(nblk):
            load[own1[cb]] += (2 * 5 + 12) / 64.0
        assert load.max() / load.mean() < 1.011, (N, gs, load)


def test_group_plan_latency_regime_and_overrides():
    # a handful of queries: the single tile is spread over as many CTAs as the balance allows (nblk / 2 at most)
    assert _group_plan(2048, 5)[0] == 16
    assert _group_plan(1024, 5)[0] == 8
    assert _group_plan(512, 300)[0] == 4
    assert _group_plan(100, 5)[0] == 1                       # 2 block-rows: nothing to share
    # many tiles at small N: one tile per CTA
    assert _group_plan(512, 1 << 20)[0] == 1
    # explicit requests are clamped to nblk / 2 and 64; 0 is handled by the caller (grouping off)
    assert _group_plan(2048, 1 << 20, requested=16)[0] == 16
    assert _group_plan(1024, 1 << 20, requested=64)[0] == 8
    assert _group_plan(8192, 1 << 20, requested=64)[0] == 64
    # from d = 28 the grouped kernel's shared-memory layout no longer fits: one tile per CTA, whatever was requested
    assert _group_plan(2048, 1 << 20, d=27)[0] == 8
    assert _group_plan(2048, 1 << 20, d=28)[0] == 1 and _group_plan(2048, 5, d=31, requested=16)[0] == 1


def test_optimizeGP_device_engine_protocol():
    """gpUtils.optimizeGP on the device engine: start points drawn as the reference draws them (gpUtils.py:227), ONE
    minimize_nll call for all restarts, the best restart (by the optimiser's own objective) installed and recomputed;
    custom hyper-priors, unsupported methods and large training sets stay on the host path."""
    from approxposterior_b200 import gpUtils

    class FakeGP(object):
        def __init__(self, fits=True):
            self.p = np.array([0.0, 1.0, 2.0]); self.calls = []; self.fits = fits; self.recomputed = 0

        def __len__(self):
            return 3

        def get_parameter_vector(self):
            return self.p.copy()

        def set_parameter_vector(self, p):
            self.p = np.asarray(p, dtype=float).copy()

        def recompute(self, quiet=False):
            self.recomputed += 1
            return True

        def can_minimize_nll(self):
            return self.fits

        def minimize_nll(self, P0, y, method="powell", options=None, default_prior=True, evaluate_only=False):
            self.calls.append(dict(P0=np.array(P0), method=method, options=options, default_prior=default_prior))
            P0 = np.atleast_2d(P0)
            res = P0 + 1.0
            f = np.array([3.0, -7.0, np.inf, 1.0])[:len(P0)]          # restart 1 wins; restart 2 failed
            return res, f, np.full(len(P0), 11)

        def log_likelihood_batch(self, P, y, return_grad=False):
            raise AssertionError("the device engine ranks restarts by the optimiser's own objective values")

    y = np.arange(5.0)
    gp = FakeGP()
    np.random.seed(9)
    out = gpUtils.optimizeGP(gp, None, y, nGPRestarts=4, method="powell")
    np.random.seed(9)
    expect_x0 = np.array([[np.median(y)] + [np.random.randn() for _ in range(2)] for _ in range(4)])
    assert out is gp and len(gp.calls) == 1 and gp.recomputed == 1
    assert np.array_equal(gp.calls[0]["P0"], expect_x0) and gp.calls[0]["default_prior"] is True
    assert np.array_equal(gp.p, expect_x0[1] + 1.0)
    assert gpUtils.optimizeGP.last_stats == dict(batches=1, evals=44, scheduler="device")
    # a custom hyper-prior cannot run inside the kernel: host lock step (which needs log_likelihood_batch -> raises here)
    with pytest.raises(AssertionError):
        gpUtils.optimizeGP(FakeGP(), None, y, nGPRestarts=2, gpHyperPrior=lambda p: 0.0)
    with pytest.raises(AssertionError):
        gpUtils.optimizeGP(FakeGP(fits=False), None, y, nGPRestarts=2)
    with pytest.raises(AssertionError):
        gpUtils.optimizeGP(FakeGP(), None, y, nGPRestarts=2, engine="lockstep")


def test_shipped_kernels_have_the_claimed_hardware_paths_and_no_spills():
    """Static check of the built libapgp.so (cuobjdump, no GPU): no kernel spills registers to local memory, the variance
    kernels and the cluster log-likelihood carry DMMA (FP64 tensor pipe), UBLKCP (bulk TMA) and SYNCS (mbarrier)
    instructions, the one-CTA Cholesky uses DMMA, the sampler has its cluster barriers (DESIGN 4.1-4.5, profiles/*_sass_summary.txt)."""
    import shutil
    import sys
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_summary
    finally:
        sys.path.pop(0)
    rows = {r["kernel"]: r for r in sass_summary.collect(os.path.join(ROOT, "approxposterior_b200", "libapgp.so"))}
    assert len(rows) >= 30
    spilled = [k for k, r in rows.items() if r["local"] != 0]
    assert not spilled, spilled
    for k in ("predict_var_group_kernel<256, 64, 4>", "predict_var_kernel<256, 64, 4>", "loglik_group_kernel",
              "minimize_nll_group_kernel"):
        r = rows[k]
        assert r["DMMA"] >= 200 and r["UBLKCP"] >= 8 and r["SYNCS"] >= 20, (k, r)
    for k in ("loglik_small_kernel", "minimize_nll_kernel", "chol_panel_kernel", "chol_update_kernel", "gemm_tile_kernel"):
        assert rows[k]["DMMA"] > 0, k
    assert rows["sampler_kernel"]["CGABAR"] > 0 and rows["sampler_kernel"]["regs"] <= 64


def test_compat_emcee_shim_is_the_oracles_emcee_flow():
    """compat.py's emcee module (product code: what the unmodified reference imports as `emcee` on the engine) against the
    oracle's emcee restatement, on a plain Python log-probability (no GP, no GPU): the same NumPy RNG flow -- chain,
    log-probabilities, blobs, accepted fractions and the final np.random state agree bit for bit; the autocorrelation time
    (one batched FFT here, emcee's per-walker FFTs there) to rounding."""
    import sys
    from oracle import refshim
    from approxposterior_b200 import compat
    lnprob = lambda x: (-0.5 * np.sum(x * x) - 0.1 * np.sum(x ** 4), 1.5)
    outs = []
    for shim in (refshim, compat):
        shim.install()
        try:
            import emcee
            assert emcee.__version__.startswith("3.0")
            np.random.seed(4)
            s = emcee.EnsembleSampler(10, 3, lnprob, blobs_dtype=[("lnprior", float)])
            for _ in s.sample(np.random.randn(10, 3), iterations=400):
                pass
            blobs = s.get_blobs()                              # structured ("lnprior") on the engine shim, plain on the oracle's
            blobs = blobs["lnprior"] if getattr(blobs.dtype, "names", None) else blobs
            outs.append((s.get_chain().copy(), s.get_log_prob().copy(), np.asarray(blobs, dtype=float).copy(),
                         np.asarray(s.acceptance_fraction).copy(), s.get_chain(discard=10, thin=3, flat=True).copy(),
                         np.random.get_state()[1].copy(), np.asarray(s.get_autocorr_time(tol=0))))
        finally:
            shim.uninstall()
            for n in [n for n in sys.modules if n == "emcee" or n.startswith("emcee.")]:
                del sys.modules[n]
    for a, b in zip(outs[0][:-1], outs[1][:-1]):
        assert np.array_equal(a, b)
    np.testing.assert_allclose(outs[1][-1], outs[0][-1], rtol=1e-13)
