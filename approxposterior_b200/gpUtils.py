"""Gaussian-process utilities: mirror of reference ``approxposterior/gpUtils.py`` on the B200 engine.

Same names, arguments and error behaviour as the reference functions (file:line cited per
function); the GP object is ``approxposterior_b200.GP`` instead of ``george.GP`` and the
restarts of ``optimizeGP`` are evaluated side by side on the device.
"""
import numpy as np
from scipy.optimize import minimize

from . import kernels
from . import _optimizers as _opt
from ._lockstep import run_lockstep
from .gp import GP

__all__ = ["defaultHyperPrior", "defaultGP", "optimizeGP"]


def defaultHyperPrior(p):
    """Flat prior keeping every log hyper-parameter in [-20, 20]; the mean (p[0]) is free.
    Reference gpUtils.py:22-43."""
    p = np.asarray(p, dtype=np.float64)
    if np.any(np.fabs(p)[1:] > 20):
        return -np.inf
    return 0.0


def _nll(p, gp, y, priorFn=None):
    """Negative log-likelihood of y under gp at hyper-parameters p (reference gpUtils.py:46-80):
    +inf if the prior rejects p, the covariance is singular, or the likelihood is not finite."""
    if priorFn is not None:
        if not np.isfinite(priorFn(p)):
            return np.inf
    try:
        gp.set_parameter_vector(p)
    except np.linalg.LinAlgError:
        return np.inf
    ll = gp.log_likelihood(y, quiet=True)
    return -ll if np.isfinite(ll) else np.inf


def _grad_nll(p, gp, y, priorFn=None):
    """Gradient of ``_nll`` (reference gpUtils.py:83-111)."""
    if priorFn is not None:
        if not np.isfinite(priorFn(p)):
            return np.full_like(p, np.inf)
    gp.set_parameter_vector(p)
    return -gp.grad_log_likelihood(y, quiet=True)


def _nll_batch(P, gp, y, priorFn=None, with_grad=False):
    """``_nll`` (and, with_grad, ``_grad_nll``) for a list of parameter vectors with one batched device
    evaluation.  Returns a list of floats, or of (nll, grad_nll) pairs."""
    P = [np.asarray(p, dtype=np.float64) for p in P]
    ok = np.array([priorFn is None or np.isfinite(priorFn(p)) for p in P], dtype=bool)
    out = np.full(len(P), np.inf)
    gout = [np.full_like(p, np.inf) for p in P]              # prior rejection: gpUtils.py:105-107
    if np.any(ok):
        Pok = np.array([p for p, k in zip(P, ok) if k])
        if with_grad:
            ll, g = gp.log_likelihood_batch(Pok, y, return_grad=True)
            for i, gi in zip(np.nonzero(ok)[0], g):
                gout[i] = -gi
        else:
            ll = gp.log_likelihood_batch(Pok, y)
        out[ok] = np.where(np.isfinite(ll), -ll, np.inf)
    if with_grad:
        return [(float(f), g) for f, g in zip(out, gout)]
    return out


def defaultGP(theta, y, order=None, white_noise=-12, fitAmp=False):
    """ExpSquared GP with a fitted constant mean and frozen white noise, factorised on theta.
    Reference gpUtils.py:114-181 (consumes one ``np.random.randn(ndim)`` for the initial metric).
    ``order`` (the reference's optional LinearKernel term) is outside the engine's scope."""
    theta = np.asarray(theta).squeeze()
    y = np.asarray(y).squeeze()
    ndim = 1 if theta.ndim <= 1 else theta.shape[-1]

    initialMetric = np.fabs(np.random.randn(ndim))
    kernel = kernels.ExpSquaredKernel(metric=initialMetric, ndim=ndim)
    if fitAmp:
        kernel = np.var(y) * kernel
    if order is not None:
        raise NotImplementedError("defaultGP(order=...) adds a LinearKernel (gpUtils.py:169-173); the B200 engine "
                                  "covers the ExpSquared path only")
    gp = GP(kernel=kernel, fit_mean=True, mean=np.median(y), white_noise=white_noise, fit_white_noise=False)
    gp.compute(theta, y=np.atleast_1d(y))
    return gp


DEVICE_OPTIMIZER = True      # module default for optimizeGP(engine=None)


def _is_default_prior(fn):
    """This module's defaultHyperPrior, or the reference's function of the same name and body (gpUtils.py:22-43) when
    the reference package calls optimizeGP through ``compat.accelerate()``: both are the |p[1:]| <= 20 box the device
    objective applies itself."""
    if fn is defaultHyperPrior:
        return True
    return getattr(fn, "__name__", "") == "defaultHyperPrior" and (getattr(fn, "__module__", "") or "").split(".")[-1] == "gpUtils"


def optimizeGP(gp, theta, y, seed=None, nGPRestarts=1, method="powell", options=None, p0=None,
               gpHyperPrior=defaultHyperPrior, batched=True, engine=None):
    """Maximise the marginal likelihood over nGPRestarts starts (reference gpUtils.py:184-257).

    Start points are drawn exactly as the reference draws them (one ``np.random.randn()`` per
    kernel parameter per restart, gpUtils.py:227; ``seed`` is accepted and unused, as there).
    ``engine="device"`` (default for Powell / Nelder-Mead with the default hyper-prior while the training
    set fits one CTA's shared memory, N <= ~220): every restart is minimised by ONE CTA of
    ``apgp_minimize_nll`` -- SciPy's algorithm restated on the device with the covariance build and the
    Cholesky inside the objective -- so the whole multistart fit is a single launch.
    ``engine="lockstep"`` / larger N: the restarts advance in lock step on the host and every round of
    objective calls is one ``log_likelihood_batch`` launch -- for gradient methods the same launch also
    returns the gradients, at every N (one restart per CTA while the training set fits one CTA's shared
    memory, one thread-block cluster per restart beyond).
    """
    y = np.asarray(y, dtype=np.float64)
    npar = len(gp.get_parameter_vector())
    x0s = []
    for _ in range(nGPRestarts):
        if p0 is None:
            x0 = [np.median(y)] + [np.random.randn() for _ in range(npar - 1)]
        else:
            x0 = np.array(p0) + np.min(p0) * 1.0e-3 * np.random.randn(len(p0))
        x0s.append(np.asarray(x0, dtype=np.float64))

    derivative_free = method in ["nelder-mead", "powell", "cg"]
    use_batch = batched and hasattr(gp, "log_likelihood_batch")

    if engine is None:
        engine = "device" if DEVICE_OPTIMIZER else "lockstep"
    on_device = (engine == "device" and use_batch and _opt.supported(method, options)
                 and (_is_default_prior(gpHyperPrior) or gpHyperPrior is None)
                 and hasattr(gp, "minimize_nll") and gp.can_minimize_nll())

    from . import dist as _dist
    if on_device and _dist.world()[1] > 1:
        # one process per GPU (torchrun): the restarts are sharded over the ranks, one all-gather picks the winner
        pbest, mbest, nfev = _dist.optimize_gp_sharded(gp, y, np.array(x0s), method=method, options=options,
                                                       default_prior=gpHyperPrior is not None)
        res, mll = [pbest], [mbest]
        optimizeGP.last_stats = dict(batches=1, evals=int(nfev), scheduler="device-sharded", world=_dist.world()[1])
    elif on_device:
        res, fres, nfev = gp.minimize_nll(np.array(x0s), y, method=method, options=options,
                                          default_prior=gpHyperPrior is not None)
        res = list(res)
        optimizeGP.last_stats = dict(batches=1, evals=int(np.sum(nfev)), scheduler="device")
        # the optimiser's own objective value at its optimum IS -log-likelihood there (gpUtils.py:243-247 recomputes it)
        mll = [(-f if np.isfinite(f) else -np.inf) for f in fres]
    elif use_batch and _opt.supported(method, options):
        # thread-free lock step: SciPy's Powell / Nelder-Mead restated as coroutines (same iterates)
        make = _opt.powell_gen if str(method).lower() == "powell" else _opt.nelder_mead_gen
        out, rounds, evals = _opt.run_generators([make(x0, **(options or {})) for x0 in x0s],
                                                 lambda P: _nll_batch(P, gp, y, gpHyperPrior))
        res = [o[0] for o in out]
        optimizeGP.last_stats = dict(batches=rounds, evals=evals, scheduler="generators")
        mll = list(gp.log_likelihood_batch(np.array(res), y))
    elif use_batch:
        # derivative-free: f(x) -> nll; gradient methods: f(x) -> (nll, grad_nll) in the same batched launch
        def worker(wid, f):
            return minimize(f, x0s[wid], method=method, jac=None if derivative_free else True, bounds=None,
                            options=options)["x"]

        res, ev = run_lockstep(nGPRestarts,
                               lambda P: _nll_batch(P, gp, y, gpHyperPrior, with_grad=not derivative_free), worker)
        optimizeGP.last_stats = dict(batches=ev.nbatches, evals=ev.nevals, scheduler="threads")
        mll = list(gp.log_likelihood_batch(np.array(res), y))
    else:
        res, mll = [], []
        jac = None if derivative_free else _grad_nll
        for x0 in x0s:
            resii = minimize(_nll, x0, args=(gp, y, gpHyperPrior), method=method, jac=jac, bounds=None,
                             options=options)["x"]
            res.append(resii)
            gp.set_parameter_vector(resii)
            gp.recompute(quiet=True)
            mll.append(gp.log_likelihood(y, quiet=True))

    ind = np.argmax(mll)
    gp.set_parameter_vector(res[ind])
    gp.recompute()
    return gp


optimizeGP.last_stats = None
