"""``GP``: the george.GP duck type approxposterior drives, backed by libapgp on a B200.

Surface kept (reference call sites):
  ctor      ``GP(kernel=, fit_mean=True, mean=, white_noise=, fit_white_noise=False)``  gpUtils.py:176-177, approx.py:712-715
  compute / recompute / computed                                                     gpUtils.py:178,244,254; utility.py:130
  predict(y, t, return_cov=False, return_var=False|True)                             approx.py:178-180; utility.py:131,178,224
  log_likelihood(y, quiet=True) / grad_log_likelihood(y, quiet=True)                 gpUtils.py:78,110,247
  get/set_parameter_vector, get_parameter_names, len()                               gpUtils.py:74,227,243; approx.py:431,706,716
  kernel / mean / white_noise attributes                                             approx.py:712-714

Batched extras (the data-parallel form of the same calls):
  predict(..) accepts any number of query rows, NumPy (host) or torch CUDA tensors;
  ``predict_utility`` fuses the AGP/BAPE/Jones epilogue and the box-prior gate;
  ``log_likelihood_batch`` evaluates many hyper-parameter vectors at once;
  ``run_ensembles`` runs the device-resident stretch-move sampler.
"""
import ctypes as C

import numpy as np

from . import _lib
from .kernels import ExpSquaredKernel, Product

__all__ = ["GP"]


def _default_device():
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except Exception:
        pass
    return 0


_HANDLE_POOL = {}            # device ordinal -> idle apgp handles (reset, buffers kept)
_HANDLE_POOL_MAX = 4


def _is_torch(a):
    return hasattr(a, "data_ptr") and hasattr(a, "is_cuda")


class GP(object):
    def __init__(self, kernel=None, fit_mean=False, mean=0.0, white_noise=-12.0, fit_white_noise=False,
                 device=None, **kwargs):
        if kernel is None or not isinstance(kernel, (ExpSquaredKernel, Product)):
            raise NotImplementedError("the B200 engine supports ExpSquaredKernel, optionally scaled by a constant")
        if fit_white_noise:
            raise NotImplementedError("white noise is frozen on this path (fit_white_noise=False, gpUtils.py:177)")
        if kwargs.get("solver") is not None:
            raise NotImplementedError("only the dense (BasicSolver-equivalent) factorisation is implemented")
        mean = float(np.asarray(mean))
        self.kernel = kernel
        self.fit_mean = bool(fit_mean)
        self.mean = float(mean)
        self.white_noise = float(white_noise)
        self.fit_white_noise = False
        self.computed = False
        self._dirty = True
        self._x = None
        self._y = None
        self._device = _default_device() if device is None else int(device)
        self._lib = _lib.load()
        pool = _HANDLE_POOL.get(self._device)
        if pool:
            h = pool.pop()                   # a recycled handle: buffers, stream and pinned staging already exist
        else:
            h = C.c_void_p()
            _lib.check(self._lib.apgp_create(C.byref(h), self._device), "apgp_create")
        self._h = h
        self._logdet = np.nan
        self._loglik = -np.inf
        self._ll_cache = None              # (parameter vector, log-likelihood) of the last deferred evaluation
        self._training_uploaded = False

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                pool = _HANDLE_POOL.setdefault(self._device, [])
                # the reference builds a fresh george.GP for every new design point (approx.py:712-717): keep a few
                # handles alive and reset them instead of destroying / re-creating streams, pinned memory and buffers
                if len(pool) < _HANDLE_POOL_MAX and self._lib.apgp_reset(h) == 0:
                    pool.append(h)
                else:
                    self._lib.apgp_destroy(h)
            except Exception:
                pass
            self._h = None

    # ------------------------------------------------------------------ parameters
    def __len__(self):
        return (1 if self.fit_mean else 0) + len(self.kernel)

    def get_parameter_names(self):
        names = ("mean:value",) if self.fit_mean else ()
        return names + tuple("kernel:" + n for n in self.kernel.get_parameter_names())

    def get_parameter_vector(self):
        head = [self.mean] if self.fit_mean else []
        return np.concatenate([head, self.kernel.get_parameter_vector()]).astype(np.float64)

    def set_parameter_vector(self, p):
        p = np.asarray(p, dtype=np.float64).ravel()
        if p.size != len(self):
            raise ValueError("dimension mismatch: expected %d parameters, got %d" % (len(self), p.size))
        if np.array_equal(p, self.get_parameter_vector()):
            return                                  # unchanged: keep the factorisation
        k = 0
        if self.fit_mean:
            self.mean = float(p[0])
            k = 1
        self.kernel.set_parameter_vector(p[k:])
        self._dirty = True

    @property
    def ndim(self):
        return self.kernel.ndim

    @property
    def log_determinant(self):
        return self._logdet

    @property
    def launch_count(self):
        return int(self._lib.apgp_launch_count(self._h))

    def set_group(self, group):
        """CTAs sharing one query tile in the variance kernel (0: one tile per CTA, -1: automatic, 2..64: fixed);
        with groups the K* panels in flight stay in L2 instead of streaming through HBM."""
        _lib.check(self._lib.apgp_set_group(self._h, int(group)), "apgp_set_group")

    def set_var_engine(self, engine):
        """Engine of the variance product in grouped predict calls: ``"i8"`` (default; int8 tensor cores, exact-integer
        split of the FP64 operands, used from N = 1024) or ``"dmma"`` (FP64 tensor cores)."""
        codes = {"dmma": 0, "i8": 1}
        if engine not in codes:
            raise ValueError("engine must be 'i8' or 'dmma'")
        _lib.check(self._lib.apgp_set_var_engine(self._h, codes[engine]), "apgp_set_var_engine")

    def set_predict_few(self, enable=True):
        """Calls of at most 16 queries use the few-query kernel (default) or, with ``enable=False``, the tiled kernels."""
        _lib.check(self._lib.apgp_set_predict_few(self._h, 1 if enable else 0), "apgp_set_predict_few")

    # ------------------------------------------------------------------ factorisation
    def _parse(self, t):
        t = np.asarray(t, dtype=np.float64)
        if t.ndim == 0:
            t = t.reshape(1, 1)
        elif t.ndim == 1:
            t = t.reshape(-1, 1)
        if t.ndim != 2 or t.shape[1] != self.ndim:
            raise ValueError("dimension mismatch")
        return np.ascontiguousarray(t)

    def compute(self, x, yerr=None, y=None, **kwargs):
        """george.GP.compute(x).  ``y`` is an optional hint (george only sees y at predict time);
        when it is omitted the factorisation is finished on the first call that supplies y.
        ``yerr``: approxposterior never passes one (gpUtils.py:178, approx.py:717), so only george's default
        (1.25e-12, whose square is added to the diagonal next to exp(white_noise)) is accepted; anything else raises
        instead of being dropped.  Note the constructor's ``white_noise`` default is -12 (what gpUtils.defaultGP
        passes), not george's None = log(1.25e-12 ** 2)."""
        if yerr is not None and np.any(np.asarray(yerr, dtype=np.float64) != 1.25e-12):
            raise NotImplementedError("per-point observational errors (yerr) are outside the engine's scope: "
                                      "the diagonal carries exp(white_noise) + (1.25e-12)^2 only")
        self._x = self._parse(x)
        self._y = None if y is None else np.ascontiguousarray(np.asarray(y, dtype=np.float64).ravel())
        if self._y is not None and self._y.size != self._x.shape[0]:
            raise ValueError("dimension mismatch")
        self._training_uploaded = False
        self._dirty = True
        self._ll_cache = None
        self.computed = False
        self.recompute()

    def _upload_training(self):
        y = self._y if self._y is not None else np.zeros(self._x.shape[0])
        _lib.check(self._lib.apgp_set_training(self._h, _lib.ptr(self._x), _lib.ptr(y), self._x.shape[0],
                                               self.ndim, 1), "apgp_set_training")
        self._training_uploaded = True

    def recompute(self, quiet=False, **kwargs):
        if not self._dirty and self.computed:
            return True
        if self._x is None:
            raise RuntimeError("You need to compute the model first")
        if not self._training_uploaded:
            self._upload_training()
        logM = np.ascontiguousarray(self.kernel.log_M, dtype=np.float64)
        _lib.check(self._lib.apgp_set_hyper(self._h, self.mean, float(self.kernel.amplitude), _lib.ptr(logM),
                                            self.white_noise), "apgp_set_hyper")
        logdet, ll, info = C.c_double(), C.c_double(), C.c_int()
        st = _lib.check(self._lib.apgp_factorize(self._h, C.byref(logdet), C.byref(ll), C.byref(info)),
                        "apgp_factorize")
        if st == _lib.APGP_NOT_POSDEF:
            self.computed = False
            self._loglik = -np.inf
            if quiet:
                return False
            raise np.linalg.LinAlgError("covariance matrix is not positive definite (pivot %d)" % info.value)
        self._logdet, self._loglik = logdet.value, ll.value
        self.computed = True
        self._dirty = False
        return True

    def append_point(self, x_new, y_new):
        """Grow the training set by one point with a bordered O(N^2) update of the factorisation (L, L^-1,
        alpha, log-determinant, log-likelihood) -- what the reference obtains by rebuilding and re-computing
        the GP from scratch for every new design point (approx.py:693-717).  Hyper-parameters are unchanged.
        Falls back to a full ``compute`` when the padded device buffers are full or the update is not
        positive definite.  Returns True if the fast path was taken."""
        x_new = np.ascontiguousarray(np.asarray(x_new, dtype=np.float64).ravel())
        y_new = float(np.asarray(y_new, dtype=np.float64).ravel()[0])
        if x_new.size != self.ndim:
            raise ValueError("dimension mismatch")
        X = np.vstack([self._x, x_new[None, :]])
        Y = np.concatenate([self._y if self._y is not None else np.zeros(self._x.shape[0]), [y_new]])
        if self.computed and not self._dirty and self._y is not None and self._training_uploaded:
            logdet, ll = C.c_double(), C.c_double()
            st = _lib.check(self._lib.apgp_append_point(self._h, _lib.ptr(x_new), y_new, C.byref(logdet), C.byref(ll)),
                            "apgp_append_point")
            if st == _lib.APGP_OK:
                self._x, self._y = np.ascontiguousarray(X), Y
                self._logdet, self._loglik = logdet.value, ll.value
                return True
        self.compute(X, y=Y)
        return False

    def _sync_y(self, y):
        """Make the device-side y (hence alpha and the stored log-likelihood) match ``y``."""
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).ravel())
        if self._x is None:
            raise RuntimeError("You need to compute the model first")
        if y.size != self._x.shape[0]:
            raise ValueError("dimension mismatch")
        if self._y is None or not np.array_equal(y, self._y):
            self._y = y.copy()
            self._training_uploaded = False
            self._dirty = True
            self._ll_cache = None

    # ------------------------------------------------------------------ predict
    def _predict_raw(self, t, want_var, utility=None, bounds=None, ybest=0.0, zeta=0.01, want_mu=True, out=None):
        opts = _lib.PredictOpts()
        opts.want_var = 1 if want_var else 0
        opts.utility = _lib.UTIL_KINDS[utility]
        opts.ybest, opts.zeta = float(ybest), float(zeta)
        if bounds is not None:
            opts.has_box = 1
            _lib.fill_bounds(opts.lo, opts.hi, bounds, self.ndim)
        if _is_torch(t):
            import torch
            if not t.is_cuda or t.dtype != torch.float64:
                raise ValueError("torch queries must be float64 CUDA tensors")
            if t.dim() != 2 or t.shape[1] != self.ndim:
                raise ValueError("dimension mismatch")
            t = t.contiguous()
            Q = t.shape[0]
            mk = lambda: torch.empty(Q, dtype=torch.float64, device=t.device)
            on_host = 0
            # order the engine's stream after the producer of `t`, and torch after the engine
            # (torch's default stream has handle 0; cudaStreamLegacy == 0x1 names it explicitly)
            sh = torch.cuda.current_stream(t.device).cuda_stream or 1
            _lib.check(self._lib.apgp_set_stream(self._h, C.c_void_p(sh)), "apgp_set_stream")
        else:
            t = self._parse(t)
            Q = t.shape[0]
            mk = lambda: np.empty(Q, dtype=np.float64)
            on_host = 1
        if out is not None:                      # caller-provided (e.g. pinned) result buffers, NumPy-style
            mu, var, util = out
            for o in (mu, var, util):
                if o is not None and (o.shape != (Q,) or (on_host and (o.dtype != np.float64 or not o.flags.c_contiguous))):
                    raise ValueError("out buffers must be contiguous float64 of shape (Q,)")
        else:
            mu = mk() if want_mu else None
            var = mk() if want_var else None
            util = mk() if utility not in (None, "none") else None
        _lib.check(self._lib.apgp_predict(self._h, _lib.ptr(t), Q, _lib.ptr(mu), _lib.ptr(var), _lib.ptr(util),
                                          C.byref(opts), on_host), "apgp_predict")
        return mu, var, util

    def predict(self, y, t, return_cov=True, return_var=False, **kwargs):
        """george.GP.predict; only the forms approxposterior uses (return_cov=False) are provided."""
        if return_cov and not return_var:
            raise NotImplementedError("predictive covariance matrices are not used by approxposterior "
                                      "(approx.py:178-180, utility.py:131); pass return_cov=False")
        self._sync_y(y)
        self.recompute()
        mu, var, _ = self._predict_raw(t, want_var=bool(return_var))
        if return_var:
            return mu, var
        return mu

    def predict_utility(self, y, t, utility, bounds=None, zeta=0.01, out=None):
        """(mu, var, util) for every row of ``t`` with the reference's utility epilogue fused in
        (utility.py:136,183,229-244) and ``+inf`` outside ``bounds`` (the priorFn gate).
        ``out=(mu, var, util)`` reuses caller-owned result buffers (pinned host memory makes the D2H
        copies asynchronous-capable and skips three allocations per call)."""
        self._sync_y(y)
        self.recompute()
        return self._predict_raw(t, True, utility=str(utility).lower(), bounds=bounds,
                                 ybest=float(np.max(self._y)), zeta=zeta, out=out)

    # ------------------------------------------------------------------ likelihood
    def log_likelihood(self, y, quiet=False):
        """george.GP.log_likelihood.  With ``quiet=True`` and changed hyper-parameters -- the call gpUtils._nll makes
        once per optimiser evaluation (gpUtils.py:74-78) -- only the log-likelihood kernel runs (covariance build +
        Cholesky + reductions, one launch); the full factorisation behind predict (explicit inverse, alpha, packed
        operands) is deferred until something needs it (recompute / predict)."""
        self._sync_y(y)
        if quiet and self._dirty and self._x is not None:
            p = self.get_parameter_vector()
            if self._ll_cache is not None and np.array_equal(self._ll_cache[0], p):
                return self._ll_cache[1]
            ll = float(self.log_likelihood_batch(p[None, :], self._y)[0])
            ll = ll if np.isfinite(ll) else -np.inf
            self._ll_cache = (p.copy(), ll)
            return ll
        if not self.recompute(quiet=quiet):
            return -np.inf
        ll = self._loglik
        return ll if np.isfinite(ll) else -np.inf

    lnlikelihood = log_likelihood

    def nll(self, vector, y, quiet=True):
        self.set_parameter_vector(vector)
        return -self.log_likelihood(y, quiet=quiet)

    def grad_log_likelihood(self, y, quiet=False):
        self._sync_y(y)
        if not self.recompute(quiet=quiet):
            return np.zeros(len(self))
        fit_amp = 1 if self.kernel.fit_amp else 0
        g = np.zeros(1 + fit_amp + self.ndim)
        _lib.check(self._lib.apgp_grad_log_likelihood(self._h, fit_amp, _lib.ptr(g)), "apgp_grad_log_likelihood")
        return g if self.fit_mean else g[1:]

    def log_likelihood_batch(self, P, y, return_grad=False):
        """log-likelihood of ``y`` for every row of ``P`` (george parameter-vector layout) in one
        batched device pass; ``-inf`` where the covariance is not positive definite
        (the quiet=True convention of gpUtils._nll, gpUtils.py:78-79).  ``return_grad`` adds the
        gradients (rows of zeros where the likelihood is -inf, as grad_log_likelihood(quiet=True)), from the
        same single launch at every N: the one-restart-per-CTA kernel while the training set fits one CTA's
        shared memory, the cluster-per-vector kernel with gradients beyond.  Leaves the GP's own
        hyper-parameters untouched."""
        P = np.ascontiguousarray(np.atleast_2d(np.asarray(P, dtype=np.float64)))
        if P.shape[1] != len(self):
            raise ValueError("dimension mismatch")
        self._sync_y(y)
        if not self._training_uploaded:
            self._upload_training()
        fit_amp = 1 if self.kernel.fit_amp else 0
        Pfull = P if self.fit_mean else np.ascontiguousarray(np.hstack([np.full((P.shape[0], 1), self.mean), P]))
        ll = np.empty(Pfull.shape[0])
        grad = np.empty_like(Pfull) if return_grad else None
        st = _lib.check(self._lib.apgp_loglik_batch(self._h, _lib.ptr(Pfull), Pfull.shape[0], Pfull.shape[1], fit_amp,
                                                    self.white_noise, _lib.ptr(ll), _lib.ptr(grad)), "apgp_loglik_batch")
        if st == _lib.APGP_NEEDS_HOST:
            # gradients requested under a forced value-only kernel (APGP_LOGLIK_PATH=group|tiled): one factorisation
            # per vector on the single-GP path (explicit inverse + trace products)
            keep = self.get_parameter_vector()
            for r in range(P.shape[0]):
                self.set_parameter_vector(P[r])
                ll[r] = self.log_likelihood(self._y, quiet=True)
                g = self.grad_log_likelihood(self._y, quiet=True)
                grad[r] = g if self.fit_mean else np.concatenate([[0.0], g])
            self.set_parameter_vector(keep)
            self.recompute(quiet=True)
        if not return_grad:
            return ll
        return ll, (grad if self.fit_mean else grad[:, 1:])

    # ------------------------------------------------------------------ device-resident optimisers
    @staticmethod
    def _opt_opts(method, options):
        """(method, options) of scipy.optimize.minimize -> apgp_opt_opts (same defaults as SciPy)."""
        m = str(method).lower()
        opts = dict(options or {})
        o = _lib.OptOpts()
        o.method = _lib.OPT_METHODS[m]
        o.adaptive = 1 if opts.get("adaptive", False) else 0
        if m == "nelder-mead":
            o.xtol, o.ftol = float(opts.get("xatol", 1e-4)), float(opts.get("fatol", 1e-4))
        else:
            o.xtol, o.ftol = float(opts.get("xtol", 1e-4)), float(opts.get("ftol", 1e-4))

        def lim(v):
            if v is None:
                return -1
            return _lib.OPT_INF if v == np.inf else int(v)
        o.maxiter, o.maxfev = lim(opts.get("maxiter")), lim(opts.get("maxfev"))
        return o

    def minimize_utility(self, y, x0, utility, bounds=None, method="nelder-mead", options=None, zeta=0.01,
                         evaluate_only=False):
        """``scipy.optimize.minimize(fn, x0[r], method=method, options=options)`` for every row of ``x0`` in ONE
        launch (one CTA per start; reference utility.py:332-371).  ``fn`` is the AGP/BAPE/Jones utility exactly
        as utility.py:99-250 evaluates it at a single point (``+inf`` outside ``bounds``), or ``"negmean"``
        (findMAP's objective, approx.py:909-914).  Returns (x [R,d], f [R], nfev [R]).  ``evaluate_only``
        returns fn(x0) -- the very function the device optimiser minimises."""
        self._sync_y(y)
        self.recompute()
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(-1, self.ndim))
        R = x0.shape[0]
        obj = _lib.PredictOpts()
        obj.want_var = 1
        obj.utility = _lib.UTIL_KINDS[str(utility).lower()]
        obj.ybest, obj.zeta = float(np.max(self._y)), float(zeta)
        if bounds is not None:
            obj.has_box = 1
            _lib.fill_bounds(obj.lo, obj.hi, bounds, self.ndim)
        o = self._opt_opts(method, options)
        x, f, stats = np.empty_like(x0), np.empty(R), np.zeros((R, 3), dtype=np.int64)
        _lib.check(self._lib.apgp_minimize_utility(self._h, C.byref(obj), C.byref(o), _lib.ptr(x0), R, _lib.ptr(x),
                                                   _lib.ptr(f), _lib.ptr(stats), 1 if evaluate_only else 0),
                   "apgp_minimize_utility")
        self.last_opt_stats = stats          # per start: evaluations, iterations, SM clock cycles
        return x, f, stats[:, 0].copy()

    def can_minimize_nll(self):
        """True when the training set fits the one-restart-per-CTA shared-memory optimiser (N <= ~220)."""
        if self._x is None:
            return False
        if not self._training_uploaded:
            self._upload_training()
        return bool(self._lib.apgp_minimize_nll_fits(self._h, len(self) if self.fit_mean else len(self) + 1))

    def minimize_nll(self, P0, y, method="powell", options=None, default_prior=True, evaluate_only=False):
        """``scipy.optimize.minimize(_nll, P0[r], method=method, options=options)`` for every row of ``P0`` in ONE
        launch (one CTA per restart; reference gpUtils.py:223-247 with _nll of gpUtils.py:46-80).
        ``default_prior`` applies gpUtils.defaultHyperPrior inside the objective.  Returns (p [R,P], nll [R], nfev [R]).
        Leaves the GP's own hyper-parameters untouched."""
        if not self.fit_mean:
            raise NotImplementedError("minimize_nll needs fit_mean=True (the gpUtils.defaultGP layout)")
        P0 = np.ascontiguousarray(np.atleast_2d(np.asarray(P0, dtype=np.float64)))
        if P0.shape[1] != len(self):
            raise ValueError("dimension mismatch")
        self._sync_y(y)
        if not self._training_uploaded:
            self._upload_training()
        R = P0.shape[0]
        o = self._opt_opts(method, options)
        p, f, stats = np.empty_like(P0), np.empty(R), np.zeros((R, 3), dtype=np.int64)
        _lib.check(self._lib.apgp_minimize_nll(self._h, C.byref(o), _lib.ptr(P0), R, P0.shape[1],
                                               1 if self.kernel.fit_amp else 0, self.white_noise,
                                               1 if default_prior else 0, _lib.ptr(p), _lib.ptr(f), _lib.ptr(stats),
                                               1 if evaluate_only else 0), "apgp_minimize_nll")
        self.last_opt_stats = stats
        return p, f, stats[:, 0].copy()

    # ------------------------------------------------------------------ sampler
    def run_ensembles(self, y, p0, nsteps, bounds, nens=1, a=2.0, seed=0, thin=1, lnprior_const=0.0, replay=None,
                      device_out=False):
        """Device-resident stretch-move sampling of the surrogate posterior mean (emcee as driven
        from approx.py:839-847).  ``p0`` is (nens*nwalkers, ndim); returns dict(chain, log_prob,
        blobs, naccepted) with chain shaped (nsteps//thin, nens*nwalkers, ndim).
        ``device_out=True`` (or a torch CUDA ``p0``): the results stay on the GPU as torch tensors -- the chain of
        65 536 walkers is never copied to the host unless asked for (``integrated_time`` works on it in place)."""
        self._sync_y(y)
        self.recompute()
        if device_out or _is_torch(p0):
            return self._run_ensembles_device(p0, nsteps, bounds, nens, a, seed, thin, lnprior_const, replay)
        p0 = np.ascontiguousarray(np.asarray(p0, dtype=np.float64).reshape(-1, self.ndim))
        W = p0.shape[0]
        if W % nens:
            raise ValueError("p0 rows must be a multiple of nens")
        nw = W // nens
        o = _lib.SamplerOpts()
        o.nens, o.nwalkers, o.nsteps, o.thin = int(nens), int(nw), int(nsteps), int(thin)
        o.a, o.seed, o.lnprior_const = float(a), int(seed) & (2**64 - 1), float(lnprior_const)
        _lib.fill_bounds(o.lo, o.hi, bounds, self.ndim)
        keep = []
        if replay is not None:
            ri = np.ascontiguousarray(replay["inds"], dtype=np.int32)
            rz = np.ascontiguousarray(replay["zz"], dtype=np.float64)
            rr = np.ascontiguousarray(replay["rint"], dtype=np.int32)
            rl = np.ascontiguousarray(replay["logu"], dtype=np.float64)
            keep = [ri, rz, rr, rl]
            o.replay_inds, o.replay_zz, o.replay_rint, o.replay_logu = (_lib.ptr(ri), _lib.ptr(rz), _lib.ptr(rr),
                                                                         _lib.ptr(rl))
        ns = nsteps // thin
        chain = np.empty((ns, W, self.ndim))
        logp = np.empty((ns, W))
        blob = np.empty((ns, W))
        nacc = np.zeros(W, dtype=np.int32)
        _lib.check(self._lib.apgp_sampler_run(self._h, C.byref(o), _lib.ptr(p0), _lib.ptr(chain), _lib.ptr(logp),
                                              _lib.ptr(blob), _lib.ptr(nacc), 1), "apgp_sampler_run")
        del keep
        return dict(chain=chain, log_prob=logp, blobs=blob, naccepted=nacc)

    def _torch_stream(self, dev):
        """Run the engine on torch's current stream of ``dev`` (so torch sees the results in stream order)."""
        import torch
        sh = torch.cuda.current_stream(dev).cuda_stream or 1
        _lib.check(self._lib.apgp_set_stream(self._h, C.c_void_p(sh)), "apgp_set_stream")

    def _run_ensembles_device(self, p0, nsteps, bounds, nens, a, seed, thin, lnprior_const, replay):
        import torch
        if replay is not None:
            raise ValueError("replayed draws are a host-side test facility: use device_out=False")
        dev = torch.device("cuda", self._device)
        if _is_torch(p0):
            p0 = p0.to(device=dev, dtype=torch.float64).reshape(-1, self.ndim).contiguous()
        else:
            p0 = torch.from_numpy(np.ascontiguousarray(np.asarray(p0, dtype=np.float64).reshape(-1, self.ndim))).to(dev)
        W = p0.shape[0]
        if W % nens:
            raise ValueError("p0 rows must be a multiple of nens")
        o = _lib.SamplerOpts()
        o.nens, o.nwalkers, o.nsteps, o.thin = int(nens), int(W // nens), int(nsteps), int(thin)
        o.a, o.seed, o.lnprior_const = float(a), int(seed) & (2**64 - 1), float(lnprior_const)
        _lib.fill_bounds(o.lo, o.hi, bounds, self.ndim)
        ns = nsteps // thin
        chain = torch.empty((ns, W, self.ndim), dtype=torch.float64, device=dev)
        logp = torch.empty((ns, W), dtype=torch.float64, device=dev)
        blob = torch.empty((ns, W), dtype=torch.float64, device=dev)
        nacc = torch.zeros(W, dtype=torch.int32, device=dev)
        self._torch_stream(dev)
        _lib.check(self._lib.apgp_sampler_run(self._h, C.byref(o), _lib.ptr(p0), _lib.ptr(chain), _lib.ptr(logp),
                                              _lib.ptr(blob), _lib.ptr(nacc), 0), "apgp_sampler_run")
        return dict(chain=chain, log_prob=logp, blobs=blob, naccepted=nacc)

    def integrated_time(self, chain, discard=0, thin=1, c=5.0):
        """emcee's integrated autocorrelation time (per dimension) of ``chain`` (n_t, n_walkers, ndim) restricted to
        ``chain[discard + thin - 1::thin]`` -- NOT multiplied by ``thin`` -- computed on the device by direct lagged sums
        over just the lags Sokal's window needs (reference mcmcUtils.py:198 via emcee's get_autocorr_time).  ``chain``
        may be a torch CUDA tensor (used in place) or a NumPy array (uploaded).  Returns (tau [ndim], window [ndim]), or
        None when the series is too long for the device kernel (callers then use the host FFT estimator)."""
        on_host = 0 if _is_torch(chain) else 1
        if on_host:
            chain = np.ascontiguousarray(np.asarray(chain, dtype=np.float64))
            if chain.ndim == 2:
                chain = chain[:, :, None]
        else:
            import torch
            if not chain.is_cuda or chain.dtype != torch.float64 or chain.dim() != 3:
                raise ValueError("device chains must be float64 CUDA tensors of shape (n_t, n_walkers, ndim)")
            chain = chain.contiguous()
            self._torch_stream(chain.device)
        n_t, W, d = chain.shape
        tau = np.empty(d)
        win = np.empty(d, dtype=np.int32)
        st = _lib.check(self._lib.apgp_integrated_time(self._h, _lib.ptr(chain), int(n_t), int(W), int(d), int(discard),
                                                       int(thin), float(c), on_host, _lib.ptr(tau), _lib.ptr(win)),
                        "apgp_integrated_time")
        if st == _lib.APGP_NEEDS_HOST:
            return None
        return tau, win

    # ------------------------------------------------------------------ diagnostics (tests)
    def _alpha(self):
        a = np.empty(self._x.shape[0])
        _lib.check(self._lib.apgp_get_alpha(self._h, _lib.ptr(a)), "apgp_get_alpha")
        return a

    def _linv(self):
        n = self._x.shape[0]
        a = np.empty((n, n))
        _lib.check(self._lib.apgp_get_linv(self._h, _lib.ptr(a)), "apgp_get_linv")
        return a

    def _chol(self):
        n = self._x.shape[0]
        a = np.empty((n, n))
        _lib.check(self._lib.apgp_get_chol(self._h, _lib.ptr(a)), "apgp_get_chol")
        return a
