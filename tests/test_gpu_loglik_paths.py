"""The batched log-likelihood (apgp_loglik_batch) and the device optimisers' objective (apgp_minimize_nll) share one
evaluator per size class (csrc/loglik.cuh), so log_likelihood_batch(P) is -minimize_nll(P, evaluate_only=True,
default_prior=False) bit for bit -- in the one-CTA class, in the cluster class at every cluster size, and for rows that
are not finite or not positive definite.  Also: which kernel apgp_loglik_batch chooses, and the per-vector fallback
of batched gradients through APGP_NEEDS_HOST."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _gp(N, d, amp=None, seed=0, white_noise=-12.0, dup=False):
    from approxposterior_b200 import GP, kernels
    rng = np.random.default_rng(seed)
    X = rng.uniform(-5, 5, size=(N, d))
    if dup:
        X[N // 2] = X[3]                                          # a duplicate point: not positive definite without noise
    y = np.sin(X).sum(axis=1) + 0.1 * rng.standard_normal(N)
    k = kernels.ExpSquaredKernel(np.full(d, 4.0), ndim=d)
    if amp is not None:
        k = amp * k
    gp = GP(kernel=k, fit_mean=True, mean=float(np.median(y)), white_noise=white_noise)
    gp._x, gp._y = X, y
    gp._upload_training()
    return gp, y


def _params(gp, R, seed):
    rng = np.random.default_rng(seed)
    P = gp.get_parameter_vector()[None, :] + 0.7 * rng.standard_normal((R, len(gp)))
    P[0, -1] = np.nan                                             # not finite: -inf / +inf without a factorisation
    if R > 2:
        P[1, 1] = np.inf
        P[2, 1:] = -30.0                                          # tiny length scales and amplitude
    return P


def _path(gp):
    from approxposterior_b200 import _lib
    p = C.c_int(-1)
    _lib.check(_lib.load().apgp_debug_last_loglik_path(gp._h, C.byref(p)), "apgp_debug_last_loglik_path")
    return p.value


def _same_bits(gp, y, P):
    ll = gp.log_likelihood_batch(P, y)
    _, f, _ = gp.minimize_nll(P, y, evaluate_only=True, default_prior=False)
    assert np.array_equal(ll, -f), np.flatnonzero(ll != -f)
    assert ll[0] == -np.inf
    return ll


@pytest.mark.parametrize("N", [40, 90, 150, 224])
@pytest.mark.parametrize("amp", [None, 2.5])
def test_small_class_is_the_optimiser_objective(N, amp):
    gp, y = _gp(N, 3, amp=amp, seed=N)
    for R in (1, 7, 64):
        ll = _same_bits(gp, y, _params(gp, R, seed=R))
        assert _path(gp) == 1
    assert np.sum(np.isfinite(ll)) > 32


@pytest.mark.parametrize("N", [230, 512, 1024])
@pytest.mark.parametrize("C_", [1, 2, 4, 8, 16])
def test_group_class_is_the_optimiser_objective(N, C_, monkeypatch):
    gp, y = _gp(N, 2, amp=1.5, seed=N)
    monkeypatch.setenv("APGP_LOGLIK_PATH", "group")
    monkeypatch.setenv("APGP_NLL_GROUP", "1")
    monkeypatch.setenv("APGP_CHOL_CLUSTER", str(C_))
    ll = _same_bits(gp, y, _params(gp, 6, seed=C_))
    assert _path(gp) == 2
    assert np.sum(np.isfinite(ll)) >= 3


@pytest.mark.parametrize("N,group", [(60, False), (300, True)])
def test_not_positive_definite_is_the_same_on_both_sides(N, group, monkeypatch):
    if group:
        monkeypatch.setenv("APGP_NLL_GROUP", "1")
    gp, y = _gp(N, 2, seed=1, white_noise=-80.0, dup=True)
    ll = _same_bits(gp, y, _params(gp, 4, seed=2))
    assert np.all(ll == -np.inf)


def test_path_choice():
    # one restart per CTA while N(N+1)/2 + N(d+3) + d + 12 doubles fit 220 KB
    d = 2
    edge = max(n for n in range(1, 256) if (n * (n + 1) // 2 + n * (d + 3) + d + 12) * 8 <= 220 * 1024)
    for N, want in ((edge, 1), (edge + 1, 2)):
        gp, y = _gp(N, d)
        gp.log_likelihood_batch(_params(gp, 3, 0), y)
        assert _path(gp) == want, (N, want)
    # a handful of large matrices (Np >= 2048, R <= 8): the multi-launch tiled sequence
    for N, R, want in ((1985, 8, 3), (1985, 9, 2), (1984, 8, 2)):
        gp, y = _gp(N, d)
        ll = gp.log_likelihood_batch(_params(gp, R, 0), y)
        assert _path(gp) == want, (N, R, want)
        assert ll[0] == -np.inf and ll[1] == -np.inf


@pytest.mark.parametrize("N,forced,want", [(100, "small", 1), (100, "group", 2), (100, "tiled", 3), (300, "small", 2),
                                           (300, "group", 2), (300, "tiled", 3)])
def test_path_override(N, forced, want, monkeypatch):
    gp, y = _gp(N, 2)
    P = _params(gp, 5, 0)
    ref = gp.log_likelihood_batch(P, y)
    monkeypatch.setenv("APGP_LOGLIK_PATH", forced)
    ll = gp.log_likelihood_batch(P, y)
    assert _path(gp) == want
    assert np.array_equal(np.isfinite(ll), np.isfinite(ref))
    fin = np.isfinite(ref)
    np.testing.assert_allclose(ll[fin], ref[fin], rtol=1e-9)           # different algorithms: agree to rounding


def test_batched_gradients_beyond_the_small_kernel_fall_back_per_vector(monkeypatch):
    from approxposterior_b200 import _lib
    gp, y = _gp(100, 2, amp=2.0)
    P = _params(gp, 5, 3)
    ll_small, g_small = gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 1
    monkeypatch.setenv("APGP_LOGLIK_PATH", "group")
    ll = np.empty(5)
    grad = np.empty_like(P)
    st = _lib.load().apgp_loglik_batch(gp._h, _lib.ptr(P), 5, P.shape[1], 1, gp.white_noise, _lib.ptr(ll), _lib.ptr(grad))
    assert st == _lib.APGP_NEEDS_HOST
    ll_f, g_f = gp.log_likelihood_batch(P, y, return_grad=True)          # one factorisation per vector
    assert np.array_equal(np.isfinite(ll_f), np.isfinite(ll_small))
    fin = np.isfinite(ll_small)
    np.testing.assert_allclose(ll_f[fin], ll_small[fin], rtol=1e-10)
    np.testing.assert_allclose(g_f[fin], g_small[fin], rtol=1e-7, atol=1e-8 * np.max(np.abs(g_small[fin])))
    assert np.all(g_f[~fin] == 0.0) and np.all(g_small[~fin] == 0.0)
