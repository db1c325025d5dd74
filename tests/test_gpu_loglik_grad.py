"""Batched log-likelihood gradients beyond the one-CTA class: loglik_grad_group_kernel, one thread-block cluster per
parameter vector and one launch for the batch (apgp_loglik_batch path 4).  Checked against the oracle's
grad_log_likelihood, against the value kernels' log-likelihood bit for bit, for bits that do not depend on the cluster
size, the row's place in the batch or the run, and end to end through optimizeGP's gradient methods."""
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
    return gp, X, y


def _params(gp, R, seed):
    rng = np.random.default_rng(seed)
    P = gp.get_parameter_vector()[None, :] + 0.7 * rng.standard_normal((R, len(gp)))
    P[0, -1] = np.nan                                             # not finite
    if R > 2:
        P[1, 1] = np.inf
        P[2, 1:] = -30.0                                          # very short length scales (and a tiny amplitude)
    return P


def _path(gp):
    from approxposterior_b200 import _lib
    p = C.c_int(-1)
    _lib.check(_lib.load().apgp_debug_last_loglik_path(gp._h, C.byref(p)), "apgp_debug_last_loglik_path")
    return p.value


def _oracle(X, d, amp, mean):
    from oracle import GPOracle
    orc = GPOracle(d, np.full(d, 4.0), amp=amp, mean=mean, white_noise=-12.0)
    orc.compute(X)
    return orc


def _check_against(ll, g, ll_ref, g_ref):
    fin = np.isfinite(ll_ref)
    assert np.array_equal(np.isfinite(ll), fin)
    assert np.all(ll[~fin] == -np.inf) and np.all(g[~fin] == 0.0)
    np.testing.assert_allclose(ll[fin], ll_ref[fin], rtol=1e-9)
    for r in np.flatnonzero(fin):
        np.testing.assert_allclose(g[r], g_ref[r], rtol=1e-7, atol=1e-8 * np.max(np.abs(g_ref[r])))


@pytest.mark.parametrize("N", [240, 300, 512, 1024, 2048])          # above the one-CTA class for every d
@pytest.mark.parametrize("d", [2, 10])
@pytest.mark.parametrize("amp", [None, 1.5])
def test_gradients_match_the_oracle(N, d, amp):
    gp, X, y = _gp(N, d, amp=amp, seed=N + d)
    P = _params(gp, 9, seed=N)
    ll, g = gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 4
    orc = _oracle(X, d, amp, gp.mean)
    ll_ref, g_ref = np.full(len(P), -np.inf), np.zeros_like(P)
    for r in range(len(P)):
        if np.all(np.isfinite(P[r])):
            orc.set_parameter_vector(P[r])
            ll_ref[r] = orc.log_likelihood(y, quiet=True)
            g_ref[r] = orc.grad_log_likelihood(y, quiet=True) if np.isfinite(ll_ref[r]) else 0.0
    assert ll[0] == -np.inf and ll[1] == -np.inf and np.isfinite(ll[2])
    assert np.sum(np.isfinite(ll_ref)) >= 5
    _check_against(ll, g, ll_ref, g_ref)


@pytest.mark.parametrize("N", [240, 512])
@pytest.mark.parametrize("C_", [1, 2, 4, 8, 16])
def test_log_likelihood_is_the_value_kernels_bits(N, C_, monkeypatch):
    gp, X, y = _gp(N, 2, amp=1.5, seed=N)
    monkeypatch.setenv("APGP_NLL_GROUP", "1")
    monkeypatch.setenv("APGP_CHOL_CLUSTER", str(C_))
    P = _params(gp, 6, seed=C_)
    ll_g, _ = gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 4
    ll_v = gp.log_likelihood_batch(P, y)
    assert _path(gp) == 2
    _, f, _ = gp.minimize_nll(P, y, evaluate_only=True, default_prior=False)
    assert np.array_equal(ll_g, ll_v) and np.array_equal(ll_g, -f)
    assert np.sum(np.isfinite(ll_g)) >= 3


@pytest.mark.parametrize("N", [300, 1024])
def test_gradient_bits_do_not_depend_on_cluster_size_batch_position_or_run(N, monkeypatch):
    gp, X, y = _gp(N, 3, amp=2.0, seed=7)
    rows = _params(gp, 5, seed=11)
    rng = np.random.default_rng(12)
    big = gp.get_parameter_vector()[None, :] + 0.5 * rng.standard_normal((64, len(gp)))
    at = [3, 17, 40, 41, 63]
    big[at] = rows
    ref = None
    for C_ in (1, 2, 4, 8, 16):
        monkeypatch.setenv("APGP_CHOL_CLUSTER", str(C_))
        for _ in range(2):
            ll, g = gp.log_likelihood_batch(rows, y, return_grad=True)
            assert _path(gp) == 4
            llb, gb = gp.log_likelihood_batch(big, y, return_grad=True)
            assert _path(gp) == 4
            if ref is None:
                ref = (ll, g)
                assert np.sum(np.isfinite(ll)) >= 3 and np.any(g != 0.0)
            assert np.array_equal(ll, ref[0]) and np.array_equal(g, ref[1]), C_
            assert np.array_equal(llb[at], ref[0]) and np.array_equal(gb[at], ref[1]), C_


@pytest.mark.parametrize("N", [90, 200])
def test_forced_cluster_kernel_agrees_with_the_small_kernel(N, monkeypatch):
    gp, X, y = _gp(N, 3, amp=2.0, seed=N)
    P = _params(gp, 7, seed=3)
    ll_s, g_s = gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 1
    monkeypatch.setenv("APGP_LOGLIK_PATH", "group_grad")
    ll, g = gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 4
    assert np.sum(np.isfinite(ll_s)) >= 4
    _check_against(ll, g, ll_s, g_s)
    gp.log_likelihood_batch(P, y)                                 # value-only under group_grad: the cluster value kernel
    assert _path(gp) == 2


def test_not_positive_definite_gives_minus_inf_and_zero_gradients():
    gp, X, y = _gp(300, 2, seed=1, white_noise=-80.0, dup=True)
    P = _params(gp, 4, seed=2)
    ll, g = gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 4
    assert np.all(ll == -np.inf) and np.all(g == 0.0)


def test_one_launch_per_chunk():
    from approxposterior_b200 import _lib
    gp, X, y = _gp(512, 10, amp=1.0, seed=5)
    P = _params(gp, 64, seed=5)
    lib = _lib.load()
    gp.log_likelihood_batch(P, y, return_grad=True)
    n0 = lib.apgp_launch_count(gp._h)
    gp.log_likelihood_batch(P, y, return_grad=True)
    assert _path(gp) == 4
    assert lib.apgp_launch_count(gp._h) - n0 == 1


def _fit(gp, y, method, monkeypatch, forced=None):
    from approxposterior_b200 import gpUtils
    paths = []
    inner = gp.log_likelihood_batch

    def recording(P, yy, return_grad=False):
        out = inner(P, yy, return_grad=return_grad)
        if return_grad:
            paths.append(_path(gp))
        return out

    monkeypatch.setattr(gp, "log_likelihood_batch", recording)
    if forced:
        monkeypatch.setenv("APGP_LOGLIK_PATH", forced)
    else:
        monkeypatch.delenv("APGP_LOGLIK_PATH", raising=False)
    gp.set_parameter_vector(gp._start)
    np.random.seed(21)
    gpUtils.optimizeGP(gp, None, y, nGPRestarts=8, method=method)
    monkeypatch.delenv("APGP_LOGLIK_PATH", raising=False)
    monkeypatch.setattr(gp, "log_likelihood_batch", inner)
    return gp.get_parameter_vector().copy(), float(gp.log_likelihood(y)), paths


@pytest.mark.parametrize("method", ["l-bfgs-b", "bfgs"])
def test_optimize_gp_gradient_methods_end_to_end(method, monkeypatch):
    gp, X, y = _gp(300, 3, amp=1.0, seed=30)
    gp._start = gp.get_parameter_vector().copy()
    p1, ll1, paths = _fit(gp, y, method, monkeypatch)
    assert paths and all(p == 4 for p in paths), paths
    p1b, ll1b, _ = _fit(gp, y, method, monkeypatch)
    assert np.array_equal(p1, p1b) and ll1 == ll1b                   # deterministic
    p2, ll2, paths2 = _fit(gp, y, method, monkeypatch, forced="group")
    assert paths2 and all(p == 2 for p in paths2)                    # the value kernel ran, gradients per vector
    p2b, ll2b, _ = _fit(gp, y, method, monkeypatch, forced="group")
    assert np.array_equal(p2, p2b) and ll2 == ll2b
    assert abs(ll1 - ll2) <= 1e-6 * abs(ll2), (ll1, ll2)
    # the starts optimizeGP draws (np.random, one randn per kernel parameter per restart)
    np.random.seed(21)
    x0 = np.array([[np.median(y)] + [np.random.randn() for _ in range(len(gp) - 1)] for _ in range(8)])
    ll0 = gp.log_likelihood_batch(x0, y)
    assert ll1 > np.max(ll0[np.isfinite(ll0)])
