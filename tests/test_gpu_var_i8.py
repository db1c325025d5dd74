"""The int8 tensor-core variance engine (predict_i8.cu) against the FP64 DMMA kernel on the same factorisation: the
mean must be bit-identical (phase 1 is shared arithmetic), the variance must agree to the FP64 product's rounding,
and against extended-precision truth the int8 split must be as accurate as the DMMA product."""
import numpy as np
import pytest

from conftest import extended_truth, synthetic_gp_problem

pytestmark = pytest.mark.gpu


def _gp(N, d, amp=None):
    from approxposterior_b200 import GP, kernels
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + d)
    kern = kernels.ExpSquaredKernel(np.exp(logM), ndim=d)
    if amp is not None:
        kern = amp * kern
    gp = GP(kernel=kern, fit_mean=True, mean=float(np.median(y)), white_noise=-12.0)
    gp.compute(X, y=y)
    return gp, X, y, logM


def _queries(X, Q, d, seed):
    import torch
    rng = np.random.default_rng(seed)
    q = rng.uniform(-5.5, 5.5, size=(Q, d))
    q[: min(12, Q) : 2] = X[: min(6, (Q + 1) // 2)]                 # on training points: var ~ 1e-6, cancellation
    q[1: min(12, Q) : 2] = X[: min(6, Q // 2)] + 1e-3
    return torch.as_tensor(q, device="cuda")


def _path(gp):
    """Kernel of the last variance call: 2 one-tile DMMA, 3 grouped DMMA, 4 grouped int8."""
    import ctypes
    from approxposterior_b200 import _lib
    p = ctypes.c_int()
    _lib.check(_lib.load().apgp_debug_last_var_path(gp._h, ctypes.byref(p)), "apgp_debug_last_var_path")
    return p.value


def _both(gp, q):
    import torch
    out = {}
    for eng in ("dmma", "i8"):
        gp.set_var_engine(eng)
        l0 = gp.launch_count
        r1 = gp._predict_raw(q, True, utility="bape", bounds=[(-5.0, 5.0)] * q.shape[1])
        assert gp.launch_count == l0 + 1                             # operands were packed with the factorisation
        assert _path(gp) == (4 if eng == "i8" else 3)                # the grouped kernel of that engine ran
        r2 = gp._predict_raw(q, True, utility="bape", bounds=[(-5.0, 5.0)] * q.shape[1])
        for a, b in zip(r1, r2):                                     # repeatable launch to launch
            assert torch.equal(a, b)
        out[eng] = r1
    gp.set_var_engine("i8")
    return out


@pytest.mark.parametrize("N,d,Q", [(1024, 5, 1000), (2048, 5, 3001), (2100, 20, 777), (8192, 5, 700)])
def test_i8_engine_matches_dmma(N, d, Q):
    import torch
    gp, X, y, _ = _gp(N, d)
    q = _queries(X, Q, d, seed=N)
    out = _both(gp, q)
    mu0, var0, u0 = out["dmma"]
    mu1, var1, u1 = out["i8"]
    assert torch.equal(mu0, mu1)
    assert float((var1 - var0).abs().max()) <= 1e-12          # as the grouped-vs-one-tile DMMA comparison
    fin = torch.isfinite(u0)
    assert torch.equal(fin, torch.isfinite(u1))


def test_i8_engine_large_amplitude():
    gp, X, y, _ = _gp(2048, 5, amp=5.7e4)
    q = _queries(X, 1500, 5, seed=3)
    out = _both(gp, q)
    import torch
    mu0, var0, _ = out["dmma"]
    mu1, var1, _ = out["i8"]
    assert torch.equal(mu0, mu1)
    assert float((var1 - var0).abs().max()) <= 5.7e4 * 1e-12


@pytest.mark.parametrize("N,d", [(1024, 2), (2100, 20)])
def test_i8_engine_error_against_extended_truth(N, d):
    gp, X, y, logM = _gp(N, d)
    Xq = np.random.default_rng(1).uniform(-5, 5, size=(777, d))
    _, var_t = extended_truth(X, y, logM, Xq, mean=float(np.median(y)), nvar=64)
    errs = {}
    for eng in ("dmma", "i8"):
        gp.set_var_engine(eng)
        _, var = gp.predict(y, Xq, return_cov=False, return_var=True)
        assert _path(gp) == (4 if eng == "i8" else 3)
        errs[eng] = float(np.abs(var[:64] - var_t).max())
    gp.set_var_engine("i8")
    assert errs["i8"] <= 2.0 * errs["dmma"] + 1e-16, errs
