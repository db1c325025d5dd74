"""The int8 variance engine (predict_i8.cu) bit for bit against its integer model (tests/i8_model.py).

The kernel computes exact integer level sums and then a fixed sequence of FP64 operations, so its variance can be
checked exactly: the operands it packed are decoded and compared with the model's digit split of amp * L^-1, the
panel it built is decoded and run through the model's level sums and FP64 epilogue, and the variance must equal the
model's bit for bit.  Because the sums are exact, a query's mean, variance and utility must not depend on its position
in the batch or on the group size either.  apgp_debug_last_var_path shows which kernel ran each call."""
import ctypes as C

import numpy as np
import pytest

from conftest import extended_truth, synthetic_gp_problem
from i8_model import (DIG, b_digits, b_rowscale, e_digits, e_value, fma, i8_levels, i8_variance, linv_decode,
                      linv_i8_bytes, panel_decode)

pytestmark = pytest.mark.gpu

PATH_FEW, PATH_ONE_TILE, PATH_GROUPED_DMMA, PATH_I8 = 1, 2, 3, 4
BOUNDS5 = (-5.0, 5.0)


# ---------------------------------------------------------------------------------------------------- helpers
def _lib():
    from approxposterior_b200 import _lib
    return _lib


def _gp(N, d, amp=None, engine=None, seed=None):
    from approxposterior_b200 import GP, kernels
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=N + d if seed is None else seed)
    kern = kernels.ExpSquaredKernel(np.exp(logM), ndim=d)
    if amp is not None:
        kern = amp * kern
    gp = GP(kernel=kern, fit_mean=True, mean=float(np.median(y)), white_noise=-12.0)
    gp.set_predict_few(False)
    if engine is not None:
        gp.set_var_engine(engine)
    gp.compute(X, y=y)
    return gp, X, y, logM


def _path(gp):
    L = _lib()
    p = C.c_int()
    L.check(L.load().apgp_debug_last_var_path(gp._h, C.byref(p)), "apgp_debug_last_var_path")
    return p.value


def _npad(gp):
    L = _lib()
    n = C.c_int()
    L.check(L.load().apgp_debug_i8_operands(gp._h, None, None, None, C.byref(n)), "apgp_debug_i8_operands")
    return n.value


def _operands(gp):
    L = _lib()
    npad = _npad(gp)
    lb = np.empty(linv_i8_bytes(npad), dtype=np.uint8)
    sc = np.empty(npad)
    L.check(L.load().apgp_debug_i8_operands(gp._h, L.ptr(lb), L.ptr(sc), None, None), "apgp_debug_i8_operands")
    return npad, lb, sc


def _panel(gp, npad):
    L = _lib()
    pn = np.empty(128 * DIG * npad, dtype=np.uint8)
    L.check(L.load().apgp_debug_i8_operands(gp._h, None, None, L.ptr(pn), None), "apgp_debug_i8_operands")
    return panel_decode(pn, npad)


def _check_pack(gp):
    """Decoded LinvI8 and i8scale equal the model's split of amp * L^-1 (rows of the padding included); returns the
    operands for the bit-exact checks, the digits on the GPU."""
    import torch
    npad, lb, sc = _operands(gp)
    N = gp._x.shape[0]
    amp = float(gp.kernel.amplitude)
    B = np.zeros((npad, npad))
    B[:N, :N] = amp * gp._linv()
    D = linv_decode(lb, npad)
    assert np.abs(D[0].astype(np.int64)).max() <= 127
    for r0 in range(0, npad, 512):                       # in row chunks: the int64 digits of N = 8192 are 3.7 GB
        bd, _ = b_digits(B[r0:r0 + 512])
        assert np.array_equal(D[:, r0:r0 + 512].astype(np.int64), bd), "LinvI8 digits, rows %d.." % r0
    assert np.array_equal(sc, b_rowscale(B)), "i8scale"
    return npad, torch.as_tensor(D, device="cuda"), sc


def _probe_queries(X, Q, d, seed):
    """On training points (E = 1 exactly: top digit 128), at 1e-3 offsets, far away (E = 0) and random."""
    rng = np.random.default_rng(seed)
    q = rng.uniform(-5.0, 5.0, size=(Q, d))
    n = X.shape[0]
    q[0::4] = X[rng.integers(0, n, size=len(q[0::4]))]
    q[1::4] = X[rng.integers(0, n, size=len(q[1::4]))] + 1e-3
    q[2::4] = 1e3 + rng.uniform(0.0, 1.0, size=(len(q[2::4]), d))
    return q


def _predict(gp, q, utility="bape", bounds=True):
    import torch
    if not isinstance(q, torch.Tensor):
        q = torch.as_tensor(q, device="cuda")
    d = q.shape[1]
    return gp._predict_raw(q, True, utility=utility, bounds=[BOUNDS5] * d if bounds else None)


def _bits(a):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _kernel_E(gp, q):
    """E[q, j] exactly as phase 1 evaluates it: scaled coordinates x_j qs and q qs (qs = sqrt(exp(-log M) / 2), the
    host's libm), s = fma(x - q, x - q, s) over the dimensions in order, then the kernel's own exp(-s)."""
    import math
    L = _lib()
    qsc = np.array([math.sqrt(0.5 * math.exp(-v)) for v in np.asarray(gp.kernel.log_M, dtype=np.float64)])
    Xs, Qs = gp._x * qsc, q * qsc
    s = np.zeros((q.shape[0], Xs.shape[0]))
    for i in range(Xs.shape[1]):
        dd = Xs[None, :, i] - Qs[:, None, i]
        s = fma(dd, dd, s)
    s = np.ascontiguousarray(s.ravel())
    E = np.empty_like(s)
    L.check(L.load().apgp_debug_exp_neg(gp._h, L.ptr(s), s.size, L.ptr(E)), "apgp_debug_exp_neg")
    return E.reshape(q.shape[0], Xs.shape[0])


def _check_exact(gp, ops, q):
    """One call of <= 128 queries: path 4; the panel holds round(E 2^55) (ties up) of the kernel's E, digit by digit;
    the variance is the model's, bit for bit.  Returns (mu, var, util) and the number of ties in the rounding."""
    npad, Ddev, sc = ops
    Q, N = q.shape[0], gp._x.shape[0]
    mu, var, util = _predict(gp, q)
    assert _path(gp) == PATH_I8
    e = _panel(gp, npad)[:, :Q]
    assert int(e[0].max()) <= 128
    ev = e_value(e)
    assert ev.min() >= 0 and ev.max() <= 2 ** 55
    E = _kernel_E(gp, q)
    bad = np.nonzero((e[:, :, :N].astype(np.int64) != e_digits(E)).any(axis=0))
    assert bad[0].size == 0, "panel != round(E 2^55) at %d entries, e.g. (q, j) = (%d, %d): E = %r" % (
        bad[0].size, bad[0][0], bad[1][0], E[bad[0][0], bad[1][0]])
    ties = int(np.count_nonzero(np.ldexp(E, 56) % 2 == 1))
    lev = i8_levels(e, Ddev)
    var_m = i8_variance(lev, sc, float(gp.kernel.amplitude))
    got = var.cpu().numpy()
    bad = np.nonzero(_bits(got) != _bits(var_m))[0]
    assert bad.size == 0, "var != model at %d queries, e.g. q=%d: %r vs %r" % (
        bad.size, bad[0], got[bad[0]], var_m[bad[0]])
    return (mu, var, util), ties


# ---------------------------------------------------------------------------------------------------- (a) pack
SHAPES = [(961, 1, None), (1025, 3, 1e-3), (2048, 5, None), (2100, 20, 5.7e4), (8192, 2, None), (1025, 27, None)]


@pytest.mark.parametrize("N,d,amp", SHAPES)
def test_i8_operands_and_variance_bit_exact(N, d, amp):
    """(a) the packed operands are the model's split; (b) 1, 77 and 128 queries at G = 2 and automatic G give the
    model's variance bit for bit."""
    gp, X, y, logM = _gp(N, d, amp)
    ops = _check_pack(gp)
    ties = 0
    for Q in (1, 77, 128):
        q = _probe_queries(X, Q, d, seed=Q + N)
        for G in (2, -1):
            gp.set_group(G)
            ties += _check_exact(gp, ops, q)[1]
    gp.set_group(-1)
    assert ties > 0                                      # the rounding of exact half-way values was exercised


def _pack_crafted(M, amp):
    from approxposterior_b200 import GP, kernels
    L = _lib()
    n = M.shape[0]
    npad = (n + 63) // 64 * 64
    gp = GP(kernel=kernels.ExpSquaredKernel(np.ones(1), ndim=1))
    out = np.empty(linv_i8_bytes(npad), dtype=np.uint8)
    rs = np.empty(npad)
    M = np.ascontiguousarray(M, dtype=np.float64)
    L.check(L.load().apgp_debug_pack_linv_i8(gp._h, L.ptr(M), n, float(amp), L.ptr(out), L.ptr(rs)),
            "apgp_debug_pack_linv_i8")
    return linv_decode(out, npad), rs, npad


def test_i8_pack_crafted_rows():
    """The row exponent at and just above the 127/128 bump threshold, powers of two, a negative maximum, a single
    entry, ties on the 2^(ex - 55) grid (llrint: to even), entries below the grid, a subnormal maximum, a zero row;
    the upper triangle (NaN here) must not be read."""
    n = 100
    t = 2.0 ** -54                                       # the grid of a row whose maximum is in [1/2, 127/128 * 2)
    M = np.triu(np.full((n, n), np.nan), 1)
    rng = np.random.default_rng(5)
    for i in range(n):
        M[i, :i + 1] = rng.standard_normal(i + 1) * 2.0 ** rng.integers(-30, 30)
    rows = {
        10: [127.0 / 128.0 * 8.0, 1.0],                  # exactly at the threshold: ex = 3, top digit 127
        11: [np.nextafter(127.0 / 128.0 * 8.0, np.inf), 1.0],   # just above: ex = 4
        12: [4.0, 2.0, 1.0, 0.5],                        # exact powers of two
        13: [-4.0, 1.0, -2.0 ** -20],                    # negative power-of-two maximum
        14: [-7.99, 3.0],                                # negative maximum, bumped
        15: [1.0, 2.5 * t, 3.5 * t, -2.5 * t, 0.5 * t, 1.5 * t, -0.5 * t],   # half way: 2, 4, -2, 0, 2, 0
        16: [1.0, 2.0 ** -60, -2.0 ** -57, 0.49 * t],    # below the grid: 0
        17: [5e-320, 1e-321, -3e-322],                   # subnormal maximum
        18: [0.0],                                       # zero row
    }
    for i, v in rows.items():
        M[i, :i + 1] = 0.0
        M[i, :len(v)] = v
    M[20, :21] = 0.0
    M[20, 20] = 3.3                                      # a single nonzero entry, on the diagonal
    for amp in (1.0, 3.0):
        D, rs, npad = _pack_crafted(M, amp)
        B = np.zeros((npad, npad))
        B[:n, :n] = amp * np.tril(np.nan_to_num(M, nan=0.0))
        bd, ex = b_digits(B)
        assert np.abs(D[0].astype(np.int64)).max() <= 127
        bad = np.nonzero((D.astype(np.int64) != bd).any(axis=(0, 2)))[0]
        assert bad.size == 0, "rows %s differ" % bad[:10]
        assert np.array_equal(rs, b_rowscale(B))
        if amp == 1.0:
            assert list(ex[10:19]) == [3, 4, 3, 3, 4, 1, 1, -1060, 0]
            assert D[0, 10, 0] == 127
            assert rs[18] == 0.0 and not D[:, 18].any() and not D[:, n:].any()


# ---------------------------------------------------------------------------------------------------- (c) invariance
def test_i8_results_do_not_depend_on_position_or_group_size():
    import torch
    N, d, amp = 2100, 20, 5.7e4
    gp, X, y, logM = _gp(N, d, amp)
    ops = _check_pack(gp)
    probes = _probe_queries(X, 128, d, seed=11)
    gp.set_group(2)
    ref = [r.clone() for r in _check_exact(gp, ops, probes)[0]]
    pt = torch.as_tensor(probes, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(3)
    nblk = _npad(gp) // 64
    groups = [2, 3, 5, 8, 16, -1, 64]                    # 148 % G: 0, 1 (a lone CTA), 3, 4, 4; 64 -> nblk // 2
    assert 2 * 16 <= nblk < 2 * 17
    for G in groups:
        gp.set_group(G)
        for Q, offsets in ((129, (0, 1)), (128 * 148 + 5, (0, 1, 127, 9000, 128 * 148 + 5 - 128)),
                           (70001, (0, 127, 35000, 70001 - 128))):
            filler = torch.rand((Q, d), generator=gen, device="cuda", dtype=torch.float64) * 10.0 - 5.0
            for o in offsets:
                q = filler.clone()
                q[o:o + 128] = pt
                out = _predict(gp, q)
                assert _path(gp) == PATH_I8, (G, Q, o)
                for name, a, r in zip(("mu", "var", "util"), out, ref):
                    assert torch.equal(a[o:o + 128], r), "%s differs: G=%d Q=%d offset=%d" % (name, G, Q, o)
        again = _predict(gp, q)
        for a, b in zip(out, again):
            assert torch.equal(a, b)
    gp.set_group(-1)
    host = gp._predict_raw(q.cpu().numpy(), True, utility="bape", bounds=[BOUNDS5] * d)
    assert _path(gp) == PATH_I8
    for a, r in zip(host, ref):
        assert np.array_equal(_bits(a[o:o + 128]), _bits(r))


# ---------------------------------------------------------------------------------------------------- (d) selection
@pytest.mark.parametrize("N,d,paths", [(960, 5, (PATH_ONE_TILE, PATH_GROUPED_DMMA)), (961, 5, (PATH_I8,)),
                                       (1025, 27, (PATH_I8,)), (1025, 28, (PATH_ONE_TILE,))])
@pytest.mark.parametrize("amp", [1e-3, 1.0, 1e3])
def test_i8_engine_selection_and_accuracy(N, d, paths, amp):
    """Which kernel runs at the edges of the engine's range, and its variance error against extended-precision truth
    is no worse than twice the DMMA engine's.  d = 28 fits the int8 kernel, but the group planner turns grouping off
    there (the DMMA kernel's shared-memory bound), so it runs the one-tile DMMA kernel."""
    gp, X, y, logM = _gp(N, d, amp)
    Xq = np.random.default_rng(N + d).uniform(-5, 5, size=(300, d))
    Xq[:8] = X[:8]
    _, var_t = extended_truth(X, y, logM, Xq, amp=amp, mean=float(np.median(y)), nvar=32)
    errs = {}
    for eng in ("dmma", "i8"):
        gp.set_var_engine(eng)
        _, var, _ = gp._predict_raw(Xq, True)
        if eng == "i8":
            assert _path(gp) in paths
        else:
            assert _path(gp) in (PATH_ONE_TILE, PATH_GROUPED_DMMA)
        errs[eng] = float(np.abs(var[:32] - var_t).max())
    assert errs["i8"] <= 2.0 * errs["dmma"] + 1e-16 * amp, errs


def test_i8_engine_selection_large_n():
    """N = 8192 (128 block-rows) is the largest the int8 kernel takes: the path and the DMMA agreement there;
    N = 8193 (129 block-rows) runs the one-tile DMMA kernel under either engine setting."""
    import torch
    for N, want in ((8192, PATH_I8), (8193, PATH_ONE_TILE)):
        gp, X, y, logM = _gp(N, 2)
        q = torch.as_tensor(_probe_queries(X, 700, 2, seed=N), device="cuda")
        res = {}
        for eng in ("dmma", "i8"):
            gp.set_var_engine(eng)
            res[eng] = _predict(gp, q)
            if eng == "i8":
                assert _path(gp) == want
        assert torch.equal(res["dmma"][0], res["i8"][0])
        assert float((res["dmma"][1] - res["i8"][1]).abs().max()) <= 1e-12
        del gp


# ---------------------------------------------------------------------------------------------------- (e) lifecycle
def test_i8_operands_follow_the_factorisation():
    """The lazy pack after a switch from dmma, append_point, a new amplitude and an i8 -> dmma -> i8 round trip (plan
    cache) must each leave the operands of the current factorisation and a bit-exact variance."""
    L = _lib()
    N, d = 1025, 3
    gp, X, y, logM = _gp(N, d, amp=2.0, engine="dmma")
    q = _probe_queries(X, 77, d, seed=1)
    _predict(gp, q)
    assert _path(gp) in (PATH_ONE_TILE, PATH_GROUPED_DMMA)
    with pytest.raises(L.ApgpError):
        _npad(gp)                                        # factored under dmma: nothing packed yet
    gp.set_var_engine("i8")
    _predict(gp, q)                                      # packs lazily
    _check_exact(gp, _check_pack(gp), q)

    rng = np.random.default_rng(2)
    for _ in range(3):
        assert gp.append_point(rng.uniform(-5, 5, size=d), float(rng.standard_normal()))
    assert gp._x.shape[0] == N + 3
    _check_exact(gp, _check_pack(gp), q)

    names = gp.get_parameter_names()
    p = gp.get_parameter_vector()
    p[names.index("kernel:k1:log_constant")] += np.log(7.0)
    gp.set_parameter_vector(p)
    gp.recompute()
    assert abs(float(gp.kernel.amplitude) - 14.0) < 1e-12
    _check_exact(gp, _check_pack(gp), q)

    gp.set_var_engine("dmma")
    _predict(gp, q)
    assert _path(gp) in (PATH_ONE_TILE, PATH_GROUPED_DMMA)
    gp.set_var_engine("i8")
    _check_exact(gp, _check_pack(gp), q)


# ---------------------------------------------------------------------------------------------------- (f) non-finite
@pytest.mark.parametrize("bounds", [True, False])
def test_i8_non_finite_queries(bounds):
    """NaN, +inf and -inf coordinates: the int8 engine gives the DMMA engine's finiteness (and NaN) pattern in mu,
    var and util, and the other rows of the batch are unchanged.  A NaN query has no digits in the panel; its
    variance must still be NaN, as the DMMA product's is."""
    import torch
    N, d = 2048, 5
    gp, X, y, logM = _gp(N, d)
    clean = torch.as_tensor(_probe_queries(X, 300, d, seed=4), device="cuda")
    q = clean.clone()
    bad = [5, 130, 131, 250]
    q[5, 2], q[130, 0], q[131, 4], q[250, 1] = float("nan"), float("inf"), float("-inf"), float("nan")
    q[250, 3] = float("inf")
    out = {}
    for eng in ("dmma", "i8"):
        gp.set_var_engine(eng)
        out[eng] = _predict(gp, q, bounds=bounds)
    assert _path(gp) == PATH_I8
    for a, b in zip(out["dmma"], out["i8"]):
        assert torch.equal(torch.isfinite(a), torch.isfinite(b))
        assert torch.equal(torch.isnan(a), torch.isnan(b))
    assert torch.isnan(out["i8"][1][[5, 250]]).all()
    ref = _predict(gp, clean, bounds=bounds)
    keep = torch.ones(300, dtype=torch.bool, device="cuda")
    keep[bad] = False
    for a, r in zip(out["i8"], ref):
        assert torch.equal(a[keep], r[keep])
    assert torch.equal(out["dmma"][0][keep], out["i8"][0][keep])
