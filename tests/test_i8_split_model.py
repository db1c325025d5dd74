"""NumPy restatement of the int8 variance engine's arithmetic (predict_i8.cu): the digit split of the kernel panel E
and of A L^{-1}, the per-level integer accumulation, the truncation to levels p + r <= 7 and the int64 / FP64
combine (tests/i8_model.py).  Digit products are summed in float64, which is exact here (every partial sum stays below
2^53).  The model's own pieces are checked here without a GPU: the byte layouts round-trip, and the emulated fma is
correctly rounded; tests/test_gpu_i8_exact.py compares the kernel with the model bit for bit."""
import random
from fractions import Fraction

import numpy as np
import pytest

from i8_model import (B_STAGE, DIG, BN, b_digits, b_rowscale, e_digits, e_value, fma, i8_levels, i8_product,
                      i8_variance, linv_decode, linv_encode, linv_i8_bytes, panel_decode, panel_encode)


def _problem(N=512, d=5, Q=96, seed=0):
    from conftest import synthetic_gp_problem
    X, y, logM, _ = synthetic_gp_problem(N, d, seed=seed)
    w = np.sqrt(0.5 * np.exp(-logM))
    K = np.exp(-(((X[:, None, :] - X[None, :, :]) * w) ** 2).sum(-1)) + np.exp(-12.0) * np.eye(N)
    L = np.linalg.cholesky(K)
    Linv = np.linalg.solve(L, np.eye(N))
    Linv = np.tril(Linv)
    rng = np.random.default_rng(seed + 1)
    Xq = rng.uniform(-5, 5, size=(Q, d))
    Xq[:6] = X[:6]                                          # var ~ noise: the cancellation case
    Xq[6:12] = X[6:12] + 1e-3
    E = np.exp(-(((Xq[:, None, :] - X[None, :, :]) * w) ** 2).sum(-1))
    return E, Linv


def test_digit_ranges_and_int32_bound():
    E, B = _problem()
    _, e, bd, acc = i8_product(E, B)
    assert e.min() >= 0 and e[1:].max() <= 255 and e[0].max() <= 128
    assert np.abs(bd[0]).max() <= 127 and bd[1:].min() >= -128 and bd[1:].max() <= 127
    assert np.abs(acc).max() < 2 ** 31
    # worst case over N <= 8192: 7 digit pairs per level, |e| <= 255, |b| <= 128
    assert 7 * 8192 * 255 * 128 < 2 ** 31


def test_variance_error_not_above_fp64_gemm():
    E, B = _problem()
    ld = np.longdouble
    Wt = E.astype(ld) @ B.astype(ld).T
    var_t = 1.0 - (Wt * Wt).sum(axis=1)
    W64 = E @ B.T
    var64 = 1.0 - np.sum(W64 * W64, axis=1)
    W8, *_ = i8_product(E, B)
    var8 = 1.0 - np.sum(W8 * W8, axis=1)
    err64 = float(np.abs(var64 - var_t).max())
    err8 = float(np.abs(var8 - var_t).max())
    assert err8 <= err64, (err8, err64)
    assert float(np.abs(W8 - Wt).max()) <= float(np.abs(W64 - Wt).max())


# ---------------------------------------------------------------------------------------------------- layouts
@pytest.mark.parametrize("npad", [64, 192, 1024])
def test_panel_layout_round_trip(npad):
    rng = np.random.default_rng(npad)
    e = rng.integers(0, 256, size=(DIG, 128, npad)).astype(np.uint8)
    buf = panel_encode(e)
    assert buf.size == 128 * DIG * npad
    assert np.array_equal(panel_decode(buf, npad), e)
    # one digit by hand: plane p, query m, column j
    p, m, j = 5, 77, npad - 3
    cb, kc, k = j // 64, (j % 64) // 16, j % 16
    c = [cc for cc in range(16) if cc // 4 + 4 * (cc % 4) == k][0]
    assert buf[cb * 57344 + p * 8192 + kc * 2048 + (m // 8) * 128 + (m % 8) * 16 + c] == e[p, m, j]
    assert np.array_equal(panel_encode(panel_decode(buf, npad)), buf)


@pytest.mark.parametrize("npad", [64, 192, 640])
def test_linv_layout_round_trip(npad):
    rng = np.random.default_rng(npad + 1)
    D = rng.integers(-128, 128, size=(DIG, npad, npad)).astype(np.int8)
    blk = np.arange(npad) // BN
    D[:, blk[:, None] < blk[None, :]] = 0                      # only the block lower triangle is stored
    buf = linv_encode(D)
    assert buf.size == linv_i8_bytes(npad)
    assert np.array_equal(linv_decode(buf, npad), D)
    r, i, j = 3, npad - 5, npad // 2 + 1
    ib, kb, ng, row = i // 64, j // 64, (i // 8) % 8, i % 8
    kc, k = (j % 64) // 16, j % 16
    c = [cc for cc in range(16) if cc // 4 + 4 * (cc % 4) == k][0]
    off = (ib * (ib + 1) // 2 + kb) * B_STAGE + kc * 7168 + r * 1024 + ng * 128 + row * 16 + c
    assert buf.view(np.int8)[off] == D[r, i, j]
    assert np.array_equal(linv_encode(linv_decode(buf, npad)), buf)


def test_digit_split_reconstructs():
    E, B = _problem(N=128, Q=32)
    e = e_digits(E)
    assert np.array_equal(e_value(e), np.floor(np.ldexp(E.astype(np.longdouble), 55) + 0.5).astype(np.int64))
    bd, ex = b_digits(B)
    X = np.zeros(B.shape, dtype=np.int64)
    for r in range(DIG):
        X = X * 256 + bd[r]
    assert np.array_equal(X, np.rint(np.ldexp(B, (55 - ex)[:, None])).astype(np.int64))
    assert np.abs(bd[0]).max() <= 127
    sc = b_rowscale(B)
    assert np.array_equal(sc, np.ldexp(1.0, ex - 38))


def _x_of(bd, i):
    return [sum(int(bd[r, i, k]) * 256 ** (DIG - 1 - r) for r in range(DIG)) for k in range(bd.shape[2])]


def test_b_digits_bump_and_ties():
    t = 2.0 ** -54                                             # the 2^(ex - 55) grid of a row with maximum 1
    B = np.zeros((6, 4))
    B[0, 0] = 127.0 / 128.0 * 2.0 ** 3                         # exactly at the threshold: no bump
    B[1, 0] = np.nextafter(127.0 / 128.0 * 2.0 ** 3, np.inf)   # just above it: bump
    B[2, :2] = [-4.0, 1.0]                                     # negative power-of-two maximum
    B[3] = [1.0, 2.5 * t, 3.5 * t, -2.5 * t]                   # half way on the grid: ties to even
    B[4, 0] = 5e-320                                           # subnormal maximum
    bd, ex = b_digits(B)
    assert list(ex) == [3, 4, 3, 1, -1060, 0]
    assert bd[0, 0, 0] == 127 and abs(int(bd[0, 1, 0])) <= 127 and bd[0, 2, 0] == -64
    assert _x_of(bd, 3) == [2 ** 54, 2, 4, -2]
    assert _x_of(bd, 4)[0] == 10120 * 2 ** 41                  # 5e-320 = 10120 * 2^-1074, exactly on the grid
    assert not bd[:, 5].any()
    assert np.array_equal(b_rowscale(B), np.array([2.0 ** -35, 2.0 ** -34, 2.0 ** -35, 2.0 ** -37, 2.0 ** -1098, 0.0]))


# ---------------------------------------------------------------------------------------------------- exact fma
def _fma_exact(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def _check_fma(a, b, c):
    got = fma(np.array(a), np.array(b), np.array(c))
    want = np.array([_fma_exact(x, y, z) for x, y, z in zip(a, b, c)])
    assert np.array_equal(got.view(np.int64), want.view(np.int64)) or np.array_equal(got, want), \
        [(x, y, z, g, w) for x, y, z, g, w in zip(a, b, c, got, want) if g != w][:5]


def test_fma_emulation_random():
    rng = np.random.default_rng(7)
    n = 20000
    a = rng.standard_normal(n) * np.exp2(rng.integers(-60, 60, n))
    b = rng.standard_normal(n) * np.exp2(rng.integers(-60, 60, n))
    c = rng.standard_normal(n) * np.exp2(rng.integers(-120, 120, n))
    _check_fma(a, b, c)
    w = np.abs(rng.standard_normal(n)) * 1e-3                  # the epilogue's case: fma(w, w, ss), ss >= 0
    _check_fma(w, w, np.abs(rng.standard_normal(n)) * 1e-6)


def test_fma_emulation_adversarial():
    rnd = random.Random(11)
    a, b, c = [], [], []
    for _ in range(4000):
        # products whose low half decides the rounding of a sum: c cancels the high part of a*b to within a few ulps,
        # or sits half an ulp of the product's exact value away (ties), or is tiny against it (sticky bits)
        x = rnd.getrandbits(53) | (1 << 52)
        y = rnd.getrandbits(53) | (1 << 52)
        ea, eb = rnd.randint(-40, 40), rnd.randint(-40, 40)
        A, Bv = float(x) * 2.0 ** (ea - 52), float(y) * 2.0 ** (eb - 52)
        p = Fraction(A) * Fraction(Bv)
        kind = rnd.randrange(5)
        if kind == 0:
            C = -float(p)                                      # exact cancellation of the rounded product
        elif kind == 1:
            C = -float(p) + rnd.choice([-1, 1]) * np.spacing(float(p)) * rnd.choice([0.5, 1, 2, 3])
        elif kind == 2:
            P = float(p)                                       # a*b + c = P + ulp(P)/2 (exactly, when c is a double)
            C = float(Fraction(P) - p + Fraction(float(np.spacing(P))) / 2)
        elif kind == 3:
            C = float(p) * 2.0 ** -rnd.randint(53, 120) * rnd.choice([-1, 1])
        else:
            C = rnd.choice([0.0, -0.0, 1.0, -1.0]) * float(p)
        if rnd.random() < 0.5:
            A = -A
        a.append(A); b.append(Bv); c.append(C)
    _check_fma(a, b, c)
    # zero, exact products, tiny products (the Fraction fall-back), half-way ties
    _check_fma([0.0, 3.0, 1e-300, 1.0 + 2.0 ** -52, 1.0 + 2.0 ** -52, 2.0 ** 995],
               [5.0, 7.0, 1e-300, 1.0 - 2.0 ** -53, 1.0 + 2.0 ** -52, 0.75],
               [1.0, -21.0, 1e-310, -1.0, -1.0, -1.0])


# ---------------------------------------------------------------------------------------------------- epilogue model
def test_i8_variance_matches_scalar_replay():
    """i8_variance (vectorised) against the epilogue written out per element with exact fma."""
    E, B = _problem(N=100, Q=12)
    npad = 128
    Bp = np.zeros((npad, npad)); Bp[:100, :100] = B * 3.0
    Ep = np.zeros((12, npad)); Ep[:, :100] = E
    e = e_digits(Ep)
    bd, _ = b_digits(Bp)
    lev = i8_levels(e, bd)
    sc = b_rowscale(Bp)
    var = i8_variance(lev, sc, 3.0)
    for q in range(12):
        tot = 0.0
        for ib in range(npad // 64):
            halves = []
            for h in range(2):
                ss = 0.0
                for j in range(ib * 64 + 32 * h, ib * 64 + 32 * h + 32):
                    L = [int(lev[s, q, j]) for s in range(8)]
                    hi = ((L[0] * 256 + L[1]) * 256 + L[2]) * 256 + L[3]
                    lo = ((L[4] * 256 + L[5]) * 256 + L[6]) * 256 + L[7]
                    w = float(Fraction(float(hi)) + Fraction(float(lo)) / 2 ** 32) * sc[j]
                    ss = _fma_exact(w, w, ss)
                halves.append(ss)
            tot += halves[0] + halves[1]
        assert var[q] == 3.0 - tot
    # and the engine's W from the levels is the model's W
    W8, *_ = i8_product(Ep, Bp)
    assert np.all(np.isfinite(W8))
