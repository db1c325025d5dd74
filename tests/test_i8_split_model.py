"""NumPy restatement of the int8 variance engine's arithmetic (predict_i8.cu): the digit split of the kernel panel E
and of A L^{-1}, the per-level integer accumulation, the truncation to levels p + r <= 7 and the int64 / FP64
combine.  Digit products are summed in float64, which is exact here (every partial sum stays below 2^53)."""
import numpy as np


DIG, LEVELS = 7, 8


def e_digits(E):
    """round(E * 2^55) (ties up) as 7 base-256 digits, most significant first; 0 <= E <= 1."""
    Ei = np.floor(np.ldexp(E.astype(np.longdouble), 55) + np.longdouble(0.5)).astype(np.uint64)
    return np.stack([((Ei >> np.uint64(8 * (DIG - 1 - p))) & np.uint64(0xFF)).astype(np.int64) for p in range(DIG)])


def b_digits(B):
    """Per row a power-of-two exponent ex (|B| <= 127/128 2^ex) and 7 balanced signed digits of round(B 2^(55-ex))."""
    mx = np.abs(B).max(axis=1)
    ex = np.where(mx > 0, np.floor(np.log2(np.where(mx > 0, mx, 1.0))).astype(np.int64) + 1, 0)
    ex = np.where(mx > np.ldexp(127.0 / 128.0, ex), ex + 1, ex)
    X = np.rint(np.ldexp(B, (55 - ex)[:, None])).astype(np.int64)
    digs = [None] * DIG
    for r in range(DIG - 1, 0, -1):
        dg = ((X + 128) & 0xFF) - 128
        X = (X - dg) >> 8
        digs[r] = dg
    digs[0] = X
    return np.stack(digs), ex


def i8_product(E, B):
    """W = E B^T as the int8 engine computes it."""
    e, b = e_digits(E), b_digits(B)
    bd, ex = b
    acc = np.zeros((LEVELS, E.shape[0], B.shape[0]))
    for p in range(DIG):
        for r in range(DIG):
            if p + r < LEVELS:
                acc[p + r] += e[p].astype(np.float64) @ bd[r].astype(np.float64).T
    acc = acc.astype(np.int64)
    hi = ((acc[0] * 256 + acc[1]) * 256 + acc[2]) * 256 + acc[3]
    lo = ((acc[4] * 256 + acc[5]) * 256 + acc[6]) * 256 + acc[7]
    return (hi.astype(np.float64) + lo.astype(np.float64) * 2.0 ** -32) * np.ldexp(1.0, ex - 38)[None, :], e, bd, acc


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
