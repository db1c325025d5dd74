"""NumPy model of the int8 variance engine (predict_i8.cu), shared by the CPU model tests and the GPU bit-exactness
tests: the digit split of the kernel panel E and of A L^{-1}, the byte layouts the kernel reads them in, the eight
exact level sums and the kernel's FP64 epilogue replayed operation for operation."""
from fractions import Fraction

import numpy as np

DIG, LEVELS = 7, 8
BM, BN = 128, 64                                   # queries per tile, rows of B per block-row (= k-stage width)
A_STAGE = DIG * BM * BN                            # panel bytes per 64-column block: 57344
B_STAGE = DIG * BN * BN                            # LinvI8 bytes per (block-row, k-stage) tile: 28672
# byte c of a 16-byte row segment holds k = c // 4 + 4 (c % 4) of its 16-wide k chunk (an involution)
KPERM = np.array([c // 4 + 4 * (c % 4) for c in range(16)])


def linv_i8_bytes(npad):
    nblk = npad // BN
    return nblk * (nblk + 1) // 2 * B_STAGE


# ---------------------------------------------------------------------------------------------------- digit split
def e_digits(E):
    """round(E * 2^55) (ties up) as 7 base-256 digits, most significant first; 0 <= E <= 1."""
    Ei = np.floor(np.ldexp(E.astype(np.longdouble), 55) + np.longdouble(0.5)).astype(np.uint64)
    return np.stack([((Ei >> np.uint64(8 * (DIG - 1 - p))) & np.uint64(0xFF)).astype(np.int64) for p in range(DIG)])


def e_value(e):
    """The integer round(E * 2^55) that 7 digits (most significant first) stand for."""
    v = np.zeros(e.shape[1:], dtype=np.int64)
    for p in range(DIG):
        v = v * 256 + e[p].astype(np.int64)
    return v


def b_exponents(B):
    """Per row the exponent ex with |B| <= 127/128 2^ex (ilogb(max) + 1, bumped once), 0 for an all-zero row."""
    mx = np.abs(B).max(axis=1)
    ex = np.frexp(mx)[1].astype(np.int64)          # mx = f 2^ex, f in [0.5, 1): ex = ilogb(mx) + 1; frexp(0) = 0
    ex = np.where(mx > np.ldexp(127.0 / 128.0, ex), ex + 1, ex)
    return ex, mx


def b_digits(B):
    """Per row a power-of-two exponent ex (|B| <= 127/128 2^ex) and 7 balanced signed digits of round(B 2^(55-ex))
    (ties to even, as llrint)."""
    ex, _ = b_exponents(B)
    X = np.rint(np.ldexp(B, (55 - ex)[:, None])).astype(np.int64)
    digs = [None] * DIG
    for r in range(DIG - 1, 0, -1):
        dg = ((X + 128) & 0xFF) - 128
        X = (X - dg) >> 8
        digs[r] = dg
    digs[0] = X
    return np.stack(digs), ex


def b_rowscale(B):
    """The kernel's row scale 2^(ex - 38) (the combine's 2^(ex - 14) and the hi/lo split's 2^-24), 0 for zero rows."""
    ex, mx = b_exponents(B)
    return np.where(mx > 0, np.ldexp(1.0, ex - 38), 0.0)


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


# ---------------------------------------------------------------------------------------------------- byte layouts
def panel_decode(buf, npad):
    """Digit panel of one 128-query tile -> [7 planes][128 queries][npad] uint8.  Byte
    cb*57344 + p*8192 + kc*2048 + (m//8)*128 + (m%8)*16 + c holds plane p of E[m, cb*64 + kc*16 + KPERM[c]]."""
    nblk = npad // BN
    a = np.asarray(buf, dtype=np.uint8)[: nblk * A_STAGE].reshape(nblk, DIG, 4, 16, 8, 16)   # cb p kc mg row c
    a = a.transpose(1, 3, 4, 0, 2, 5)[..., KPERM]                                          # p mg row cb kc k
    return np.ascontiguousarray(a.reshape(DIG, BM, npad))


def panel_encode(e):
    """Inverse of panel_decode: [7][128][npad] digits -> bytes."""
    npad = e.shape[2]
    a = np.asarray(e, dtype=np.uint8).reshape(DIG, 16, 8, npad // BN, 4, 16)[..., KPERM]
    return np.ascontiguousarray(a.transpose(3, 0, 4, 1, 2, 5)).ravel()


def linv_decode(buf, npad):
    """LinvI8 -> [7 planes][npad rows][npad columns] int8, zero above the stored block triangle.  Byte
    (ib(ib+1)/2 + kb)*28672 + kc*7168 + r*1024 + ng*128 + row*16 + c holds signed digit r of row ib*64 + ng*8 + row,
    column kb*64 + kc*16 + KPERM[c]."""
    nblk = npad // BN
    buf = np.asarray(buf, dtype=np.uint8).view(np.int8)
    D = np.zeros((DIG, npad, npad), dtype=np.int8)
    for ib in range(nblk):
        off = ib * (ib + 1) // 2 * B_STAGE
        t = buf[off: off + (ib + 1) * B_STAGE].reshape(ib + 1, 4, DIG, 8, 8, 16)          # kb kc r ng row c
        t = t.transpose(2, 3, 4, 0, 1, 5)[..., KPERM]                                    # r ng row kb kc k
        D[:, ib * BN:(ib + 1) * BN, :(ib + 1) * BN] = t.reshape(DIG, BN, (ib + 1) * BN)
    return D


def linv_encode(D):
    """Inverse of linv_decode on the block lower triangle: [7][npad][npad] signed digits -> bytes."""
    npad = D.shape[1]
    nblk = npad // BN
    D = np.asarray(D).astype(np.int8)
    out = np.zeros(linv_i8_bytes(npad), dtype=np.int8)
    for ib in range(nblk):
        off = ib * (ib + 1) // 2 * B_STAGE
        t = D[:, ib * BN:(ib + 1) * BN, :(ib + 1) * BN].reshape(DIG, 8, 8, ib + 1, 4, 16)[..., KPERM]
        out[off: off + (ib + 1) * B_STAGE] = t.transpose(3, 4, 0, 1, 2, 5).ravel()
    return out.view(np.uint8)


# ---------------------------------------------------------------------------------------------------- level sums
def i8_levels(e, b):
    """The eight level sums acc_s = sum_{p+r=s} e_p b_r^T of [7][Q][npad] panel digits and [7][npad][npad] B digits,
    as int64 [8][Q][npad].  Each is an integer below 7 npad 255 128 < 2^31, so float64 products are exact in any
    summation order.  e and b may be NumPy arrays or torch tensors; with a CUDA tensor the products run there."""
    try:
        import torch
    except ImportError:                                            # pragma: no cover
        torch = None
    if torch is not None and (isinstance(e, torch.Tensor) or isinstance(b, torch.Tensor)):
        dev = b.device if isinstance(b, torch.Tensor) else e.device
        et = torch.as_tensor(np.asarray(e) if not isinstance(e, torch.Tensor) else e, device=dev).to(torch.float64)
        acc = torch.zeros((LEVELS, et.shape[1], et.shape[2]), dtype=torch.float64, device=dev)
        for r in range(DIG):
            br = (b[r] if isinstance(b, torch.Tensor) else torch.as_tensor(np.asarray(b[r]), device=dev))
            br = br.to(torch.float64)
            for p in range(min(DIG, LEVELS - r)):
                acc[p + r] += et[p] @ br.T
        return acc.cpu().numpy().astype(np.int64)
    ef = np.asarray(e, dtype=np.float64)
    acc = np.zeros((LEVELS, ef.shape[1], ef.shape[2]))
    for r in range(DIG):
        br = np.asarray(b[r], dtype=np.float64)
        for p in range(min(DIG, LEVELS - r)):
            acc[p + r] += ef[p] @ br.T
    return acc.astype(np.int64)


# ---------------------------------------------------------------------------------------------------- exact fma
_SPLIT = 134217729.0                                   # 2^27 + 1 (Veltkamp)


def _two_sum(a, b):
    s = a + b
    bp = s - a
    ap = s - bp
    return s, (a - ap) + (b - bp)


def _two_prod(a, b):
    p = a * b
    ca, cb = _SPLIT * a, _SPLIT * b
    ah, bh = ca - (ca - a), cb - (cb - b)
    al, bl = a - ah, b - bh
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _fma_fraction(a, b, c):
    if not (np.isfinite(a) and np.isfinite(b) and np.isfinite(c)):
        return a * b + c
    v = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    if v == 0:                                          # exact zero: the sign of a*b + c in round-to-nearest
        return float(a) * float(b) + float(c)
    return float(v)                                     # int / int true division is correctly rounded


def fma(a, b, c):
    """Correctly rounded a*b + c (round to nearest even) on float64 arrays: Boldo and Melquiond's emulation
    (exact product, TwoSum, the low parts added with rounding to odd, one final rounding).  Elements outside its
    proven range (products near underflow, operands near overflow, non-finite values) are done with Fraction."""
    a, b, c = np.broadcast_arrays(np.asarray(a, np.float64), np.asarray(b, np.float64), np.asarray(c, np.float64))
    with np.errstate(all="ignore"):
        uh, ul = _two_prod(a, b)
        th, tl = _two_sum(c, uh)
        z, err = _two_sum(tl, ul)
        even = (z.view(np.int64) & 1) == 0
        z = np.where((err != 0) & even, np.nextafter(z, np.where(err > 0, np.inf, -np.inf)), z)   # round to odd
        out = th + z
        big = 2.0 ** 990
        risky = ~(np.isfinite(a) & np.isfinite(b) & np.isfinite(c)) | (np.abs(a) > big) | (np.abs(b) > big) | \
            (np.abs(c) > big) | ((a != 0) & (b != 0) & (np.abs(a * b) < 2.0 ** -900)) | (np.abs(out) > big)
    out = np.array(out, dtype=np.float64)
    if risky.any():
        for idx in zip(*np.nonzero(risky)):
            out[idx] = _fma_fraction(a[idx], b[idx], c[idx])
    return out


# ---------------------------------------------------------------------------------------------------- epilogue
def i8_variance(levels, rowscale, amp):
    """Replay of the kernel's FP64 epilogue and finaliser on [8][Q][npad] level sums:
    w = (f64(hi) + f64(lo) 2^-32) sc_i; per (query, block-row, 32-column half) ss = fma(w, w, ss) over the half's
    columns in ascending order from 0; a block-row's part is ss_half0 + ss_half1; tot adds the parts in block-row
    order; var = amp - tot."""
    L = np.asarray(levels, dtype=np.int64)
    hi = ((L[0] * 256 + L[1]) * 256 + L[2]) * 256 + L[3]
    lo = ((L[4] * 256 + L[5]) * 256 + L[6]) * 256 + L[7]
    w = (hi.astype(np.float64) + lo.astype(np.float64) * 2.0 ** -32) * np.asarray(rowscale, np.float64)[None, :]
    Q, npad = w.shape
    w = w.reshape(Q, npad // BN, 2, BN // 2)
    ss = np.zeros((Q, npad // BN, 2))
    for c in range(BN // 2):
        ss = fma(w[..., c], w[..., c], ss)
    part = ss[..., 0] + ss[..., 1]
    tot = np.zeros(Q)
    for ib in range(npad // BN):
        tot = tot + part[:, ib]
    return amp - tot
