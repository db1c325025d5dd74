// Factor path for sm_100a: covariance build, batched blocked Cholesky, triangular inverse,
// log-likelihood and its gradient.  Everything works on 64x64 tiles multiplied on the FP64
// tensor pipe (DMMA.8x8x4) and is batched over a leading "restart" axis so that the R
// hyper-parameter vectors of gpUtils.optimizeGP's restarts factor side by side.
//
// Replaces (reference call sites):
//   george.GP.compute / recompute            gpUtils.py:178,244,254  approx.py:717
//   george.GP.log_likelihood(y, quiet=True)  gpUtils.py:78,247
//   george.GP.grad_log_likelihood            gpUtils.py:110
// george's BasicSolver does K = kernel(X) + (yerr^2 + exp(white_noise)) I, scipy cholesky,
// log|K| = 2 sum log L_ii, ll = -1/2 (N log 2pi + log|K|) - 1/2 r^T K^{-1} r.
//
// Padding: N is padded to Np (multiple of 64) with an identity block, so L and L^{-1} pad with
// the identity and the rhs with zeros; nothing downstream needs edge handling.
#include "apgp_internal.h"
#include "loglik.cuh"
#include <math.h>
#include <stdlib.h>
#include <stdio.h>

namespace apgp {
namespace {

constexpr int T = 64;          // tile edge
constexpr int LDS_ = 68;       // padded smem leading dimension: conflict-free DMMA fragment loads
constexpr int GT = 128;        // threads per tile group: 4 warps, each a 32x32 sub-tile
constexpr size_t TILE_SMEM = (size_t)2 * T * LDS_ * sizeof(double);

// ---- tile movers ------------------------------------------------------------------------
// dst[r][c] (smem, ld 68) = src[r*ld + c]          (row-major 64x64 block)
__device__ __forceinline__ void load_tile_n(double* dst, const double* __restrict__ src, int ld, int tid) {
#pragma unroll 4
  for (int e = tid; e < T * (T / 2); e += GT) {
    int r = e >> 5, c2 = (e & 31) * 2;
    double2 v = *reinterpret_cast<const double2*>(src + (size_t)r * ld + c2);
    dst[r * LDS_ + c2] = v.x; dst[r * LDS_ + c2 + 1] = v.y;
  }
}
// dst[r][c] = src[c*ld + r]                        (transpose while staging)
__device__ __forceinline__ void load_tile_t(double* dst, const double* __restrict__ src, int ld, int tid) {
#pragma unroll 4
  for (int e = tid; e < T * (T / 2); e += GT) {
    int c = e >> 5, r2 = (e & 31) * 2;
    double2 v = *reinterpret_cast<const double2*>(src + (size_t)c * ld + r2);
    dst[r2 * LDS_ + c] = v.x; dst[(r2 + 1) * LDS_ + c] = v.y;
  }
}

struct Acc { double v[4][4][2]; };

__device__ __forceinline__ void acc_zero(Acc& a) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { a.v[i][j][0] = 0.0; a.v[i][j][1] = 0.0; }
}

// acc += As(64x64, [m][k]) * Bs(64x64, [n][k])^T ; warp (wm,wn) owns rows wm*32.., cols wn*32..
__device__ __forceinline__ void tile_mma(const double* As, const double* Bs, Acc& acc, int wm, int wn, int lane) {
  const double* ap = As + (wm * 32 + (lane >> 2)) * LDS_ + (lane & 3);
  const double* bp = Bs + (wn * 32 + (lane >> 2)) * LDS_ + (lane & 3);
#pragma unroll 4
  for (int k4 = 0; k4 < T / 4; ++k4) {
    double a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { a[i] = ap[i * 8 * LDS_ + k4 * 4]; b[i] = bp[i * 8 * LDS_ + k4 * 4]; }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) dmma884(acc.v[i][j][0], acc.v[i][j][1], a[i], b[j]);
  }
}

// C[r*ld + c] = beta*C + alpha*acc     (64x64 block)
__device__ __forceinline__ void store_acc(double* __restrict__ C, int ld, const Acc& acc, double alpha, double beta,
                                          int wm, int wn, int lane) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int r = wm * 32 + i * 8 + (lane >> 2), c = wn * 32 + j * 8 + 2 * (lane & 3);
      double2* p = reinterpret_cast<double2*>(C + (size_t)r * ld + c);
      double2 o;
      if (beta != 0.0) { o = *p; o.x = beta * o.x + alpha * acc.v[i][j][0]; o.y = beta * o.y + alpha * acc.v[i][j][1]; }
      else { o.x = alpha * acc.v[i][j][0]; o.y = alpha * acc.v[i][j][1]; }
      *p = o;
    }
}

// ---- covariance build -------------------------------------------------------------------
// hyper row: [mean, amp, noise_var, invM_0 .. invM_{d-1}]
__global__ void build_K_kernel(const double* __restrict__ X, const double* __restrict__ y, int N, int d, int Np,
                               const double* __restrict__ hyper, double* __restrict__ K, double* __restrict__ r,
                               double* __restrict__ logdet, int* __restrict__ info) {
  const int rr = blockIdx.y;
  const double* h = hyper + (size_t)rr * (3 + d);
  const int nb = Np / T;
  // lower-triangular tile index -> (bi, bj)
  int t = blockIdx.x;
  int bi = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
  while (bi * (bi + 1) / 2 > t) --bi;
  int bj = t - bi * (bi + 1) / 2;
  (void)nb;
  double* Kr = K + (size_t)rr * Np * Np;
  const double amp = h[1], noise = h[2];
  for (int e = threadIdx.x; e < T * T; e += blockDim.x) {
    int i = bi * T + (e >> 6), j = bj * T + (e & 63);
    double v;
    if (i < N && j < N) {
      double s = 0.0;
      for (int c = 0; c < d; ++c) {
        double df = X[(size_t)i * d + c] - X[(size_t)j * d + c];
        s += df * df * h[3 + c];
      }
      v = amp * exp(-0.5 * s);
      if (i == j) v += noise;
    } else {
      v = (i == j) ? 1.0 : 0.0;
    }
    Kr[(size_t)i * Np + j] = v;
  }
  if (bj == 0) {
    for (int e = threadIdx.x; e < T; e += blockDim.x) {
      int i = bi * T + e;
      r[(size_t)rr * Np + i] = (i < N) ? (y[i] - h[0]) : 0.0;
    }
  }
  if (t == 0 && threadIdx.x == 0) { logdet[rr] = 0.0; info[rr] = 0; }
}

// ---- step k, diagonal block: D = chol(A_kk), Dinv = D^{-1}, z_k = Dinv r_k, logdet += 2 sum log D_ii
// One CTA per restart.  The 64x64 block is factored by the blocked in-shared-memory routine of chol_small.cuh with
// 65 right-hand sides riding along: r_k (-> z_k) and the 64 unit vectors, whose solutions are the columns of D^{-1}.
// (The first version -- one thread per row, three barriers per column, then a 64-step substitution per column of the
// inverse -- took 127 us per block and was the whole cost of a tiled factorisation: 0.14 ms per block column at any
// batch size up to 8.)
constexpr int DIAG_THREADS = 256;
constexpr int DIAG_LDR = T + 1;                 // odd row stride of the right-hand-side block: conflict-free row threads
constexpr size_t DIAG_SMEM = (size_t)(T * (T + 1) / 2 + (T + 1) * DIAG_LDR + T) * sizeof(double);
__global__ void __launch_bounds__(DIAG_THREADS, 1) chol_diag_kernel(FactorBatch fb, int k) {
  extern __shared__ __align__(16) double dsm[];
  double* S = dsm;                              // packed lower triangle of the block
  double* R = S + T * (T + 1) / 2;              // [1 + T][DIAG_LDR]: row 0 = r_k, row 1 + c = e_c
  double* dg = R + (T + 1) * DIAG_LDR;          // [T] pivots
  __shared__ int bad;
  __shared__ double red[DIAG_THREADS / 32];
  const int rr = blockIdx.x, tid = threadIdx.x;
  const int Np = fb.Np;
  double* A = fb.K + (size_t)rr * Np * Np + (size_t)k * T * Np + k * T;
  double* rk = fb.r + (size_t)rr * Np + k * T;
  if (tid == 0) bad = 0;
  for (int e = tid; e < T * T; e += DIAG_THREADS) {
    const int i = e >> 6, j = e & 63;
    if (j <= i) S[i * (i + 1) / 2 + j] = A[(size_t)i * Np + j];
    R[(1 + i) * DIAG_LDR + j] = (i == j) ? 1.0 : 0.0;
  }
  if (tid < T) R[tid] = rk[tid];
  __syncthreads();
  chol_packed_blocked<DIAG_THREADS, false>(S, R, dg, T, &bad, true, T + 1, DIAG_LDR);
  double* Dg = fb.Dinv + ((size_t)rr * (Np / T) + k) * T * T;
  for (int e = tid; e < T * T; e += DIAG_THREADS) {
    const int i = e >> 6, j = e & 63;
    A[(size_t)i * Np + j] = (j <= i) ? S[i * (i + 1) / 2 + j] : 0.0;
    Dg[e] = (j <= i) ? R[(1 + j) * DIAG_LDR + i] : 0.0;       // D^{-1}[i][j] = (solution for e_j)[i]
  }
  if (tid < T) rk[tid] = R[tid];
  double lg = (tid < T) ? log(dg[tid]) : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lg += __shfl_xor_sync(0xffffffffu, lg, o);
  if ((tid & 31) == 0) red[tid >> 5] = lg;
  __syncthreads();
  if (tid == 0) {
    fb.logdet[rr] += 2.0 * (red[0] + red[1]);
    if (bad) atomicCAS(&fb.info[rr], 0, k * T + bad);        // 1-based index of the first failing pivot
  }
}

// ---- step k, panel: L_ik = A_ik * Dinv_k^T ; r_i -= L_ik z_k        grid (nb-k-1, R)
__global__ void __launch_bounds__(GT) chol_panel_kernel(FactorBatch fb, int k) {
  extern __shared__ __align__(16) double sm[];
  double* As = sm; double* Bs = sm + T * LDS_;
  const int rr = blockIdx.y, bi = k + 1 + blockIdx.x, tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31, wm = warp >> 1, wn = warp & 1;
  const int Np = fb.Np;
  double* Kr = fb.K + (size_t)rr * Np * Np;
  double* Aik = Kr + (size_t)bi * T * Np + k * T;
  const double* Dg = fb.Dinv + ((size_t)rr * (Np / T) + k) * T * T;
  load_tile_n(As, Aik, Np, tid);
  load_tile_n(Bs, Dg, T, tid);
  __syncthreads();
  Acc acc; acc_zero(acc);
  tile_mma(As, Bs, acc, wm, wn, lane);
  __syncthreads();
  store_acc(Aik, Np, acc, 1.0, 0.0, wm, wn, lane);
  // stash L_ik in smem (reuse As) for the rhs update
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int r = wm * 32 + i * 8 + (lane >> 2), c = wn * 32 + j * 8 + 2 * (lane & 3);
      As[r * LDS_ + c] = acc.v[i][j][0]; As[r * LDS_ + c + 1] = acc.v[i][j][1];
    }
  double* zk = fb.r + (size_t)rr * Np + k * T;
  if (tid < T) Bs[tid] = zk[tid];
  __syncthreads();
  if (tid < T) {
    double s = 0.0;
    for (int c = 0; c < T; ++c) s += As[tid * LDS_ + c] * Bs[c];
    fb.r[(size_t)rr * Np + bi * T + tid] -= s;
  }
}

// ---- step k, trailing update: A_ij -= L_ik L_jk^T  for i >= j > k     grid (pairs, R)
__global__ void __launch_bounds__(GT) chol_update_kernel(FactorBatch fb, int k) {
  extern __shared__ __align__(16) double sm[];
  double* As = sm; double* Bs = sm + T * LDS_;
  const int rr = blockIdx.y, tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31, wm = warp >> 1, wn = warp & 1;
  int t = blockIdx.x;
  int a = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((a + 1) * (a + 2) / 2 <= t) ++a;
  while (a * (a + 1) / 2 > t) --a;
  const int b = t - a * (a + 1) / 2;
  const int bi = k + 1 + a, bj = k + 1 + b;
  const int Np = fb.Np;
  double* Kr = fb.K + (size_t)rr * Np * Np;
  load_tile_n(As, Kr + (size_t)bi * T * Np + k * T, Np, tid);
  load_tile_n(Bs, Kr + (size_t)bj * T * Np + k * T, Np, tid);
  __syncthreads();
  Acc acc; acc_zero(acc);
  tile_mma(As, Bs, acc, wm, wn, lane);
  store_acc(Kr + (size_t)bi * T * Np + bj * T, Np, acc, -1.0, 1.0, wm, wn, lane);
}

// ---- generic 64-tile GEMM used by the triangular inverse and K^{-1} -----------------------
// C(tile mi,nj) = alpha * sum_{kt in [k0,k1)} opA(mi,kt) * opB(kt,nj)
struct GemmDesc {
  const double* A; int lda; int ta;   // ta=0: A[(m)*lda + k]   ta=1: A[(k)*lda + m]
  const double* B; int ldb; int tb;   // tb=0: B[(k)*ldb + n]   tb=1: B[(n)*ldb + k]
  double* C; int ldc;
  double alpha;
  int mt, nt, kt;                     // tiles
  int tri;                            // 0: full k range; 1: k in [nj, kt) (B lower-tri, NN); 2: k in [0, mi] (A lower-tri);
                                      // 3: k in [max(mi,nj), kt) (A^T A of lower-tri), only mi>=nj computed
  long strideA, strideB, strideC;     // batch strides (blockIdx.y)
};
__global__ void __launch_bounds__(GT) gemm_tile_kernel(GemmDesc g) {
  extern __shared__ __align__(16) double sm[];
  double* As = sm; double* Bs = sm + T * LDS_;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wm = warp >> 1, wn = warp & 1;
  const int mi = blockIdx.x / g.nt, nj = blockIdx.x % g.nt;
  const double* A = g.A + (size_t)blockIdx.y * g.strideA;
  const double* B = g.B + (size_t)blockIdx.y * g.strideB;
  double* C = g.C + (size_t)blockIdx.y * g.strideC;
  int k0 = 0, k1 = g.kt;
  if (g.tri == 1) k0 = nj;
  else if (g.tri == 2) k1 = min(g.kt, mi + 1);
  else if (g.tri == 3) { if (mi < nj) return; k0 = mi; }
  Acc acc; acc_zero(acc);
  for (int kt = k0; kt < k1; ++kt) {
    if (g.ta) load_tile_t(As, A + (size_t)kt * T * g.lda + mi * T, g.lda, tid);
    else load_tile_n(As, A + (size_t)mi * T * g.lda + kt * T, g.lda, tid);
    if (g.tb) load_tile_n(Bs, B + (size_t)nj * T * g.ldb + kt * T, g.ldb, tid);
    else load_tile_t(Bs, B + (size_t)kt * T * g.ldb + nj * T, g.ldb, tid);
    __syncthreads();
    tile_mma(As, Bs, acc, wm, wn, lane);
    __syncthreads();
  }
  store_acc(C + (size_t)mi * T * g.ldc + nj * T, g.ldc, acc, g.alpha, 0.0, wm, wn, lane);
}

__global__ void init_linv_kernel(const double* __restrict__ Dinv, int Np, double* __restrict__ Linv) {
  // zero everything, then drop the inverted diagonal blocks in place
  const long total = (long)Np * Np;
  for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int i = (int)(idx / Np), j = (int)(idx - (long)i * Np);
    double v = 0.0;
    if ((i / T) == (j / T)) v = Dinv[((size_t)(i / T) * T + (i % T)) * T + (j % T)];
    Linv[idx] = v;
  }
}

// alpha[j] = sum_{i>=j} Linv[i][j] z[i]      grid Np/64, block 256 = 64 columns x 4 row groups
__global__ void __launch_bounds__(256) linvT_matvec_kernel(const double* __restrict__ Linv, int Np,
                                                           const double* __restrict__ z, double* __restrict__ alpha) {
  __shared__ double part[4][T];
  const int c = threadIdx.x & 63, g = threadIdx.x >> 6;
  const int j = blockIdx.x * T + c;
  double s = 0.0;
  for (int i = blockIdx.x * T + g; i < Np; i += 4) s += Linv[(size_t)i * Np + j] * z[i];
  part[g][c] = s;
  __syncthreads();
  if (g == 0) alpha[j] = (part[0][c] + part[1][c]) + (part[2][c] + part[3][c]);
}

// ---- one step of iterative refinement for alpha = K^{-1}(y - m) -------------------------------------------
// alpha comes out of the explicit inverse (alpha = L^{-T} L^{-1} r), whose forward error was measured at 3-12x the
// LAPACK oracle's on ill-conditioned problems (cond(K) ~ 1e6: profiles/r02_parity_errors_before_refinement.txt).
// One refinement step with the residual carried in double-double brings it to the oracle's level or below:
//   res = (y - m) - K alpha     (K rebuilt on the fly with the expression build_K_kernel uses; one warp per row)
//   alpha += L^{-T} (L^{-1} res)
__global__ void __launch_bounds__(256) alpha_residual_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                                             int N, int d, const double* __restrict__ h,
                                                             const double* __restrict__ alpha, double* __restrict__ res,
                                                             int Np) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= Np) return;
  if (i >= N) { if (lane == 0) res[i] = 0.0; return; }
  const double amp = h[1], noise = h[2];
  double hi = 0.0, lo = 0.0;
  for (int j = lane; j < N; j += 32) {
    double s = 0.0;
    for (int c = 0; c < d; ++c) {
      double df = X[(size_t)i * d + c] - X[(size_t)j * d + c];
      s += df * df * h[3 + c];
    }
    double v = amp * exp(-0.5 * s);
    if (i == j) v += noise;
    const double a = alpha[j];
    const double p = v * a, pe = fma(v, a, -p);                 // two-product
    const double t = hi + p, bb = t - hi;                        // two-sum
    lo += ((hi - (t - bb)) + (p - bb)) + pe;
    hi = t;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double h2 = __shfl_xor_sync(0xffffffffu, hi, o), l2 = __shfl_xor_sync(0xffffffffu, lo, o);
    const double t = hi + h2, bb = t - hi;
    lo += ((hi - (t - bb)) + (h2 - bb)) + l2;
    hi = t;
  }
  if (lane == 0) res[i] = ((y[i] - h[0]) - hi) - lo;
}
__global__ void axpy_kernel(int n, const double* __restrict__ x, double* __restrict__ y) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) y[i] += x[i];
}

__global__ void loglik_finish_kernel(FactorBatch fb, double* __restrict__ ll) {
  const int rr = blockIdx.x;
  __shared__ double red[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < fb.Np; i += blockDim.x) { double z = fb.r[(size_t)rr * fb.Np + i]; s += z * z; }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) {
    double v = -0.5 * red[0] - 0.5 * fb.logdet[rr] - 0.5 * fb.N * 1.8378770664093454836;  // log(2 pi)
    if (fb.info[rr] != 0 || !(v == v) || v == INFINITY || v == -INFINITY) v = -INFINITY;
    ll[rr] = v;
  }
}

// gradient reduction over the lower triangle of G = alpha alpha^T - K^{-1}:
//   g_c   = 1/2 sum_ab G_ab Kk_ab            (d/d log_constant, dK = K_kernel)
//   g_i   = 1/2 sum_ab G_ab Kk_ab * 1/2 D_i^2 / M_i
// out[0] = sum alpha ; out[1] = g_c ; out[2+i] = g_i       (host drops out[1] when !fit_amp)
__global__ void __launch_bounds__(256) grad_reduce_kernel(const double* __restrict__ X, int N, int d, int Np,
                                                          const double* __restrict__ Kinv,
                                                          const double* __restrict__ alpha,
                                                          const double* __restrict__ hyper, double* __restrict__ part) {
  // part: [ntiles][2 + d] per-tile partial sums (slot 0 = this tile's share of sum(alpha), tile 0 only); they are added
  // in tile order by grad_finish_kernel, so the gradient does not depend on the order the tiles happen to finish in
  // (the first version met in atomicAdds and differed in the last bits from run to run and from GPU to GPU)
  __shared__ double red[256];
  int t = blockIdx.x;
  double* out = part + (size_t)t * (2 + d);
  int bi = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
  while (bi * (bi + 1) / 2 > t) --bi;
  const int bj = t - bi * (bi + 1) / 2;
  const double amp = hyper[1];
  double accs[APGP_MAXD + 1];
  for (int c = 0; c <= d; ++c) accs[c] = 0.0;
  for (int e = threadIdx.x; e < T * T; e += 256) {
    int i = bi * T + (e >> 6), j = bj * T + (e & 63);
    if (i < N && j <= i) {
      double s = 0.0;
      double df2[APGP_MAXD];
      for (int c = 0; c < d; ++c) {
        double df = X[(size_t)i * d + c] - X[(size_t)j * d + c];
        df2[c] = 0.5 * df * df * hyper[3 + c];
        s += df2[c];
      }
      double kk = amp * exp(-s);
      double G = alpha[i] * alpha[j] - Kinv[(size_t)i * Np + j];
      double w = (i == j) ? 0.5 : 1.0;        // off-diagonal pairs appear twice in the full trace
      double gk = w * G * kk;
      accs[0] += gk;
      for (int c = 0; c < d; ++c) accs[1 + c] += gk * df2[c];
    }
  }
  for (int c = 0; c <= d; ++c) {
    red[threadIdx.x] = accs[c];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) out[1 + c] = red[0];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = 0.0;
  if (t == 0) {
    double s = 0.0;
    for (int i = threadIdx.x; i < N; i += 256) s += alpha[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) out[0] = red[0];
  }
}
__global__ void grad_finish_kernel(const double* __restrict__ part, int ntiles, int d, double* __restrict__ out) {
  const int c = threadIdx.x;
  if (c >= 2 + d) return;
  double s = 0.0;
  for (int t = 0; t < ntiles; ++t) s += part[(size_t)t * (2 + d) + c];
  out[c] = s;
}


// ---- one restart per CTA: the small evaluator of loglik.cuh (N <= ~224), one parameter vector of P [R][1 + fit_amp + d]
//      per CTA.  Replaces one gpUtils._nll evaluation (gpUtils.py:46-80) per CTA; a vector that is not finite gives -inf
//      without being factorised.
//      With grad_out != nullptr the CTA goes on to alpha = L^{-T} z, inverts L in place, forms K^{-1} pair by pair
//      and reduces  dl/dp = 1/2 tr[(alpha alpha^T - K^{-1}) dK/dp]  (george.GP.grad_log_likelihood, gpUtils.py:110):
//      grad_out[r] = [ sum(alpha), d/dlog_constant, d/dlog M_0 .. ]   (the host drops the amplitude slot if unused).
__global__ void __launch_bounds__(LL_NT, 1) loglik_small_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                                              int N, int d, const double* __restrict__ Pv, int fit_amp,
                                                              double noise, double* __restrict__ ll_out,
                                                              double* __restrict__ grad_out) {
  extern __shared__ __align__(16) double sm[];
  const SmallLL L = SmallLL::carve(sm, N, d);
  __shared__ double red[256];
  const int tid = threadIdx.x;
  const int P = 1 + fit_amp + d;
  const double* p = Pv + (size_t)blockIdx.x * P;
  if (!nll_row_finite(p, P)) { if (tid == 0) ll_out[blockIdx.x] = -INFINITY; return; }
  for (int e = tid; e < N * d; e += LL_NT) L.X[e] = X[e];
  for (int i = tid; i < N; i += LL_NT) L.y[i] = y[i];
  nll_hyp(p, d, fit_amp, noise, L.hyp);
  const double ll = loglik_small(L, N, d, grad_out != nullptr);      // L in K, z in r, diag(L) in col
  if (tid == 0) ll_out[blockIdx.x] = ll;
  double* K = L.K; double* r = L.r; double* col = L.col;
  const double* xs = L.X; const double* h = L.hyp;
  const double amp = h[1];
  if (grad_out == nullptr) return;
  double* g_out = grad_out + (size_t)blockIdx.x * (2 + d);
  __syncthreads();
  if (*L.bad) {                                       // quiet=True convention: zeros when the factorisation failed
    for (int c = tid; c < 2 + d; c += 256) g_out[c] = 0.0;
    return;
  }
  // ---- alpha = L^{-T} z (in r): back substitution, row j of L is contiguous
  for (int j = N - 1; j >= 0; --j) {
    const double* Lj = K + (size_t)j * (j + 1) / 2;
    const double aj = r[j] / Lj[j];
    __syncthreads();
    if (tid == 0) r[j] = aj;
    for (int i = tid; i < j; i += 256) r[i] -= Lj[i] * aj;
    __syncthreads();
  }
  // ---- L <- L^{-1} in place, column by column from the right:
  //      inv[j][j] = 1/L_jj ; inv[i][j] = -inv_jj * sum_{k=j+1..i} inv[i][k] L[k][j]   (i > j)
  for (int j = N - 1; j >= 0; --j) {
    const double ljj = K[(size_t)j * (j + 1) / 2 + j];
    for (int i = j + 1 + tid; i < N; i += 256) col[i] = K[(size_t)i * (i + 1) / 2 + j];
    __syncthreads();
    const double ijj = 1.0 / ljj;
    for (int i = j + 1 + tid; i < N; i += 256) {
      const double* Ii = K + (size_t)i * (i + 1) / 2;
      double s = 0.0;
      for (int k = j + 1; k <= i; ++k) s += Ii[k] * col[k];
      K[(size_t)i * (i + 1) / 2 + j] = -s * ijj;
    }
    if (tid == 0) K[(size_t)j * (j + 1) / 2 + j] = ijj;
    __syncthreads();
  }
  // ---- pairs (a >= b): K^{-1}_ab = sum_{c >= a} inv[c][a] inv[c][b], then the trace products
  double accs[APGP_MAXD + 1];
  for (int c = 0; c <= d; ++c) accs[c] = 0.0;
  const int npairs = N * (N + 1) / 2;
  for (int pidx = tid; pidx < npairs; pidx += 256) {
    int a = (int)((sqrt(8.0 * pidx + 1.0) - 1.0) * 0.5);
    while ((a + 1) * (a + 2) / 2 <= pidx) ++a;
    while (a * (a + 1) / 2 > pidx) --a;
    const int b = pidx - a * (a + 1) / 2;
    double kinv = 0.0;
    for (int cc = a; cc < N; ++cc) {
      const double* Ic = K + (size_t)cc * (cc + 1) / 2;
      kinv = fma(Ic[a], Ic[b], kinv);
    }
    double s = 0.0, df2[APGP_MAXD];
    for (int c = 0; c < d; ++c) {
      const double df = xs[a * d + c] - xs[b * d + c];
      df2[c] = 0.5 * df * df * h[3 + c];
      s += df2[c];
    }
    const double gk = ((a == b) ? 0.5 : 1.0) * (r[a] * r[b] - kinv) * amp * exp(-s);
    accs[0] += gk;
    for (int c = 0; c < d; ++c) accs[1 + c] += gk * df2[c];
  }
  for (int c = 0; c <= d; ++c) {
    red[tid] = accs[c];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
    if (tid == 0) g_out[1 + c] = red[0];
    __syncthreads();
  }
  double sa = 0.0;
  for (int i = tid; i < N; i += 256) sa += r[i];
  red[tid] = sa;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
  if (tid == 0) g_out[0] = red[0];
}


// ---- bordered (rank-1) append of one design point: O(N^2) instead of the O(N^3) refactor the reference
//      performs for every new point (approx.py:693-717).  With l = L^{-1} k(X, x_new):
//        L'    = [L 0; l^T lam]            lam^2 = kappa - l^T l
//        L'^-1 = [L^-1 0; -(l^T L^-1)/lam  1/lam]
//        z'    = [z; (r_new - l^T z)/lam]  alpha' = [alpha + w z_N; z_N/lam],  w = -(l^T L^-1)/lam
__global__ void append_kvec_kernel(const double* __restrict__ X, int N, int d, const double* __restrict__ xnew,
                                   const double* __restrict__ hyper, double* __restrict__ kvec) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  double s = 0.0;
  for (int c = 0; c < d; ++c) { const double df = X[(size_t)j * d + c] - xnew[c]; s += df * df * hyper[3 + c]; }
  kvec[j] = hyper[1] * exp(-0.5 * s);
}
// l_i = sum_{j<=i} Linv[i][j] k_j : one warp per row
__global__ void __launch_bounds__(256) append_linv_rows_kernel(const double* __restrict__ Linv, int Np, int N,
                                                               const double* __restrict__ kvec, double* __restrict__ l) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= N) return;
  double s = 0.0;
  for (int j = lane; j <= i; j += 32) s += Linv[(size_t)i * Np + j] * kvec[j];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) l[i] = s;
}
// single CTA: everything that is O(N).  u = l^T L^-1 (computed by linvT_matvec into `u`).
// scal: [0] logdet, [1] loglik (in/out).  status: 0 ok, 1 not positive definite.
__global__ void __launch_bounds__(256) append_finish_kernel(double* __restrict__ L, double* __restrict__ Linv, int Np, int N,
                                                            const double* __restrict__ l, const double* __restrict__ u,
                                                            double* __restrict__ z, double* __restrict__ alpha,
                                                            double kappa, double rnew, double* __restrict__ scal,
                                                            int* __restrict__ status) {
  __shared__ double red[256];
  __shared__ double sh[3];
  const int tid = threadIdx.x;
  double a = 0.0, b = 0.0, zz = 0.0;
  for (int i = tid; i < N; i += 256) { a += l[i] * l[i]; b += l[i] * z[i]; zz += z[i] * z[i]; }
  for (int k = 0; k < 3; ++k) {
    red[tid] = (k == 0) ? a : (k == 1 ? b : zz);
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
    if (tid == 0) sh[k] = red[0];
    __syncthreads();
  }
  const double lam2 = kappa - sh[0];
  if (!(lam2 > 0.0) || !(lam2 < INFINITY)) { if (tid == 0) *status = 1; return; }
  const double lam = sqrt(lam2), ilam = 1.0 / lam;
  const double zN = (rnew - sh[1]) * ilam;
  for (int j = tid; j < N; j += 256) {
    const double w = -u[j] * ilam;
    L[(size_t)N * Np + j] = l[j];
    Linv[(size_t)N * Np + j] = w;
    alpha[j] += w * zN;
  }
  if (tid == 0) {
    L[(size_t)N * Np + N] = lam;
    Linv[(size_t)N * Np + N] = ilam;
    z[N] = zN;
    alpha[N] = zN * ilam;
    const double logdet = scal[0] + 2.0 * log(lam);
    scal[0] = logdet;
    scal[1] = -0.5 * (sh[2] + zN * zN) - 0.5 * logdet - 0.5 * (N + 1) * 1.8378770664093454836;
    *status = 0;
  }
}

// ---- fused log-likelihood for N beyond one CTA's shared memory: one CLUSTER of C CTAs per hyper-parameter vector
//      (chol_group.cuh).  grid = R * C CTAs, cluster dimension C; ws = per-restart workspace described by GroupWs.
__global__ void __launch_bounds__(CG_THREADS, 1) loglik_group_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                                                     int N, int d, int Np, int C,
                                                                     const double* __restrict__ Pv, int fit_amp, double noise,
                                                                     GroupWs ws, double* __restrict__ ll_out) {
  extern __shared__ __align__(16) double gsm[];
  __shared__ double hyp[3 + APGP_MAXD];
  const int rr = blockIdx.x / C, rank = (C > 1) ? cg_cluster_ctarank() : 0;
  const int P = 1 + fit_amp + d;
  const double* p = Pv + (size_t)rr * P;
  if (!nll_row_finite(p, P)) { if (rank == 0 && threadIdx.x == 0) ll_out[rr] = -INFINITY; return; }   // uniform in the cluster
  nll_hyp(p, d, fit_amp, noise, hyp);
  __syncthreads();
  const CholGroup g = cg_make(ws, rr, N, Np, d, C, rank, X, y);
  const double ll = chol_group_loglik<true>(g, hyp, gsm, 0ull);
  if (rank == 0 && threadIdx.x == 0) ll_out[rr] = ll;
}

// ---- the same cluster class with gradients (loglik_grad_group_kernel): after chol_group_loglik, per restart
//        W = L^{-1}                     column block by column block, each column block by one CTA of the cluster
//        alpha = W^T z                  by the owner of the column block, on the way
//        K^{-1}_ab = sum_{k >= a} W_ka^T W_kb   one lower tile at a time, reduced at once into the trace products
//      dl/dp = 1/2 tr[(alpha alpha^T - K^{-1}) dK/dp] (george.GP.grad_log_likelihood, gpUtils.py:110), as grad_reduce_kernel.
//      W is kept TRANSPOSED, tile-major in a second triangle next to L: tile (i, j), i >= j, holds T_ij = W_ij^T.  In that
//      form every product is  A B^T  of two row-major tiles -- the operand form of cg_update_phase -- and the triangular
//      step is the panel solve of the factorisation (cg_trsm_dmma, X = P L_ii^{-T}) with the diagonal block's inverted 8x8
//      blocks the factorisation left in Dinv:
//        T_jj = I L_jj^{-T},   T_ij = -(sum_{j <= k < i} T_kj L_ik^T) L_ii^{-T}   (i > j),
//        K^{-1}_ab = sum_{k >= a} T_ka T_kb^T,   alpha_a = sum_{k >= a} T_ka z_k.
struct GradWs {
  double* T; double* alpha; double* part;  // per restart: transposed inverse (nb(nb+1)/2 tiles), alpha [Np], [ntiles][2 + d]
  size_t sT, sA, sPart;
};
size_t gg_restart_bytes(int Np, int d) {
  const size_t nb = Np / CG_T, nt = nb * (nb + 1) / 2;
  return (nt * CG_TILE + Np + nt * (2 + d)) * sizeof(double);
}
size_t gg_ws_bytes(int Np, int d, int R) { return (cg_ws_bytes(Np, R) + 255) / 256 * 256 + (size_t)R * gg_restart_bytes(Np, d); }
GradWs gg_ws_carve(void* ws_bytes, int Np, int d, int R) {
  const size_t nb = Np / CG_T, nt = nb * (nb + 1) / 2;
  GradWs w;
  char* base = static_cast<char*>(ws_bytes) + (cg_ws_bytes(Np, R) + 255) / 256 * 256;
  w.T = reinterpret_cast<double*>(base); w.sT = nt * CG_TILE; base += (size_t)R * w.sT * 8;
  w.alpha = reinterpret_cast<double*>(base); w.sA = Np; base += (size_t)R * w.sA * 8;
  w.part = reinterpret_cast<double*>(base); w.sPart = nt * (2 + d);
  return w;
}

// dynamic shared memory of the gradient phases: two operand pairs of the product pipeline, the tile being solved, L_ii,
// the inverted 8x8 diagonal blocks of L_ii and z_i.  The factorisation (CG_SMEM_DOUBLES) runs in the same allocation.
constexpr int GG_P = 4 * CG_TILE, GG_L = 5 * CG_TILE, GG_AUX = 6 * CG_TILE, GG_Z = GG_AUX + 8 * 64;
constexpr size_t GG_SMEM_DOUBLES = GG_Z + CG_T;
static_assert(GG_SMEM_DOUBLES >= CG_SMEM_DOUBLES, "the factorisation runs in the gradient kernel's shared memory");
static_assert(GG_SMEM_DOUBLES * 8 <= 227 * 1024, "one CTA per SM");
static_assert(2 * APGP_MAXD * CG_T + 2 * CG_T <= CG_TILE, "inputs and alpha of a tile pair fit the solve tile");
static_assert((1 + APGP_MAXD) * 8 <= CG_TILE, "warp partials fit the L_ii tile");

__device__ __forceinline__ double* gg_tile(double* base, int i, int j) { return base + (size_t)(i * (i + 1) / 2 + j) * CG_TILE; }
// column blocks of W dealt out in snake order (0, 1, .., C-1, C-1, .., 0, 0, ..): column j costs ~(nb - j)^2 / 2 products
__device__ __forceinline__ int gg_col_owner(int j, int C) { const int r = j % C; return ((j / C) & 1) ? C - 1 - r : r; }

// acc = sum_{t < cnt} A_t B_t^T over 64x64 tiles of global memory (tile-major [64][CG_LD]; tiles(t, A_t, B_t) names them),
// by all 8 warps, warp tile 32x16 as in cg_update_phase.  The operand pair of product t + 1 arrives by bulk TMA while
// product t is multiplied; `used` counts the products this CTA has taken through the two slots (slot used & 1, mbarrier
// phase (used >> 1) & 1), identical in every thread.  The products are added in t order: the bits do not depend on the CTA.
template <class F>
__device__ __forceinline__ void gg_chain(double* sm, uint64_t* full, uint32_t& used, int cnt, F tiles, double (&acc)[4][2][2]) {
  const int tid = threadIdx.x, w8 = tid >> 5, lane = tid & 31, wm = w8 >> 2, wn = w8 & 3;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }
  if (cnt == 0) return;
  auto issue = [&](int t, uint32_t slot) {
    const double* A; const double* B;
    tiles(t, A, B);
    mbar_arrive_expect_tx(&full[slot], 2u * CG_TILE * 8u);
    bulk_g2s(sm + (size_t)slot * 2 * CG_TILE, A, CG_TILE * 8, &full[slot]);
    bulk_g2s(sm + (size_t)slot * 2 * CG_TILE + CG_TILE, B, CG_TILE * 8, &full[slot]);
  };
  fence_proxy_async();                                 // tiles this CTA stored through the generic proxy -> bulk copies
  __syncthreads();
  if (tid == 0) issue(0, used & 1u);
  for (int t = 0; t < cnt; ++t, ++used) {
    const uint32_t slot = used & 1u;
    mbar_wait(&full[slot], (used >> 1) & 1u);
    __syncthreads();                                   // everyone is done with product t - 1: its slot can be refilled
    if (tid == 0 && t + 1 < cnt) issue(t + 1, slot ^ 1u);
    const double* As = sm + (size_t)slot * 2 * CG_TILE;
    const double* ap = As + (wm * 32 + (lane >> 2)) * CG_LD + (lane & 3);
    const double* bp = As + CG_TILE + (wn * 16 + (lane >> 2)) * CG_LD + (lane & 3);
#pragma unroll 4
    for (int k4 = 0; k4 < CG_T / 4; ++k4) {
      double av[4], bv[2];
#pragma unroll
      for (int a = 0; a < 4; ++a) av[a] = ap[a * 8 * CG_LD + k4 * 4];
#pragma unroll
      for (int b = 0; b < 2; ++b) bv[b] = bp[b * 8 * CG_LD + k4 * 4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) dmma884(acc[a][b][0], acc[a][b][1], av[a], bv[b]);
    }
  }
}

// all CTAs of the cluster (or the CTA when C = 1) have finished their global writes; they are visible to every one of them
__device__ __forceinline__ void gg_cluster_sync(int C) {
  __threadfence();
  if (C > 1) asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;\n" ::: "memory");
  else __syncthreads();
}

// this CTA's column blocks of T = W^T (and alpha on those rows)
__device__ __forceinline__ void gg_inverse_phase(const CholGroup& g, double* T, double* alpha, double* sm, uint64_t* full,
                                                 uint64_t* lbar, uint32_t& used, uint32_t& lused) {
  const int tid = threadIdx.x, w8 = tid >> 5, lane = tid & 31, wm = w8 >> 2, wn = w8 & 3;
  const int nb = g.nb, row = w8 * 8 + (lane >> 2), q = lane & 3;
  double* const Ps = sm + GG_P;
  double* const Ls = sm + GG_L;
  double* const aux = sm + GG_AUX;
  double* const zb = sm + GG_Z;
  for (int j = 0; j < nb; ++j) {
    if (gg_col_owner(j, g.C) != g.rank) continue;
    double al = 0.0;                                   // alpha_{64 j + row}: sum over i of (T_ij z_i)[row], i ascending
    for (int i = j; i < nb; ++i) {
      fence_proxy_async();
      __syncthreads();                                 // the previous step is done with Ls, Ps, aux, zb
      if (tid == 0) {
        mbar_arrive_expect_tx(lbar, CG_TILE * 8u);
        bulk_g2s(Ls, cg_tile_ptr(g, i, i), CG_TILE * 8, lbar);
      }
      const double* Dg = g.Dinv + (size_t)i * CG_T * CG_T + CG_T;
      for (int e = tid; e < 8 * 64; e += CG_THREADS) aux[e] = __ldcg(Dg + e);
      if (tid < CG_T) zb[tid] = __ldcg(g.r + i * CG_T + tid);
      double acc[4][2][2];
      gg_chain(sm, full, used, i - j, [&](int t, const double*& A, const double*& B) {
        A = gg_tile(T, j + t, j); B = cg_tile_ptr(g, i, j + t);
      }, acc);
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 2; ++b) {
          const int r = wm * 32 + a * 8 + (lane >> 2), c = wn * 16 + b * 8 + 2 * q;
          double2 o;
          if (i == j) { o.x = (r == c) ? 1.0 : 0.0; o.y = (r == c + 1) ? 1.0 : 0.0; }
          else { o.x = -acc[a][b][0]; o.y = -acc[a][b][1]; }
          *reinterpret_cast<double2*>(Ps + r * CG_LD + c) = o;
        }
      __syncthreads();
      mbar_wait(lbar, lused & 1u); ++lused;
      double* const Ts[1] = {Ps};
      cg_trsm_dmma<1>(Ts, Ls, aux, w8, lane);          // warp w8 solves rows 8 w8 .. 8 w8 + 7: T_ij
      const double* xr = Ps + row * CG_LD;
      double s = 0.0;
#pragma unroll
      for (int m = 0; m < CG_T / 4; ++m) s = fma(xr[q + 4 * m], zb[q + 4 * m], s);
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      al += s;
      double* Tij = gg_tile(T, i, j);
#pragma unroll
      for (int rr = 0; rr < 8; ++rr) {
        const int off = (w8 * 8 + rr) * CG_LD + 2 * lane;
        *reinterpret_cast<double2*>(Tij + off) = *reinterpret_cast<const double2*>(Ps + off);
      }
    }
    if (q == 0) alpha[j * CG_T + row] = al;
  }
}

// this CTA's lower tiles of K^{-1} (tile t = a(a+1)/2 + b belongs to CTA t mod C), each reduced at once into
// part[t] = [t == 0 ? sum alpha : 0, 1/2 sum G Kk, 1/2 sum G Kk (1/2 D_c^2 / M_c) ..]; padding rows and columns excluded
__device__ __forceinline__ void gg_reduce_phase(const CholGroup& g, double* T, const double* alpha, double* part,
                                                const double* hyp, double* sm, uint64_t* full, uint32_t& used) {
  const int tid = threadIdx.x, w8 = tid >> 5, lane = tid & 31, wm = w8 >> 2, wn = w8 & 3;
  const int nb = g.nb, N = g.N, d = g.d, C = g.C, me = g.rank;
  double* const Xa = sm + GG_P;                        // [d][64] inputs of the tile's row block, then of its column block
  double* const Xb = Xa + APGP_MAXD * CG_T;
  double* const aa_ = Xb + APGP_MAXD * CG_T;           // alpha of the row block, then of the column block
  double* const ab_ = aa_ + CG_T;
  double* const wred = sm + GG_L;                      // [1 + d][8] warp partials
  const double amp = hyp[1];
  if (me == 0) {                                       // tile 0 is rank 0's: sum alpha in a fixed order
    double sa = 0.0;
    for (int i = tid; i < N; i += CG_THREADS) sa += __ldcg(alpha + i);
    sa = cta_sum<CG_THREADS>(sa, wred);
    if (tid == 0) part[0] = sa;
  }
  int t = -1;
  for (int a = 0; a < nb; ++a)
    for (int b = 0; b <= a; ++b) {
      if (++t % C != me) continue;
      double acc[4][2][2];
      gg_chain(sm, full, used, nb - a, [&](int s, const double*& A, const double*& B) {
        A = gg_tile(T, a + s, a); B = gg_tile(T, a + s, b);
      }, acc);
      __syncthreads();                                 // the previous tile's reduction is done with Xa .. wred
      for (int e = tid; e < CG_T * d; e += CG_THREADS) {
        const int r = e / d, c = e - r * d;
        const int ga = a * CG_T + r, gb = b * CG_T + r;
        Xa[c * CG_T + r] = (ga < N) ? g.X[(size_t)ga * d + c] : 0.0;
        Xb[c * CG_T + r] = (gb < N) ? g.X[(size_t)gb * d + c] : 0.0;
      }
      if (tid < CG_T) { aa_[tid] = __ldcg(alpha + a * CG_T + tid); ab_[tid] = __ldcg(alpha + b * CG_T + tid); }
      __syncthreads();
      // this thread's 16 entries, in the accumulator layout: rows wm*32 + 8 u + lane/4, columns wn*16 + 8 v + 2 (lane%4) + h
      double gk[4][2][2];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v) { gk[u][v][0] = 0.0; gk[u][v][1] = 0.0; }
      const int r0 = wm * 32 + (lane >> 2), c0 = wn * 16 + 2 * (lane & 3);
      for (int c = 0; c < d; ++c) {
        const double im = hyp[3 + c];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 2; ++v)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const double df = Xa[c * CG_T + r0 + 8 * u] - Xb[c * CG_T + c0 + 8 * v + h];
              gk[u][v][h] += 0.5 * df * df * im;       // sum_c of 1/2 D_c^2 / M_c
            }
      }
      double v0 = 0.0;
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 2; ++v)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int pl = r0 + 8 * u, ql = c0 + 8 * v + h, p = a * CG_T + pl, qq = b * CG_T + ql;
            const double kk = amp * exp(-gk[u][v][h]);
            const double G = aa_[pl] * ab_[ql] - acc[u][v][h];
            const double w = (p == qq) ? 0.5 : 1.0;    // off-diagonal pairs appear twice in the full trace
            const bool on = p < N && qq < N && (a != b || ql <= pl);
            gk[u][v][h] = on ? w * G * kk : 0.0;
            v0 += gk[u][v][h];
          }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v0 += __shfl_xor_sync(0xffffffffu, v0, o);
      if (lane == 0) wred[w8] = v0;
      for (int c = 0; c < d; ++c) {
        const double im = hyp[3 + c];
        double vc = 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 2; ++v)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const double df = Xa[c * CG_T + r0 + 8 * u] - Xb[c * CG_T + c0 + 8 * v + h];
              vc += gk[u][v][h] * (0.5 * df * df * im);
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) vc += __shfl_xor_sync(0xffffffffu, vc, o);
        if (lane == 0) wred[(1 + c) * 8 + w8] = vc;
      }
      __syncthreads();
      double* pt = part + (size_t)t * (2 + d);
      if (tid <= d) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += wred[tid * 8 + w];
        pt[1 + tid] = s;
      }
      if (tid == 0 && t != 0) pt[0] = 0.0;
    }
}

// grid = R * C CTAs, cluster dimension C, as loglik_group_kernel (whose ll it returns bit for bit); grad_out [R][2 + d]:
// [sum alpha, d/dlog_constant, d/dlog M_0 ..] (loglik_small_kernel's layout), zeros where ll is -inf.
__global__ void __launch_bounds__(CG_THREADS, 1) loglik_grad_group_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                                                          int N, int d, int Np, int C,
                                                                          const double* __restrict__ Pv, int fit_amp, double noise,
                                                                          GroupWs ws, GradWs gw, double* __restrict__ ll_out,
                                                                          double* __restrict__ grad_out) {
  extern __shared__ __align__(16) double gsm[];
  __shared__ double hyp[3 + APGP_MAXD];
  __shared__ __align__(8) uint64_t bars[3];            // operand slots 0 / 1 of gg_chain, L_ii
  const int tid = threadIdx.x;
  const int rr = blockIdx.x / C, rank = (C > 1) ? cg_cluster_ctarank() : 0;
  const int P = 1 + fit_amp + d;
  const double* p = Pv + (size_t)rr * P;
  double* gout = grad_out + (size_t)rr * (2 + d);
  if (!nll_row_finite(p, P)) {                         // uniform in the cluster
    if (rank == 0) { if (tid == 0) ll_out[rr] = -INFINITY; if (tid < 2 + d) gout[tid] = 0.0; }
    return;
  }
  nll_hyp(p, d, fit_amp, noise, hyp);
  __syncthreads();
  const CholGroup g = cg_make(ws, rr, N, Np, d, C, rank, X, y);
  const double ll = chol_group_loglik<true>(g, hyp, gsm, 0ull);
  if (rank == 0 && tid == 0) ll_out[rr] = ll;
  if (ll == -INFINITY) {                               // the same bits in every CTA: the whole cluster leaves
    if (rank == 0 && tid < 2 + d) gout[tid] = 0.0;
    return;
  }
  // every CTA has acquired flag A of the last block (C > 1) inside chol_group_loglik: all of L, Dinv and z are visible
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_init(&bars[2], 1); mbar_fence_init(); }
  __syncthreads();
  double* T = gw.T + rr * gw.sT;
  double* alpha = gw.alpha + rr * gw.sA;
  double* part = gw.part + rr * gw.sPart;
  uint32_t used = 0, lused = 0;
  gg_inverse_phase(g, T, alpha, gsm, bars, &bars[2], used, lused);
  gg_cluster_sync(C);
  gg_reduce_phase(g, T, alpha, part, hyp, gsm, bars, used);
  gg_cluster_sync(C);
  if (rank == 0 && tid < 2 + d) {                      // per-tile partials in tile order, whichever CTA owned each tile
    const int nt = g.nb * (g.nb + 1) / 2;
    double s = 0.0;
    for (int t = 0; t < nt; ++t) s += __ldcg(part + (size_t)t * (2 + d) + tid);
    gout[tid] = s;
  }
}

PerDeviceOnce g_attr_done;
int ensure_attrs() {
  if (!g_attr_done.needed()) return 0;
  cudaError_t e;
  e = cudaFuncSetAttribute(chol_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DIAG_SMEM); if (e) return (int)e;
  e = cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TILE_SMEM); if (e) return (int)e;
  e = cudaFuncSetAttribute(chol_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TILE_SMEM); if (e) return (int)e;
  e = cudaFuncSetAttribute(gemm_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TILE_SMEM); if (e) return (int)e;
  e = cudaFuncSetAttribute(loglik_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024); if (e) return (int)e;
  e = cudaFuncSetAttribute(loglik_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CG_SMEM_DOUBLES * 8)); if (e) return (int)e;
  e = cudaFuncSetAttribute(loglik_group_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1); if (e) return (int)e;
  e = cudaFuncSetAttribute(loglik_grad_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(GG_SMEM_DOUBLES * 8)); if (e) return (int)e;
  e = cudaFuncSetAttribute(loglik_grad_group_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1); if (e) return (int)e;
  g_attr_done.mark();
  return 0;
}

}  // namespace

int launch_build_K(const double* X, const double* y, int N, int d, const double* hyper, const FactorBatch& fb,
                   cudaStream_t st) {
  const int nb = fb.Np / T;
  dim3 grid(nb * (nb + 1) / 2, fb.R);
  build_K_kernel<<<grid, 256, 0, st>>>(X, y, N, d, fb.Np, hyper, fb.K, fb.r, fb.logdet, fb.info);
  return (int)cudaGetLastError();
}

int launch_cholesky(const FactorBatch& fb, int num_sms, cudaStream_t st, int* launches) {
  (void)num_sms;
  int e = ensure_attrs(); if (e) return e;
  const int nb = fb.Np / T;
  for (int k = 0; k < nb; ++k) {
    chol_diag_kernel<<<fb.R, DIAG_THREADS, DIAG_SMEM, st>>>(fb, k);
    if (launches) ++*launches;
    const int rem = nb - k - 1;
    if (rem > 0) {
      chol_panel_kernel<<<dim3(rem, fb.R), GT, TILE_SMEM, st>>>(fb, k);
      chol_update_kernel<<<dim3(rem * (rem + 1) / 2, fb.R), GT, TILE_SMEM, st>>>(fb, k);
      if (launches) *launches += 2;
    }
  }
  return (int)cudaGetLastError();
}

// Recursive-doubling inverse of a lower-triangular matrix whose diagonal 64-blocks are already
// inverted:  [L11 0; L21 L22]^{-1} = [X11 0; -X22 (L21 X11)  X22].
int launch_tri_inverse(const double* L, const double* Dinv, int Np, double* Linv, double* work, cudaStream_t st,
                       int* launches) {
  int e = ensure_attrs(); if (e) return e;
  const int nb = Np / T;
  init_linv_kernel<<<148 * 4, 256, 0, st>>>(Dinv, Np, Linv);
  if (launches) ++*launches;
  for (int s = 1; s < nb; s *= 2) {
    // pairs p: first block tiles [2ps, 2ps+s), second [2ps+s, min(2ps+2s, nb))
    for (int p0 = 0; p0 + s < nb; p0 += 2 * s) {
      const int r2 = ((p0 + 2 * s <= nb) ? s : (nb - p0 - s));      // tiles in second block
      const double* L21 = L + (size_t)(p0 + s) * T * Np + (size_t)p0 * T;
      const double* X11 = Linv + (size_t)p0 * T * Np + (size_t)p0 * T;
      const double* X22 = Linv + (size_t)(p0 + s) * T * Np + (size_t)(p0 + s) * T;
      double* X21 = Linv + (size_t)(p0 + s) * T * Np + (size_t)p0 * T;
      double* Tm = work + (size_t)(p0 + s) * T * Np + (size_t)p0 * T;
      GemmDesc g1{L21, Np, 0, X11, Np, 0, Tm, Np, 1.0, r2, s, s, 1, 0, 0, 0};
      gemm_tile_kernel<<<dim3(r2 * s, 1), GT, TILE_SMEM, st>>>(g1);
      GemmDesc g2{X22, Np, 0, Tm, Np, 0, X21, Np, -1.0, r2, s, r2, 2, 0, 0, 0};
      gemm_tile_kernel<<<dim3(r2 * s, 1), GT, TILE_SMEM, st>>>(g2);
      if (launches) *launches += 2;
    }
  }
  return (int)cudaGetLastError();
}

size_t loglik_small_smem(int N, int d) { return SmallLL::doubles(N, d) * sizeof(double); }

int launch_loglik_small(const double* X, const double* y, int N, int d, const double* P, int fit_amp, double noise, int R,
                        double* ll, double* grad, cudaStream_t st) {
  int e = ensure_attrs(); if (e) return e;
  loglik_small_kernel<<<R, LL_NT, loglik_small_smem(N, d), st>>>(X, y, N, d, P, fit_amp, noise, ll, grad);
  return (int)cudaGetLastError();
}

// cluster size for the fused group kernels: as many CTAs per restart as fit the GPU in one wave (power of two, at most
// 16), but no more than the tile count can feed (nb - 1 panel tiles at the first step).  APGP_CHOL_CLUSTER overrides.
int chol_group_cluster(int Np, int R, int num_sms) {
  const int nb = Np / T;
  int C = 1;
  // 16-CTA clusters (non-portable size) only pay for a handful of vectors: measured at R = 8, N = 1024 a batch takes
  // 0.91 ms with C = 8 and 1.31 ms with C = 16 (few GPCs can host a 16-CTA cluster at a time); R = 1: 0.90 vs 0.67 ms
  const int maxC = (R <= 4) ? 16 : 8;
  while (C * 2 <= maxC && (long)R * C * 2 <= num_sms && C * 2 <= (nb > 1 ? nb - 1 : 1) * 2) C *= 2;
  if (const char* v = getenv("APGP_CHOL_CLUSTER")) { const int c = atoi(v); if (c == 1 || c == 2 || c == 4 || c == 8 || c == 16) C = c; }
  return C;
}
size_t chol_group_ws_bytes(int Np, int R) { return cg_ws_bytes(Np, R); }
// R clusters of C CTAs (CG_THREADS each): launch(cfg, C); a cluster size that cannot be scheduled is halved (C = 1 always
// can), C returns the size that ran
template <class F>
static cudaError_t launch_clusters(int& C, int R, size_t smem, cudaStream_t st, F launch) {
  for (;;) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(R * C)); cfg.blockDim = dim3(CG_THREADS);
    cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const cudaError_t ce = launch(cfg, C);
    if (ce == cudaSuccess || C == 1) return ce;
    (void)cudaGetLastError();
    C >>= 1;
  }
}
size_t loglik_grad_group_ws_bytes(int Np, int d, int R) { return gg_ws_bytes(Np, d, R); }
// ws: loglik_grad_group_ws_bytes(Np, d, R) bytes; grad [R][2 + d].  One launch for all R vectors.
int launch_loglik_grad_group(const double* X, const double* y, int N, int d, int Np, const double* P, int fit_amp,
                             double noise, int R, int num_sms, void* ws_bytes, double* ll, double* grad, cudaStream_t st) {
  int e = ensure_attrs(); if (e) return e;
  GroupWs ws = cg_ws_carve(ws_bytes, Np, R);
  GradWs gw = gg_ws_carve(ws_bytes, Np, d, R);
  cudaError_t ce = cudaMemsetAsync(ws.flags, 0, (size_t)R * 16, st);
  if (ce != cudaSuccess) return (int)ce;
  int C = chol_group_cluster(Np, R, num_sms);
  ce = launch_clusters(C, R, GG_SMEM_DOUBLES * 8, st, [&](const cudaLaunchConfig_t& cfg, int c) {
    return cudaLaunchKernelEx(&cfg, loglik_grad_group_kernel, X, y, N, d, Np, c, P, fit_amp, noise, ws, gw, ll, grad);
  });
  return (int)ce;
}
// ws: chol_group_ws_bytes(Np, R) bytes.  P [R][1 + fit_amp + d] as for launch_loglik_small.  One launch for all R vectors.
int launch_loglik_group(const double* X, const double* y, int N, int d, int Np, const double* P, int fit_amp, double noise,
                        int R, int num_sms, void* ws_bytes, double* ll, cudaStream_t st) {
  int e = ensure_attrs(); if (e) return e;
  GroupWs ws = cg_ws_carve(ws_bytes, Np, R);
  cudaError_t ce = cudaMemsetAsync(ws.flags, 0, (size_t)R * 16, st);
  if (ce != cudaSuccess) return (int)ce;
  int C = chol_group_cluster(Np, R, num_sms);
  ce = launch_clusters(C, R, CG_SMEM_DOUBLES * 8, st, [&](const cudaLaunchConfig_t& cfg, int c) {
    return cudaLaunchKernelEx(&cfg, loglik_group_kernel, X, y, N, d, Np, c, P, fit_amp, noise, ws, ll);
  });
#ifdef APGP_PROF_CG
  if (getenv("APGP_PROF_PRINT")) {
    cudaStreamSynchronize(st);
    long long h[2][24];
    cudaMemcpyFromSymbol(h, g_cgprof, sizeof(h));
    for (int b = 0; b < 2; ++b) {
      fprintf(stderr, "[cgprof] N=%d R=%d C=%d cta=%d cycles:", N, R, C, b);
      for (int i = 0; i < 23; ++i) fprintf(stderr, " %lld", h[b][i]);
      fprintf(stderr, "\n");
    }
    long long z[2][24] = {};
    cudaMemcpyToSymbol(g_cgprof, z, sizeof(z));
  }
#endif
  return (int)ce;
}

int launch_append_point(const double* X, int N, int d, int Np, const double* xnew_dev, const double* hyper_dev, double kappa,
                        double rnew, double* L, double* Linv, double* z, double* alpha, double* kvec, double* lvec,
                        double* uvec, double* scal, int* status, cudaStream_t st, int* launches) {
  append_kvec_kernel<<<(N + 255) / 256, 256, 0, st>>>(X, N, d, xnew_dev, hyper_dev, kvec);
  cudaMemsetAsync(lvec, 0, sizeof(double) * Np, st);
  append_linv_rows_kernel<<<(N + 7) / 8, 256, 0, st>>>(Linv, Np, N, kvec, lvec);
  linvT_matvec_kernel<<<Np / T, 256, 0, st>>>(Linv, Np, lvec, uvec);      // u_j = sum_{i>=j} Linv[i][j] l_i
  append_finish_kernel<<<1, 256, 0, st>>>(L, Linv, Np, N, lvec, uvec, z, alpha, kappa, rnew, scal, status);
  if (launches) *launches += 4;
  return (int)cudaGetLastError();
}

int launch_linvT_matvec(const double* Linv, int Np, const double* z, double* alpha, cudaStream_t st) {
  linvT_matvec_kernel<<<Np / T, 256, 0, st>>>(Linv, Np, z, alpha);
  return (int)cudaGetLastError();
}

int launch_refine_alpha(const double* X, const double* y, int N, int d, int Np, const double* hyper_dev,
                        const double* Linv, double* alpha, double* w1, double* w2, cudaStream_t st, int* launches) {
  alpha_residual_kernel<<<(Np + 7) / 8, 256, 0, st>>>(X, y, N, d, hyper_dev, alpha, w1, Np);
  cudaMemsetAsync(w2, 0, sizeof(double) * Np, st);
  append_linv_rows_kernel<<<(Np + 7) / 8, 256, 0, st>>>(Linv, Np, Np, w1, w2);       // w2 = L^{-1} res
  linvT_matvec_kernel<<<Np / T, 256, 0, st>>>(Linv, Np, w2, w1);                      // w1 = L^{-T} w2
  axpy_kernel<<<(Np + 255) / 256, 256, 0, st>>>(Np, w1, alpha);
  if (launches) *launches += 4;
  return (int)cudaGetLastError();
}

int launch_loglik_finish(const FactorBatch& fb, double* ll, cudaStream_t st) {
  loglik_finish_kernel<<<fb.R, 256, 0, st>>>(fb, ll);
  return (int)cudaGetLastError();
}

size_t grad_loglik_doubles(int Np, int d) { const size_t nb = Np / T; return (size_t)(2 + d) * (1 + nb * (nb + 1) / 2); }

int launch_grad_loglik(const double* X, int N, int d, int Np, const double* Linv, const double* alpha,
                       const double* hyper_dev, int fit_amp, double* work, double* grad_dev, cudaStream_t st,
                       int* launches) {
  (void)fit_amp;
  int e = ensure_attrs(); if (e) return e;
  const int nb = Np / T;
  // Kinv (lower tiles) = Linv^T Linv
  GemmDesc g{Linv, Np, 1, Linv, Np, 0, work, Np, 1.0, nb, nb, nb, 3, 0, 0, 0};
  gemm_tile_kernel<<<dim3(nb * nb, 1), GT, TILE_SMEM, st>>>(g);
  // grad_dev: [2 + d] result, followed by [ntiles][2 + d] per-tile partials (grad_loglik_doubles(Np, d) in all)
  const int ntiles = nb * (nb + 1) / 2;
  grad_reduce_kernel<<<ntiles, 256, 0, st>>>(X, N, d, Np, work, alpha, hyper_dev, grad_dev + (2 + d));
  grad_finish_kernel<<<1, 64, 0, st>>>(grad_dev + (2 + d), ntiles, d, grad_dev);
  if (launches) *launches += 3;
  return (int)cudaGetLastError();
}

}  // namespace apgp
