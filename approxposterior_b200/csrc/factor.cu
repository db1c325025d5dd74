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
// ws: chol_group_ws_bytes(Np, R) bytes.  P [R][1 + fit_amp + d] as for launch_loglik_small.  One launch for all R vectors.
int launch_loglik_group(const double* X, const double* y, int N, int d, int Np, const double* P, int fit_amp, double noise,
                        int R, int num_sms, void* ws_bytes, double* ll, cudaStream_t st) {
  int e = ensure_attrs(); if (e) return e;
  GroupWs ws = cg_ws_carve(ws_bytes, Np, R);
  cudaError_t ce = cudaMemsetAsync(ws.flags, 0, (size_t)R * 16, st);
  if (ce != cudaSuccess) return (int)ce;
  int C = chol_group_cluster(Np, R, num_sms);
  for (;;) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(R * C)); cfg.blockDim = dim3(CG_THREADS);
    cfg.dynamicSmemBytes = CG_SMEM_DOUBLES * 8; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, loglik_group_kernel, X, y, N, d, Np, C, P, fit_amp, noise, ws, ll);
    if (ce == cudaSuccess || C == 1) break;
    (void)cudaGetLastError();                // the cluster could not be scheduled: halve it (C = 1 always can)
    C >>= 1;
  }
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
