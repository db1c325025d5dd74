// One log-likelihood evaluator per size class, ll = -1/2 |z|^2 - log|L| - N/2 log 2pi with z = L^{-1}(y - m) (gpUtils._nll,
// reference gpUtils.py:46-80), shared by the batched log-likelihood (factor.cu) and the device optimisers' objective
// (optimize.cu):
//   small  one CTA per parameter vector, everything in shared memory (loglik_small below);
//   group  one thread-block cluster per parameter vector, the matrix in L2-resident global memory (chol_group.cuh).
// optimize.cu is compiled with -fmad=false, factor.cu with contraction on.  Every multiply-add of both evaluators is
// written out -- fma() where it is fused, __dmul_rn / __dadd_rn / __dsub_rn where it is not -- so they round the same in
// both translation units and the two entry points return the same bits (tests/test_loglik_contraction.py checks the SASS).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <type_traits>
#include "common.cuh"
#include "chol_small.cuh"
#include "chol_group.cuh"

namespace apgp {

constexpr double LOG_2PI = 1.8378770664093454836;
constexpr int LL_NT = 256;                         // threads of the small evaluator's CTA

// p = [mean, (log_constant), log M_0 ..] (george order, P entries) is finite in every entry
__device__ __forceinline__ bool nll_row_finite(const double* p, int P) {
  bool fin = true;
  for (int k = 0; k < P; ++k) { const double v = p[k]; fin = fin && (v == v) && (fabs(v) < INFINITY); }
  return fin;
}

// The hyper row [mean, amplitude, noise variance, 1/M_0 .. 1/M_{d-1}] of p; amplitude d e^{p_1} when fitted, else 1.
// Thread 0 writes the scalars, thread c < d writes 1/M_c; the caller makes them visible to the CTA.
__device__ __forceinline__ void nll_hyp(const double* p, int d, int fit_amp, double noise, double* hyp) {
  const int tid = threadIdx.x;
  if (tid == 0) { hyp[0] = p[0]; hyp[1] = fit_amp ? (double)d * exp(p[1]) : 1.0; hyp[2] = noise; }
  if (tid < d) hyp[3 + tid] = exp(-p[1 + fit_amp + tid]);
}

// Shared memory of the small evaluator, carved from the start of the dynamic shared memory: packed lower triangle of K
// (-> L), X [N][d], y [N], r [N] (-> z), diag(L) [N], hyper row [3 + d], reduction slots, failure flag.
struct SmallLL {
  double *K, *X, *y, *r, *col, *hyp, *red;
  int* bad;
  static constexpr int NRED = LL_NT / 32;
  __host__ __device__ static size_t doubles(int N, int d) {
    return (size_t)N * (N + 1) / 2 + (size_t)N * (d + 3) + 3 + d + NRED + 1;
  }
  __device__ static SmallLL carve(double* base, int N, int d) {
    SmallLL L;
    L.K = base; L.X = L.K + (size_t)N * (N + 1) / 2; L.y = L.X + (size_t)N * d; L.r = L.y + N; L.col = L.r + N;
    L.hyp = L.col + N; L.red = L.hyp + 3 + d; L.bad = reinterpret_cast<int*>(L.red + NRED);
    return L;
  }
};

// The small class: N + 1 <= LL_NT and SmallLL::doubles(N, d) within the CTA's shared memory.  X and y are staged and the
// hyper row is written (nll_hyp) by the caller; the first barrier here publishes them.  Covariance build, Cholesky with
// the forward substitution riding along (r <- z, col <- diag(L); with store_diag the whole of L is left in K), and the
// two reductions.  Returns ll, or -inf when K is not positive definite or ll is not finite, to every thread.
__device__ __forceinline__ double loglik_small(const SmallLL& L, int N, int d, bool store_diag) {
  const int tid = threadIdx.x;
  PROF_T(t_e0);
  __syncthreads();
  const double mean = L.hyp[0], amp = L.hyp[1], noise = L.hyp[2];
  const double* invM = L.hyp + 3;
  const double* X = L.X;
  if (tid == 0) *L.bad = 0;
  for (int i = tid; i < N; i += LL_NT) L.r[i] = L.y[i] - mean;
  PROF_T(t_b0);
  // covariance: the packed triangle is one linear array, so element e = i(i+1)/2 + j goes to thread e mod LL_NT ((i, j)
  // recovered with a float sqrt + integer fix-up); two or four elements are in flight per thread so their distance and
  // exp chains overlap
  {
    const int total = N * (N + 1) / 2;
    auto build = [&](auto uc) {
      constexpr int U = decltype(uc)::value;
      for (int e0 = tid; e0 < total; e0 += U * LL_NT) {
        int ii[U], jj[U];
        bool on[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int e = e0 + u * LL_NT;
          on[u] = e < total;
          int i = (int)((sqrtf(8.0f * (float)e + 1.0f) - 1.0f) * 0.5f);
          if ((i + 1) * (i + 2) / 2 <= e) ++i;
          if (i * (i + 1) / 2 > e) --i;
          if (!on[u]) i = 0;
          ii[u] = i;
          jj[u] = on[u] ? e - i * (i + 1) / 2 : 0;
        }
        double sv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) sv[u] = 0.0;
        for (int c = 0; c < d; ++c) {
          const double m = invM[c];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const double da = X[ii[u] * d + c] - X[jj[u] * d + c];
            sv[u] = fma(da * da, m, sv[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          double v = __dmul_rn(amp, exp(-0.5 * sv[u]));
          if (ii[u] == jj[u]) v = __dadd_rn(v, noise);
          if (on[u]) L.K[e0 + u * LL_NT] = v;
        }
      }
    };
    // measured (cycles per evaluation, 2 -> 4 in flight): N = 50 +1000, 70 +800, 90 -700, 200 -7000, N = 200 / d = 10 -26000
    if (total > 12 * LL_NT) build(std::integral_constant<int, 4>{}); else build(std::integral_constant<int, 2>{});
  }
  PROF_ADD(7, t_b0);
  __syncthreads();
  PROF_ADD(2, t_e0);                                            // prologue + covariance build
  chol_packed_blocked<LL_NT>(L.K, L.r, L.col, N, L.bad, store_diag);
  PROF_T(t_e1);
  double zpart = 0.0, lpart = 0.0;
  for (int i = tid; i < N; i += LL_NT) { zpart = fma(L.r[i], L.r[i], zpart); lpart += log(L.col[i]); }
  const double ssq = cta_sum<LL_NT>(zpart, L.red);
  const double logdet = cta_sum<LL_NT>(lpart, L.red);
  const bool bad = (*L.bad != 0);
  PROF_ADD(3, t_e1);                                            // log-det + |z|^2 reductions
  const double ll = __dsub_rn(__dsub_rn(__dmul_rn(-0.5, ssq), logdet), __dmul_rn(__dmul_rn(0.5, (double)N), LOG_2PI));
  if (bad || !(ll == ll) || !(fabs(ll) < INFINITY)) return -INFINITY;
  return ll;
}

}  // namespace apgp
