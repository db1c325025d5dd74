// Compiled twice by tests/test_loglik_contraction.py, with and without -fmad=false: the two log-likelihood evaluators of
// loglik.cuh must compile to the same FP64 arithmetic either way (factor.cu and optimize.cu differ in that flag).
// With -DOPAQUE_LOG every log() of the evaluators becomes an opaque stand-in, which leaves the code the project owns:
// libdevice's log itself contracts one a*b + a*b into fma(a, b, a*b) under -fmad, which rounds to the same 2 (a*b).
#include <cuda_runtime.h>
#include <math.h>
#ifdef OPAQUE_LOG
__device__ __forceinline__ double opaque_log(double x) { double r; asm volatile("mov.b64 %0, %1;" : "=d"(r) : "d"(x)); return r; }
#define log(x) opaque_log(x)
#endif
#include "../../approxposterior_b200/csrc/loglik.cuh"

namespace apgp {

__global__ void __launch_bounds__(LL_NT, 1) probe_small(const double* p, int N, int d, double* out) {
  extern __shared__ __align__(16) double sm[];
  const SmallLL L = SmallLL::carve(sm, N, d);
  nll_hyp(p, d, 1, 1e-6, L.hyp);
  const double ll = loglik_small(L, N, d, false);
  if (threadIdx.x == 0) *out = ll;
}

__global__ void __launch_bounds__(CG_THREADS, 1) probe_group(GroupWs ws, const double* X, const double* y, const double* hyp,
                                                             int N, int Np, int d, double* out) {
  extern __shared__ __align__(16) double gsm[];
  const CholGroup g = cg_make(ws, 0, N, Np, d, 1, 0, X, y);
  const double ll = chol_group_loglik<true>(g, hyp, gsm, 0ull);
  if (threadIdx.x == 0) *out = ll;
}

}  // namespace apgp
