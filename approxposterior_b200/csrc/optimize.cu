// Device-resident local optimisers: SciPy's Nelder-Mead and Powell (bracket + Brent line search) restated
// for one CTA per restart, so a whole multistart minimisation is ONE launch instead of one host<->device
// round trip per objective evaluation.
//
// Replaces the inner loops of (reference call sites):
//   utility.minimizeObjective   utility.py:332-371  scipy.optimize.minimize(fn, t0, method="nelder-mead",
//                                                   options={"adaptive": True}) per restart, fn = AGP/BAPE/Jones
//                                                   utility (utility.py:99-250) or -mean (findMAP, approx.py:909-914)
//   gpUtils.optimizeGP          gpUtils.py:223-247  scipy.optimize.minimize(_nll, x0, method="powell") per restart,
//                                                   _nll = gpUtils.py:46-80 behind defaultHyperPrior (gpUtils.py:22-43)
//
// The optimiser statements follow SciPy 1.18's _minimize_neldermead / _minimize_powell / bracket / Brent in the
// same floating-point order as approxposterior_b200/_optimizers.py (which is checked point-for-point against
// SciPy); this translation unit is compiled with -fmad=false so that no multiply-add is contracted and the
// optimiser arithmetic rounds exactly as NumPy's does.  Objective code asks for fused multiply-adds explicitly.
//
// Execution model inside a CTA: control flow is uniform -- every thread carries the optimiser's scalars in
// registers and takes the same branches; vectors (simplex, direction set) live in shared memory and are updated
// element-wise by threads i < n; an objective evaluation is a CTA-cooperative function that returns the same
// value to every thread.
//
// Licence note: nelder_mead_dev, powell_dev, bracket_dev and brent_dev restate algorithms of SciPy 1.18
// (scipy/optimize/_optimize.py), which is distributed under the BSD 3-Clause licence --
// Copyright (c) 2001-2002 Enthought, Inc. 2003, SciPy Developers.  All rights reserved.  Redistribution and use in
// source and binary forms, with or without modification, are permitted provided that the copyright notice, the list
// of conditions and the disclaimer of the BSD 3-Clause licence are retained (full text in
// approxposterior_b200/_optimizers.py); neither the name of the copyright holder nor the names of its contributors
// may be used to endorse or promote products derived from this software without specific prior written permission.
// THIS SOFTWARE IS PROVIDED "AS IS", WITHOUT WARRANTIES OF ANY KIND.
#include "apgp_internal.h"
#include "loglik.cuh"
#include <math.h>
#include <stdlib.h>

namespace apgp {
namespace {

constexpr int OT = 256;                 // threads per CTA
constexpr int OW = OT / 32;
// The objectives are __noinline__ on purpose: the optimisers call them from ~20 places, and inlining every copy
// made 600 KB of SASS per kernel (37 600 instructions; 6 400 now, +11 % speed: profiles/r01_optimizers.md).
// A non-inlined member cannot see that the struct's pointers are shared-memory addresses, so the structs carry
// OFFSETS (in doubles) from the dynamic shared-memory base and eval() rebuilds typed shared pointers from them.

// ------------------------------------------------------------------------------------------------------
// Objective 1: acquisition utility at one point (single-query george.GP.predict(return_var=True) + epilogue)
// ------------------------------------------------------------------------------------------------------
struct UtilObj {
  int N, d, Npad, ldL;
  int all_smem;            // scaled training set AND packed L^-1 are resident in shared memory
  int oXs, oL;             // offsets of the shared copies: xs [d+1][Npad] (row d = alphaA), packed L^-1 rows
  const double* gXs;       // global fallbacks: [d][Npad] scaled SoA, [Npad] alphaA, row-major L^-1 (ld = ldL)
  const double* gAlpha;
  const double* gL;
  double amp, mean, ybest, zeta;
  int kind, has_box;
  int oLo, oHi, oQs, oE, oRed;   // shared: lo/hi/qscale [d], E [N], red [OW]

  template <bool SM>
  __device__ __forceinline__ double eval_t(int ox) const {
    extern __shared__ __align__(16) double smem_dyn[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double* x = smem_dyn + ox;
    const double* lo = smem_dyn + oLo; const double* hi = smem_dyn + oHi; const double* qscale = smem_dyn + oQs;
    double* E = smem_dyn + oE; double* red = smem_dyn + oRed;
    const double* Xs = SM ? smem_dyn + oXs : gXs;
    const double* alphaA = SM ? smem_dyn + oXs + (size_t)d * Npad : gAlpha;
    __syncthreads();                                     // x visible; previous evaluation's reads of E done
    bool ok = true;
    for (int i = 0; i < d; ++i) {
      const double v = x[i];
      ok = ok && (v == v) && (fabs(v) < INFINITY);
      if (has_box) ok = ok && (v >= lo[i]) && (v <= hi[i]);
    }
    if (!ok) return INFINITY;                            // the priorFn gate (utility.py:126,173,219)
    double part = 0.0;
    for (int j = tid; j < N; j += OT) {
      double s = 0.0;
      for (int i = 0; i < d; ++i) { const double t = Xs[(size_t)i * Npad + j] - x[i] * qscale[i]; s = fma(t, t, s); }
      const double e = exp(-s);
      E[j] = e;
      part = fma(e, alphaA[j], part);
    }
    const double mu = mean + cta_sum<OT>(part, red);         // (its barriers also publish E)
    if (kind == 4) return -mu;                           // findMAP objective: -(GP mean)
    double acc = 0.0;
    for (int i = warp; i < N; i += OW) {
      const double* Li = SM ? smem_dyn + oL + (size_t)i * (i + 1) / 2 : gL + (size_t)i * ldL;
      double s = 0.0;
      for (int j = lane; j <= i; j += 32) s = fma(Li[j], E[j], s);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const double v = amp * s;
      acc = fma(v, v, acc);                               // identical in all lanes of the warp
    }
    __syncthreads();
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    double tot = 0.0;
#pragma unroll
    for (int w = 0; w < OW; ++w) tot += red[w];
    const double var = amp - tot;
    return utility_eval(kind, mu, var, ybest, zeta);
  }

  __device__ __noinline__ double eval(int ox) const { return all_smem ? eval_t<true>(ox) : eval_t<false>(ox); }
};

// ------------------------------------------------------------------------------------------------------
// Objective 2: negative log-likelihood at one hyper-parameter vector (gpUtils._nll) behind defaultHyperPrior:
// the small evaluator of loglik.cuh, everything in this CTA's shared memory.
// ------------------------------------------------------------------------------------------------------
struct NllObj {
  int N, d, P, fit_amp, default_prior;
  double noise;            // exp(white_noise) + TINY^2

  __device__ __noinline__ double eval(int ox) const {
    extern __shared__ __align__(16) double smem_dyn[];
    const double* p = smem_dyn + ox;
    const SmallLL L = SmallLL::carve(smem_dyn, N, d);
    __syncthreads();
    if (!nll_row_finite(p, P)) return INFINITY;
    if (default_prior)                                   // gpUtils.defaultHyperPrior: |p[1:]| <= 20
      for (int k = 1; k < P; ++k) if (fabs(p[k]) > 20.0) return INFINITY;
    nll_hyp(p, d, fit_amp, noise, L.hyp);
    return -loglik_small(L, N, d, false);
  }
};

// ------------------------------------------------------------------------------------------------------
// Objective 2b: the same negative log-likelihood for training sets beyond one CTA's shared memory (N > ~220):
// a CLUSTER of C CTAs evaluates it cooperatively (chol_group.cuh: matrix in L2-resident global memory, fused
// build + look-ahead Cholesky + reductions).  Every CTA of the cluster runs the optimiser redundantly on its own
// replica of the state; the objective returns identical bits to all of them, so they stay in lock step.
// ------------------------------------------------------------------------------------------------------
struct NllGroupObj {
  int d, P, fit_amp, default_prior;
  double noise;
  CholGroup g;
  int oHyp, oTiles;         // shared: hyp [3 + d], tile buffers [CG_SMEM_DOUBLES]
  unsigned long long epoch; // evaluations that reached the factorisation (identical in every thread of the cluster)

  __device__ __noinline__ double eval(int ox) {
    extern __shared__ __align__(16) double smem_dyn[];
    const double* p = smem_dyn + ox;
    double* hyp = smem_dyn + oHyp;
    __syncthreads();
    if (!nll_row_finite(p, P)) return INFINITY;
    if (default_prior)                                   // gpUtils.defaultHyperPrior: |p[1:]| <= 20
      for (int k = 1; k < P; ++k) if (fabs(p[k]) > 20.0) return INFINITY;
    nll_hyp(p, d, fit_amp, noise, hyp);
    __syncthreads();
    const double ll = chol_group_loglik<true>(g, hyp, smem_dyn + oTiles, epoch);
    ++epoch;
    return -ll;
  }
};

// ------------------------------------------------------------------------------------------------------
// Optimiser workspace (shared memory, n = number of free variables)
// ------------------------------------------------------------------------------------------------------
struct OptWork {
  double* sim;     // NM: [(n+1)][n] simplex            Powell: direc [n][n] (+ one spare row)
  double* tmp;     // NM: [(n+1)][n] reorder scratch     Powell: unused
  double* fsim;    // NM: [n+1]
  double* v0;      // [n]  NM: xbar      Powell: x
  double* v1;      // [n]  NM: trial     Powell: x1
  double* v2;      // [n]  NM: trial 2   Powell: current direction
  double* v3;      // [n]  evaluation point
  int* perm;       // [n+1]
  const double* base;  // dynamic shared-memory base: evaluation points travel as offsets from it
  __device__ __forceinline__ int off(const double* q) const { return (int)(q - base); }
  static __host__ __device__ size_t doubles(int n) { return (size_t)2 * (n + 1) * n + (n + 1) + 4 * n + (n + 2) / 2 + 1; }
  __device__ void carve(double* base, int n) {
    sim = base; tmp = sim + (size_t)(n + 1) * n; fsim = tmp + (size_t)(n + 1) * n;
    v0 = fsim + (n + 1); v1 = v0 + n; v2 = v1 + n; v3 = v2 + n; perm = reinterpret_cast<int*>(v3 + n);
  }
};

struct OptOpts {            // resolved on the host with SciPy's default rules
  int method;               // 0 Nelder-Mead, 1 Powell
  double xtol, ftol;        // NM: xatol, fatol        Powell: xtol, ftol
  long long maxiter, maxfun;
  double c_r1, c_r2, c_e1, c_e2, c_c1, c_c2, c_cc1, c_cc2, sigma;   // NM coefficients (1+rho, rho, 1+rho*chi, ...)
};

// a < b in NumPy's sort order (NaN last)
__device__ __forceinline__ bool sort_less(double a, double b) { return a < b || (b != b && a == a); }

// stable argsort of fsim + row permutation of sim (np.argsort / np.take of _minimize_neldermead)
__device__ void nm_sort(OptWork& w, int n) {
  const int tid = threadIdx.x;
  __syncthreads();
  if (tid == 0) {
    for (int k = 0; k <= n; ++k) w.perm[k] = k;
    for (int k = 1; k <= n; ++k) {
      const int pk = w.perm[k];
      const double fk = w.fsim[pk];
      int m = k - 1;
      while (m >= 0 && sort_less(fk, w.fsim[w.perm[m]])) { w.perm[m + 1] = w.perm[m]; --m; }
      w.perm[m + 1] = pk;
    }
  }
  __syncthreads();
  for (int e = tid; e < (n + 1) * n; e += OT) { const int k = e / n, i = e - k * n; w.tmp[e] = w.sim[w.perm[k] * n + i]; }
  double fk = 0.0;
  if (tid <= n) fk = w.fsim[w.perm[tid]];
  __syncthreads();
  for (int e = tid; e < (n + 1) * n; e += OT) w.sim[e] = w.tmp[e];
  if (tid <= n) w.fsim[tid] = fk;
  __syncthreads();
}

#define NM_EV(dst, xptr)                                  \
  do {                                                    \
    if (ncalls >= o.maxfun) goto iter_end;                \
    ++ncalls;                                             \
    dst = f.eval(w.off(xptr));                                   \
  } while (0)

// scipy.optimize._optimize._minimize_neldermead; x0 in w.sim[0..n); result: w.sim[0..n), return f
template <class Obj>
__device__ double nelder_mead_dev(Obj& f, int n, const OptOpts& o, OptWork& w, long long& nfev, long long& nit) {
  const int tid = threadIdx.x;
  long long ncalls = 0, iterations = 1;
  __syncthreads();
  for (int e = tid; e < n * n; e += OT) {
    const int k = e / n, i = e - k * n;
    double v = w.sim[i];
    if (i == k) v = (v != 0.0) ? (1.0 + 0.05) * v : 0.00025;
    w.sim[(k + 1) * n + i] = v;
  }
  if (tid <= n) w.fsim[tid] = INFINITY;
  __syncthreads();
  for (int k = 0; k <= n; ++k) {
    if (ncalls >= o.maxfun) break;
    ++ncalls;
    const double v = f.eval(w.off(w.sim + k * n));
    if (tid == 0) w.fsim[k] = v;
  }
  nm_sort(w, n);
  while (ncalls < o.maxfun && iterations < o.maxiter) {
    double fxr = 0.0, fxe = 0.0, fxc = 0.0, fxcc = 0.0;
    int doshrink = 0;
    {
      // np.max(|sim[1:] - sim[0]|) <= xatol and np.max(|fsim[0] - fsim[1:]|) <= fatol  (a NaN makes it false)
      int okc = 1;
      for (int e = n + tid; e < (n + 1) * n; e += OT) {
        const double dv = fabs(w.sim[e] - w.sim[e % n]);
        if (!(dv <= o.xtol)) okc = 0;
      }
      if (tid >= 1 && tid <= n) {
        const double dv = fabs(w.fsim[0] - w.fsim[tid]);
        if (!(dv <= o.ftol)) okc = 0;
      }
      if (__syncthreads_and(okc)) break;
    }
    __syncthreads();
    if (tid < n) {                                        // xbar = add.reduce(sim[:-1], 0) / N ; xr
      double s = w.sim[tid];
      for (int k = 1; k < n; ++k) s += w.sim[k * n + tid];
      const double xb = s / (double)n;
      w.v0[tid] = xb;
      w.v1[tid] = o.c_r1 * xb - o.c_r2 * w.sim[n * n + tid];
    }
    NM_EV(fxr, w.v1);
    if (fxr < w.fsim[0]) {
      if (tid < n) w.v2[tid] = o.c_e1 * w.v0[tid] - o.c_e2 * w.sim[n * n + tid];
      NM_EV(fxe, w.v2);
      __syncthreads();
      if (fxe < fxr) { if (tid < n) w.sim[n * n + tid] = w.v2[tid]; if (tid == 0) w.fsim[n] = fxe; }
      else { if (tid < n) w.sim[n * n + tid] = w.v1[tid]; if (tid == 0) w.fsim[n] = fxr; }
    } else {
      if (fxr < w.fsim[n - 1]) {
        __syncthreads();
        if (tid < n) w.sim[n * n + tid] = w.v1[tid];
        if (tid == 0) w.fsim[n] = fxr;
      } else {
        if (fxr < w.fsim[n]) {
          if (tid < n) w.v2[tid] = o.c_c1 * w.v0[tid] - o.c_c2 * w.sim[n * n + tid];
          NM_EV(fxc, w.v2);
          __syncthreads();
          if (fxc <= fxr) { if (tid < n) w.sim[n * n + tid] = w.v2[tid]; if (tid == 0) w.fsim[n] = fxc; }
          else doshrink = 1;
        } else {
          if (tid < n) w.v2[tid] = o.c_cc1 * w.v0[tid] + o.c_cc2 * w.sim[n * n + tid];
          NM_EV(fxcc, w.v2);
          __syncthreads();
          if (fxcc < w.fsim[n]) {
            __syncthreads();                              // everyone has compared against the old fsim[n]
            if (tid < n) w.sim[n * n + tid] = w.v2[tid];
            if (tid == 0) w.fsim[n] = fxcc;
          } else doshrink = 1;
        }
        if (doshrink) {
          for (int j = 1; j <= n; ++j) {
            __syncthreads();
            if (tid < n) w.sim[j * n + tid] = w.sim[tid] + o.sigma * (w.sim[j * n + tid] - w.sim[tid]);
            double fj;
            NM_EV(fj, w.sim + j * n);
            if (tid == 0) w.fsim[j] = fj;
          }
        }
      }
    }
    ++iterations;
  iter_end:
    nm_sort(w, n);
  }
  nfev = ncalls; nit = iterations;
  __syncthreads();
  return w.fsim[0];
}
#undef NM_EV

// ---- Powell -----------------------------------------------------------------------------------------
struct PCtx { long long ncalls, maxfun; };

// f(p + alpha * xi): p = w.v0, xi = w.v2, evaluation point built in w.v3.  false = maxfun reached (SciPy raises).
template <class Obj>
__device__ __forceinline__ bool line_ev(Obj& f, int n, OptWork& w, PCtx& c, double alpha, double& out) {
  if (c.ncalls >= c.maxfun) return false;
  ++c.ncalls;
  __syncthreads();
  if (threadIdx.x < n) w.v3[threadIdx.x] = w.v0[threadIdx.x] + alpha * w.v2[threadIdx.x];
  out = f.eval(w.off(w.v3));
  return true;
}

// scipy.optimize.bracket(func, xa=0, xb=1); status 0 valid, 1 invalid bracket, 2 aborted (maxfun)
template <class Obj>
__device__ int bracket_dev(Obj& f, int n, OptWork& w, PCtx& c, double& xa, double& xb, double& xc, double& fa,
                           double& fb, double& fc) {
  const double gold = 1.618034, verysmall = 1e-21, grow_limit = 110.0;
  xa = 0.0; xb = 1.0;
  if (!line_ev(f, n, w, c, xa, fa)) return 2;
  if (!line_ev(f, n, w, c, xb, fb)) return 2;
  if (fa < fb) { double t = xa; xa = xb; xb = t; t = fa; fa = fb; fb = t; }
  xc = xb + gold * (xb - xa);
  if (!line_ev(f, n, w, c, xc, fc)) return 2;
  int it = 0;
  while (fc < fb) {
    const double tmp1 = (xb - xa) * (fb - fc);
    const double tmp2 = (xb - xc) * (fb - fa);
    const double val = tmp2 - tmp1;
    const double denom = (fabs(val) < verysmall) ? 2.0 * verysmall : 2.0 * val;
    double wv = xb - ((xb - xc) * tmp2 - (xb - xa) * tmp1) / denom;
    const double wlim = xb + grow_limit * (xc - xb);
    if (it > 1000) return 1;
    ++it;
    double fw;
    if ((wv - xc) * (xb - wv) > 0.0) {
      if (!line_ev(f, n, w, c, wv, fw)) return 2;
      if (fw < fc) { xa = xb; xb = wv; fa = fb; fb = fw; break; }
      else if (fw > fb) { xc = wv; fc = fw; break; }
      wv = xc + gold * (xc - xb);
      if (!line_ev(f, n, w, c, wv, fw)) return 2;
    } else if ((wv - wlim) * (wlim - xc) >= 0.0) {
      wv = wlim;
      if (!line_ev(f, n, w, c, wv, fw)) return 2;
    } else if ((wv - wlim) * (xc - wv) > 0.0) {
      if (!line_ev(f, n, w, c, wv, fw)) return 2;
      if (fw < fc) {
        xb = xc; xc = wv; wv = xc + gold * (xc - xb); fb = fc; fc = fw;
        if (!line_ev(f, n, w, c, wv, fw)) return 2;
      }
    } else {
      wv = xc + gold * (xc - xb);
      if (!line_ev(f, n, w, c, wv, fw)) return 2;
    }
    xa = xb; xb = xc; xc = wv; fa = fb; fb = fc; fc = fw;
  }
  const bool cond1 = (fb < fc && fb <= fa) || (fb < fa && fb <= fc);
  const bool cond2 = (xa < xb && xb < xc) || (xc < xb && xb < xa);
  const bool cond3 = (fabs(xa) < INFINITY) && (fabs(xb) < INFINITY) && (fabs(xc) < INFINITY);
  return (cond1 && cond2 && cond3) ? 0 : 1;
}

// Brent's line minimisation as _linesearch_powell drives it (bracket, then Brent.optimize; an invalid bracket
// falls back to its best point).  false = aborted by maxfun.
template <class Obj>
__device__ bool brent_dev(Obj& f, int n, OptWork& w, PCtx& c, double tol, double& xmin, double& fmin) {
  double xa, xb, xc, fa, fb, fc;
  const int st = bracket_dev(f, n, w, c, xa, xb, xc, fa, fb, fc);
  if (st == 2) return false;
  if (st == 1) {
    if (xa != xa || xb != xb || xc != xc || fa != fa || fb != fb || fc != fc) { xmin = NAN; fmin = NAN; return true; }
    xmin = xa; fmin = fa;
    if (fb < fmin) { xmin = xb; fmin = fb; }
    if (fc < fmin) { xmin = xc; fmin = fc; }
    return true;
  }
  const double mintol = 1.0e-11, cg = 0.3819660;
  double x = xb, wv = xb, v = xb, fx = fb, fw = fb, fv = fb, a, b, deltax = 0.0, rat = 0.0, u, fu;
  if (xa < xc) { a = xa; b = xc; } else { a = xc; b = xa; }
  int it = 0;
  while (it < 500) {
    const double tol1 = tol * fabs(x) + mintol;
    const double tol2 = 2.0 * tol1;
    const double xmid = 0.5 * (a + b);
    if (fabs(x - xmid) < (tol2 - 0.5 * (b - a))) break;
    if (fabs(deltax) <= tol1) {
      deltax = (x >= xmid) ? (a - x) : (b - x);
      rat = cg * deltax;
    } else {
      const double tmp1 = (x - wv) * (fx - fv);
      double tmp2 = (x - v) * (fx - fw);
      double p = (x - v) * tmp2 - (x - wv) * tmp1;
      tmp2 = 2.0 * (tmp2 - tmp1);
      if (tmp2 > 0.0) p = -p;
      tmp2 = fabs(tmp2);
      const double dx_temp = deltax;
      deltax = rat;
      if ((p > tmp2 * (a - x)) && (p < tmp2 * (b - x)) && (fabs(p) < fabs(0.5 * tmp2 * dx_temp))) {
        rat = p * 1.0 / tmp2;
        u = x + rat;
        if ((u - a) < tol2 || (b - u) < tol2) rat = (xmid - x >= 0) ? tol1 : -tol1;
      } else {
        deltax = (x >= xmid) ? (a - x) : (b - x);
        rat = cg * deltax;
      }
    }
    if (fabs(rat) < tol1) u = (rat >= 0) ? x + tol1 : x - tol1;
    else u = x + rat;
    if (!line_ev(f, n, w, c, u, fu)) return false;
    if (fu > fx) {
      if (u < x) a = u; else b = u;
      if ((fu <= fw) || (wv == x)) { v = wv; wv = u; fv = fw; fw = fu; }
      else if ((fu <= fv) || (v == x) || (v == wv)) { v = u; fv = fu; }
    } else {
      if (u >= x) a = x; else b = x;
      v = wv; wv = x; x = u; fv = fw; fw = fx; fx = fu;
    }
    ++it;
  }
  xmin = x; fmin = fx;
  return true;
}

// _linesearch_powell (unbounded): minimise along w.v2 from w.v0; on success w.v2 <- alpha*xi, w.v0 <- p + xi
template <class Obj>
__device__ bool linesearch_dev(Obj& f, int n, OptWork& w, PCtx& c, double tol, double& fval) {
  __syncthreads();
  bool any = false;
  for (int i = 0; i < n; ++i) any = any || (w.v2[i] != 0.0);       // np.any(xi) (NaN counts as nonzero)
  if (!any) return true;
  double amin, fret;
  if (!brent_dev(f, n, w, c, tol, amin, fret)) return false;
  __syncthreads();
  if (threadIdx.x < n) {
    const double xi = amin * w.v2[threadIdx.x];
    w.v2[threadIdx.x] = xi;
    w.v0[threadIdx.x] = w.v0[threadIdx.x] + xi;
  }
  __syncthreads();
  fval = fret;
  return true;
}

// scipy.optimize._optimize._minimize_powell (no bounds); x0 in w.v0; result in w.v0, returns f
template <class Obj>
__device__ double powell_dev(Obj& f, int n, const OptOpts& o, OptWork& w, long long& nfev, long long& nit) {
  const int tid = threadIdx.x;
  PCtx c{0, o.maxfun};
  double* direc = w.sim;
  __syncthreads();
  for (int e = tid; e < n * n; e += OT) direc[e] = ((e / n) == (e % n)) ? 1.0 : 0.0;
  if (tid < n) w.v1[tid] = w.v0[tid];                    // x1 = x.copy()
  __syncthreads();
  double fval = 0.0;
  long long it = 0;
  if (c.ncalls >= c.maxfun) { nfev = 0; nit = 0; return fval; }
  ++c.ncalls;
  fval = f.eval(w.off(w.v0));
  while (true) {
    const double fx = fval;
    int bigind = 0;
    double delta = 0.0;
    bool aborted = false;
    for (int i = 0; i < n; ++i) {
      __syncthreads();
      if (tid < n) w.v2[tid] = direc[i * n + tid];
      const double fx2 = fval;
      if (!linesearch_dev(f, n, w, c, o.xtol * 100.0, fval)) { aborted = true; break; }
      if ((fx2 - fval) > delta) { delta = fx2 - fval; bigind = i; }
    }
    if (aborted) break;
    ++it;
    const double bnd = o.ftol * (fabs(fx) + fabs(fval)) + 1e-20;
    if (2.0 * (fx - fval) <= bnd) break;
    if (c.ncalls >= c.maxfun) break;
    if (it >= o.maxiter) break;
    if (fx != fx && fval != fval) break;
    __syncthreads();
    if (tid < n) {                                        // direc1 = x - x1 ; x1 = x ; x2 = x + direc1
      const double xv = w.v0[tid];
      const double d1 = xv - w.v1[tid];
      w.v2[tid] = d1;
      w.v1[tid] = xv;
      w.v3[tid] = xv + d1;
    }
    if (c.ncalls >= c.maxfun) break;
    ++c.ncalls;
    const double fx2 = f.eval(w.off(w.v3));
    if (fx > fx2) {
      double t = 2.0 * (fx + fx2 - 2.0 * fval);
      double temp = (fx - fval - delta);
      t *= temp * temp;
      temp = fx - fx2;
      t -= delta * temp * temp;
      if (t < 0.0) {
        if (!linesearch_dev(f, n, w, c, o.xtol * 100.0, fval)) break;
        bool any = false;
        for (int i = 0; i < n; ++i) any = any || (w.v2[i] != 0.0);
        if (any) {
          __syncthreads();
          if (tid < n) { direc[bigind * n + tid] = direc[(n - 1) * n + tid]; }
          __syncthreads();
          if (tid < n) { direc[(n - 1) * n + tid] = w.v2[tid]; }
          __syncthreads();
        }
      }
    }
  }
  nfev = c.ncalls; nit = it;
  __syncthreads();
  return fval;
}

// ------------------------------------------------------------------------------------------------------
// Kernels: one CTA per start.  mode 0 = evaluate the objective at the given points only (test hook: the
// host restatement of the optimisers can then be driven by exactly the function the device minimises).
// ------------------------------------------------------------------------------------------------------
struct UtilKernelParams {
  int N, d, Npad, ldL, all_smem;
  const double* Xs; const double* alphaA; const double* Linv;
  double amp, mean, ybest, zeta;
  int kind, has_box;
  double lo[APGP_MAXD], hi[APGP_MAXD], qscale[APGP_MAXD];
  const double* x0;        // [R][d]
  double* x_out;           // [R][d]
  double* f_out;           // [R]
  long long* stats;        // [R][3] nfev, nit, SM cycles
  int mode;                // 0 evaluate, 1 minimise
  OptOpts opt;
};

__global__ void __launch_bounds__(OT, 1) minimize_utility_kernel(const __grid_constant__ UtilKernelParams p) {
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, n = p.d;
  double* cur = sm;
  double* lo = cur; cur += n; double* hi = cur; cur += n; double* qs = cur; cur += n;
  double* E = cur; cur += p.N;
  double* red = cur; cur += OW;
  OptWork w; w.carve(cur, n); w.base = sm; cur += OptWork::doubles(n);
  UtilObj f;
  f.N = p.N; f.d = n; f.Npad = p.Npad; f.ldL = p.ldL; f.all_smem = p.all_smem;
  f.gXs = p.Xs; f.gAlpha = p.alphaA; f.gL = p.Linv;
  f.amp = p.amp; f.mean = p.mean; f.ybest = p.ybest; f.zeta = p.zeta; f.kind = p.kind; f.has_box = p.has_box;
  f.oLo = (int)(lo - sm); f.oHi = (int)(hi - sm); f.oQs = (int)(qs - sm); f.oE = (int)(E - sm); f.oRed = (int)(red - sm);
  f.oXs = 0; f.oL = 0;
  if (p.all_smem) {                                      // resident copies: scaled training set (+ alpha row), packed L^-1
    double* xs = cur; cur += (size_t)(n + 1) * p.Npad;
    for (int e = tid; e < n * p.Npad; e += OT) xs[e] = p.Xs[e];
    for (int e = tid; e < p.Npad; e += OT) xs[(size_t)n * p.Npad + e] = p.alphaA[e];
    f.oXs = (int)(xs - sm);
    if (p.kind != 4) {
      double* lp = cur;
      for (int i = tid >> 5; i < p.N; i += OW) {
        const double* src = p.Linv + (size_t)i * p.ldL;
        double* dst = lp + (size_t)i * (i + 1) / 2;
        for (int j = tid & 31; j <= i; j += 32) dst[j] = src[j];
      }
      f.oL = (int)(lp - sm);
    }
  }
  if (tid < n) { lo[tid] = p.lo[tid]; hi[tid] = p.hi[tid]; qs[tid] = p.qscale[tid]; }
  const double* x0 = p.x0 + (size_t)blockIdx.x * n;
  double* start = (p.opt.method == 1 && p.mode == 1) ? w.v0 : w.sim;
  if (tid < n) start[tid] = x0[tid];
  __syncthreads();
  double fbest; long long nfev = 1, nit = 0;
  const long long t_start = clock64();
  if (p.mode == 0) fbest = f.eval(w.off(start));
  else if (p.opt.method == 0) fbest = nelder_mead_dev(f, n, p.opt, w, nfev, nit);
  else fbest = powell_dev(f, n, p.opt, w, nfev, nit);
  __syncthreads();
  if (tid < n) p.x_out[(size_t)blockIdx.x * n + tid] = start[tid];
  if (tid == 0) {
    p.f_out[blockIdx.x] = fbest;
    if (p.stats) { p.stats[3 * blockIdx.x] = nfev; p.stats[3 * blockIdx.x + 1] = nit; p.stats[3 * blockIdx.x + 2] = clock64() - t_start; }
  }
}

struct NllKernelParams {
  int N, d, P, fit_amp, default_prior;
  double noise;
  const double* X; const double* y;
  const double* p0;        // [R][P]
  double* p_out;           // [R][P]
  double* f_out;           // [R]
  long long* stats;        // [R][3]
  int mode;
  OptOpts opt;
};

__global__ void __launch_bounds__(OT, 1) minimize_nll_kernel(const __grid_constant__ NllKernelParams p) {
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, n = p.P;
  const SmallLL L = SmallLL::carve(sm, p.N, p.d);
  OptWork w; w.carve(sm + SmallLL::doubles(p.N, p.d), n); w.base = sm;
  for (int e = tid; e < p.N * p.d; e += OT) L.X[e] = p.X[e];
  for (int e = tid; e < p.N; e += OT) L.y[e] = p.y[e];
  NllObj f{p.N, p.d, p.P, p.fit_amp, p.default_prior, p.noise};
  const double* x0 = p.p0 + (size_t)blockIdx.x * n;
  double* start = (p.opt.method == 1 && p.mode == 1) ? w.v0 : w.sim;
  if (tid < n) start[tid] = x0[tid];
  __syncthreads();
  double fbest; long long nfev = 1, nit = 0;
  const long long t_start = clock64();
  if (p.mode == 0) fbest = f.eval(w.off(start));
  else if (p.opt.method == 0) fbest = nelder_mead_dev(f, n, p.opt, w, nfev, nit);
  else fbest = powell_dev(f, n, p.opt, w, nfev, nit);
  __syncthreads();
  if (tid < n) p.p_out[(size_t)blockIdx.x * n + tid] = start[tid];
  if (tid == 0) {
    p.f_out[blockIdx.x] = fbest;
    if (p.stats) { p.stats[3 * blockIdx.x] = nfev; p.stats[3 * blockIdx.x + 1] = nit; p.stats[3 * blockIdx.x + 2] = clock64() - t_start; }
  }
}

struct NllGroupKernelParams {
  int N, d, Np, P, fit_amp, default_prior, C;
  double noise;
  const double* X; const double* y;
  GroupWs ws;
  const double* p0; double* p_out; double* f_out; long long* stats;
  int mode;
  OptOpts opt;
};

__global__ void __launch_bounds__(OT, 1) minimize_nll_group_kernel(const __grid_constant__ NllGroupKernelParams p) {
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, n = p.P;
  const int rr = blockIdx.x / p.C;
  const int rank = (p.C > 1) ? cg_cluster_ctarank() : 0;
  double* cur = sm;
  double* tiles = cur; cur += CG_SMEM_DOUBLES;
  double* hyp = cur; cur += 4 + APGP_MAXD;
  OptWork w; w.carve(cur, n); w.base = sm;
  NllGroupObj f;
  f.d = p.d; f.P = p.P; f.fit_amp = p.fit_amp; f.default_prior = p.default_prior; f.noise = p.noise;
  f.g = cg_make(p.ws, rr, p.N, p.Np, p.d, p.C, rank, p.X, p.y);
  f.oHyp = (int)(hyp - sm); f.oTiles = (int)(tiles - sm); f.epoch = 0ull;
  const double* x0 = p.p0 + (size_t)rr * n;
  double* start = (p.opt.method == 1 && p.mode == 1) ? w.v0 : w.sim;
  if (tid < n) start[tid] = x0[tid];
  __syncthreads();
  double fbest; long long nfev = 1, nit = 0;
  const long long t_start = clock64();
  if (p.mode == 0) fbest = f.eval(w.off(start));
  else if (p.opt.method == 0) fbest = nelder_mead_dev(f, n, p.opt, w, nfev, nit);
  else fbest = powell_dev(f, n, p.opt, w, nfev, nit);
  __syncthreads();
  if (rank == 0) {
    if (tid < n) p.p_out[(size_t)rr * n + tid] = start[tid];
    if (tid == 0) {
      p.f_out[rr] = fbest;
      if (p.stats) { p.stats[3 * rr] = nfev; p.stats[3 * rr + 1] = nit; p.stats[3 * rr + 2] = clock64() - t_start; }
    }
  }
}

constexpr size_t SMEM_CAP = 220 * 1024;
PerDeviceOnce g_opt_attr;
int ensure_opt_attrs() {
  if (!g_opt_attr.needed()) return 0;
  cudaError_t e;
  e = cudaFuncSetAttribute(minimize_utility_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_CAP); if (e) return (int)e;
  e = cudaFuncSetAttribute(minimize_nll_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_CAP); if (e) return (int)e;
  e = cudaFuncSetAttribute(minimize_nll_group_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_CAP); if (e) return (int)e;
  e = cudaFuncSetAttribute(minimize_nll_group_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1); if (e) return (int)e;
  g_opt_attr.mark();
  return 0;
}

void fill_opt(OptOpts& o, const OptimizeParams& q, int n) {
  o.method = q.method; o.xtol = q.xtol; o.ftol = q.ftol; o.maxiter = q.maxiter; o.maxfun = q.maxfun;
  // coefficients exactly as SciPy forms them (Python floats): rho = 1; adaptive: chi = 1 + 2/dim,
  // psi = 0.75 - 1/(2 dim), sigma = 1 - 1/dim; else chi = 2, psi = 0.5, sigma = 0.5
  const double dim = (double)n;
  const double rho = 1.0;
  const double chi = q.adaptive ? 1.0 + 2.0 / dim : 2.0;
  const double psi = q.adaptive ? 0.75 - 1.0 / (2.0 * dim) : 0.5;
  const double sigma = q.adaptive ? 1.0 - 1.0 / dim : 0.5;
  o.c_r1 = 1.0 + rho; o.c_r2 = rho;
  o.c_e1 = 1.0 + rho * chi; o.c_e2 = rho * chi;
  o.c_c1 = 1.0 + psi * rho; o.c_c2 = psi * rho;
  o.c_cc1 = 1.0 - psi; o.c_cc2 = psi;
  o.sigma = sigma;
}

}  // namespace

size_t minimize_nll_smem(int N, int d, int P) {
  return (SmallLL::doubles(N, d) + OptWork::doubles(P)) * sizeof(double);
}
bool minimize_nll_fits(int N, int d, int P) { return minimize_nll_smem(N, d, P) <= SMEM_CAP && P + 1 <= OT && N < OT; }

#ifdef APGP_PROF
int read_prof(long long* out16) {
  cudaError_t e = cudaMemcpyFromSymbol(out16, g_prof, sizeof(long long) * 16);
  long long z[16] = {};
  cudaMemcpyToSymbol(g_prof, z, sizeof(z));
  return (int)e;
}
#else
int read_prof(long long* out16) { for (int i = 0; i < 16; ++i) out16[i] = 0; return 0; }
#endif

int launch_minimize_utility(const UtilityPointParams& u, const OptimizeParams& q, int R, const double* x0_dev,
                            double* x_out_dev, double* f_out_dev, long long* stats_dev, int mode, cudaStream_t st) {
  int e = ensure_opt_attrs(); if (e) return e;
  UtilKernelParams p;
  p.N = u.N; p.d = u.d; p.Npad = u.Npad; p.ldL = u.ldL;
  p.Xs = u.Xs; p.alphaA = u.alphaA; p.Linv = u.Linv;
  p.amp = u.amp; p.mean = u.mean; p.ybest = u.ybest; p.zeta = u.zeta; p.kind = u.kind; p.has_box = u.has_box;
  for (int i = 0; i < u.d; ++i) { p.lo[i] = u.lo[i]; p.hi[i] = u.hi[i]; p.qscale[i] = u.qscale[i]; }
  p.x0 = x0_dev; p.x_out = x_out_dev; p.f_out = f_out_dev; p.stats = stats_dev; p.mode = mode;
  fill_opt(p.opt, q, u.d);
  // shared-memory plan: fixed part, then -- if both fit -- the scaled training set and the packed L^-1
  size_t base = ((size_t)3 * u.d + u.N + OW + OptWork::doubles(u.d)) * 8;
  const size_t xs_b = (size_t)(u.d + 1) * u.Npad * 8;
  const size_t lp_b = (size_t)u.N * (u.N + 1) / 2 * 8;
  const size_t resident = xs_b + (u.kind != 4 ? lp_b : 0);
  p.all_smem = (base + resident <= SMEM_CAP) ? 1 : 0;     // else the objective streams both from global (L2)
  if (p.all_smem) base += resident;
  minimize_utility_kernel<<<R, OT, base, st>>>(p);
  return (int)cudaGetLastError();
}

int launch_minimize_nll(const double* X_dev, const double* y_dev, int N, int d, int P, int fit_amp, int default_prior,
                        double noise, const OptimizeParams& q, int R, const double* p0_dev, double* p_out_dev,
                        double* f_out_dev, long long* stats_dev, int mode, cudaStream_t st) {
  int e = ensure_opt_attrs(); if (e) return e;
  NllKernelParams p;
  p.N = N; p.d = d; p.P = P; p.fit_amp = fit_amp; p.default_prior = default_prior; p.noise = noise;
  p.X = X_dev; p.y = y_dev; p.p0 = p0_dev; p.p_out = p_out_dev; p.f_out = f_out_dev; p.stats = stats_dev; p.mode = mode;
  fill_opt(p.opt, q, P);
  minimize_nll_kernel<<<R, OT, minimize_nll_smem(N, d, P), st>>>(p);
  return (int)cudaGetLastError();
}

size_t minimize_nll_group_smem(int P) { return (CG_SMEM_DOUBLES + 4 + APGP_MAXD + OptWork::doubles(P)) * sizeof(double); }
bool minimize_nll_group_fits(int P) { return minimize_nll_group_smem(P) <= SMEM_CAP && P + 1 <= OT; }

// One CLUSTER of C CTAs per restart; ws_bytes: chol_group_ws_bytes(Np, R).  Same contract as launch_minimize_nll.
int launch_minimize_nll_group(const double* X_dev, const double* y_dev, int N, int d, int Np, int P, int fit_amp,
                              int default_prior, double noise, const OptimizeParams& q, int R, int num_sms, void* ws_bytes,
                              const double* p0_dev, double* p_out_dev, double* f_out_dev, long long* stats_dev, int mode,
                              cudaStream_t st) {
  int e = ensure_opt_attrs(); if (e) return e;
  NllGroupKernelParams p;
  p.N = N; p.d = d; p.Np = Np; p.P = P; p.fit_amp = fit_amp; p.default_prior = default_prior; p.noise = noise;
  p.X = X_dev; p.y = y_dev; p.ws = cg_ws_carve(ws_bytes, Np, R);
  p.p0 = p0_dev; p.p_out = p_out_dev; p.f_out = f_out_dev; p.stats = stats_dev; p.mode = mode;
  fill_opt(p.opt, q, P);
  cudaError_t ce = cudaMemsetAsync(p.ws.flags, 0, (size_t)R * 16, st);
  if (ce != cudaSuccess) return (int)ce;
  int C = chol_group_cluster(Np, R, num_sms);
  for (;;) {
    p.C = C;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(R * C)); cfg.blockDim = dim3(OT);
    cfg.dynamicSmemBytes = minimize_nll_group_smem(P); cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, minimize_nll_group_kernel, p);
    if (ce == cudaSuccess || C == 1) break;
    (void)cudaGetLastError();
    C >>= 1;
  }
  return (int)ce;
}

}  // namespace apgp
