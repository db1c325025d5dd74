// Device building blocks of the tiled variance kernels: predict_var_kernel and predict_var_group_kernel (predict.cu,
// FP64 DMMA) and predict_var_i8_kernel (predict_i8.cu, int8 tensor cores).
//
// Phase 1 -- the kernel values E[q,j] of a query tile, their contribution to the mean, and the panel that phase 2
// multiplies -- is written once here.  The kernels differ only in how they store the panel (a store functor), so
// all three compute the same E and the same mean in the same order: the int8 engine's mean is the DMMA engine's mean
// by construction.  Phase 2's operand stream (stream_operands: panel and B operand through the mbarrier ring) is
// shared too; the kernels differ in the stage sizes and in how they consume a stage (the two DMMA kernels share one
// block-row, dmma_block_row in predict.cu).  The grouped kernels also share their group scaffold (GroupCtx, and
// launch_grouped on the host) and the per-query output.
#pragma once
#include "apgp_internal.h"

namespace apgp {

// the tile's scaled queries, qs[i][m] = Xq[q0 + m][i] * qscale[i] (0 beyond Q), staged by the NCONS builder threads
template <int BM, int NCONS>
__device__ __forceinline__ void stage_queries(double* qs, const PredictParams& p, int d, long long q0, int tid) {
  for (int e = tid; e < d * BM; e += NCONS) {
    int i = e / BM, m = e - i * BM;
    long long q = q0 + m;
    qs[e] = (q < p.Q) ? p.Xq[q * d + i] * p.qscale[i] : 0.0;
  }
}

// Phase 1 over ncols (a multiple of 16) staged training columns: xs[i * ld + j] the scaled inputs, al[j] alpha.
// Warp w builds the m8 query blocks w, w + NCW, ... (their exp chains interleave: 4R-way ILP); lane l holds query row
// l / 4 of each block and, in the 16-wide step jb, the columns jb + l % 4 + {0, 4, 8, 12} -- the DMMA A-fragment
// order.  Adds E . alpha to macc and hands each block's four kernel values to store(jb, mb, e).
template <int BM, int NCW, class Store>
__device__ __forceinline__ void panel_columns(const double* xs, int ld, const double* al, int ncols, const double* qs,
                                              int d, const double* etab, int warp, int lane,
                                              double (&macc)[BM / (8 * NCW)], Store&& store) {
  constexpr int R = BM / (8 * NCW);
  for (int jb = 0; jb < ncols; jb += 16) {
    const int jj = jb + (lane & 3);
    double s[R][4] = {};
    for (int i = 0; i < d; ++i) {
      const double* xr = xs + i * ld + jj;
      const double x0 = xr[0], x1 = xr[4], x2 = xr[8], x3 = xr[12];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const double qv = qs[i * BM + (warp + r * NCW) * 8 + (lane >> 2)];
        const double d0 = x0 - qv, d1 = x1 - qv, d2 = x2 - qv, d3 = x3 - qv;
        s[r][0] = fma(d0, d0, s[r][0]); s[r][1] = fma(d1, d1, s[r][1]);
        s[r][2] = fma(d2, d2, s[r][2]); s[r][3] = fma(d3, d3, s[r][3]);
      }
    }
    const double a0 = al[jj], a1 = al[jj + 4], a2 = al[jj + 8], a3 = al[jj + 12];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      double e[4];
      e[0] = exp_neg(s[r][0], etab); e[1] = exp_neg(s[r][1], etab);
      e[2] = exp_neg(s[r][2], etab); e[3] = exp_neg(s[r][3], etab);
      macc[r] = fma(e[0], a0, macc[r]); macc[r] = fma(e[1], a1, macc[r]);
      macc[r] = fma(e[2], a2, macc[r]); macc[r] = fma(e[3], a3, macc[r]);
      store(jb, warp + r * NCW, e);
    }
  }
}

// the DMMA kernels' panel: doubles in A-fragment order, [k4 block of column col][m8 block mb][lane]
template <int BM>
__device__ __forceinline__ void store_dmma_panel(double* panel, int col, int mb, int lane, const double (&e)[4]) {
  double* dst = panel + ((size_t)(col >> 2) * (BM / 8) + mb) * 32 + lane;
  dst[0] = e[0]; dst[(BM / 8) * 32] = e[1]; dst[2 * (BM / 8) * 32] = e[2]; dst[3 * (BM / 8) * 32] = e[3];
}

// per-lane partial sums of panel_columns' query rows, added over the four lanes of each row and stored per query
template <int R, int NCW>
__device__ __forceinline__ void store_row_sums(const double (&v)[R], double* dst, int warp, int lane) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    double t = v[r];
    t += __shfl_xor_sync(0xffffffffu, t, 1);
    t += __shfl_xor_sync(0xffffffffu, t, 2);
    if ((lane & 3) == 0) dst[(warp + r * NCW) * 8 + (lane >> 2)] = t;
  }
}

// one query's outputs: mean, variance, and the utility (+inf outside the prior box).  d is the caller's copy of p.d:
// reading it again from the parameter space here costs the few-query kernel 8 registers
__device__ __forceinline__ void write_query(const PredictParams& p, int d, long long q, double mu, double var) {
  if (p.mu) p.mu[q] = mu;
  if (p.var) p.var[q] = var;
  if (p.util) {
    bool ok = true;
    if (p.has_box) {
      for (int i = 0; i < d; ++i) {
        const double x = p.Xq[q * d + i];
        ok = ok && (x >= p.lo[i]) && (x <= p.hi[i]);
      }
    }
    p.util[q] = ok ? utility_eval(p.utility_kind, mu, var, p.ybest, p.zeta) : INFINITY;
  }
}

// The prologue every tiled kernel shares: the 2^(j/64) table of exp_neg, and the mbarriers of the NSTAGE operand ring
// (full: the producer's expect_tx; empty: ncons consumer arrivals) and of phase 1's training-set staging.  The fence
// also covers barriers the caller initialised before it.  The caller synchronises the CTA afterwards.
template <int NSTAGE>
__device__ __forceinline__ void init_tile_smem(double* etab, uint64_t* full, uint64_t* empty, uint64_t* stagebar,
                                               uint32_t ncons) {
  const int tid = threadIdx.x;
  if (tid < 64) etab[tid] = exp2((double)tid * (1.0 / 64.0));
  if (tid == 0) {
    for (int s = 0; s < NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], ncons); }
    mbar_init(stagebar, 1);
    mbar_fence_init();
  }
}

// Phase 2's operand stream, run by the producer lane: for every block-row ib with mine(ib), its (ib + 1) KPB k-stages
// (KPB per block-row height) through the NSTAGE ring, each one A_BYTES of the panel a followed by B_BYTES of the
// block-row's B operand, which starts KPB ib(ib + 1)/2 stages into b.  it: the ring position, advanced in the same
// sequence by the consumers.
template <int NSTAGE, int A_BYTES, int B_BYTES, int KPB, class Mine>
__device__ __forceinline__ void stream_operands(void* ring, const void* a, const void* b, int nblk, uint64_t* full,
                                                uint64_t* empty, uint32_t& it, Mine&& mine) {
  unsigned char* const ring8 = static_cast<unsigned char*>(ring);
  const unsigned char* const a8 = static_cast<const unsigned char*>(a);
  for (int ib = 0; ib < nblk; ++ib) {
    if (!mine(ib)) continue;
    const int nk = (ib + 1) * KPB;
    const unsigned char* bsrc = static_cast<const unsigned char*>(b) + (size_t)KPB * ((size_t)ib * (ib + 1) / 2) * B_BYTES;
    for (int kb = 0; kb < nk; ++kb, ++it) {
      const int s = it % NSTAGE;
      const uint32_t ph = (it / NSTAGE) & 1u;
      mbar_wait(&empty[s], ph ^ 1u);
      unsigned char* dst = ring8 + (size_t)s * (A_BYTES + B_BYTES);
      mbar_arrive_expect_tx(&full[s], A_BYTES + B_BYTES);
      bulk_g2s(dst, a8 + (size_t)kb * A_BYTES, A_BYTES, &full[s]);
      bulk_g2s(dst + A_BYTES, bsrc + (size_t)kb * B_BYTES, B_BYTES, &full[s]);
    }
  }
}

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---------------------------------------------------------------------------------------------
// Group scaffold of the grouped kernels (predict.cu describes the scheme): G consecutive CTAs, the ranks of a group,
// share each query tile of the group's contiguous range.  Per tile: phase 1 (group_phase1), one barrier, the
// finaliser of the previous tile, phase 2.  Partial sums are kept per 64-column block (mean) and per block-row
// (variance) and added in block order by the finaliser, so a query's result does not depend on which rank -- or how
// large a group -- computed the pieces.
// ---------------------------------------------------------------------------------------------
template <int BM, int BN>
struct GroupCtx {
  int nblk, grp, rank, gs;
  long long t_begin, t_end;      // the group's tiles
  int sl0, sl1;                  // my slice of each tile's queries (finaliser)
  int* arrive;                   // the group's barrier counter
  double* part_mu;               // [2 buffers][nblk][BM]
  double* part_ss;               // [2 buffers][nblk][BM]

  __device__ __forceinline__ GroupCtx(const PredictParams& p, int G) {
    nblk = p.Npad / BN;
    grp = blockIdx.x / G; rank = blockIdx.x % G;
    gs = min(G, (int)gridDim.x - grp * G);                 // ranks in my group
    const long long ntiles = (p.Q + BM - 1) / BM;
    // contiguous share of the tiles, proportional to the group's size; rounding up hands the odd tiles to the first
    // (full-size) groups -- a single-tile call must not land on the smaller last group
    t_begin = (ntiles * (long long)(grp * G) + gridDim.x - 1) / gridDim.x;
    t_end = (ntiles * (long long)(grp * G + gs) + gridDim.x - 1) / gridDim.x;
    sl0 = BM * rank / gs; sl1 = BM * (rank + 1) / gs;
    arrive = p.grp_arrive + grp;
    part_mu = p.grp_part + (size_t)grp * 4 * nblk * BM;
    part_ss = part_mu + (size_t)2 * nblk * BM;
  }

  // work split planned on the host (plan_group_split): full groups use table 0, a smaller last group table 1.
  // owner_s[ib]: the rank of block-row ib (phase 2); myblk_s[0 .. *nmine_s): the 64-column blocks I build (phase 1)
  __device__ __forceinline__ void load_plan(const PredictParams& p, int G, int* owner_s, int* myblk_s, int* nmine_s) const {
    const int* tab = p.grp_plan + (gs == G ? 0 : 2 * GROUP_MAX_BLOCKS);
    for (int e = threadIdx.x; e < nblk; e += blockDim.x) owner_s[e] = tab[e];
    if (threadIdx.x == 0) {
      int n = 0;
      for (int e = 0; e < nblk; ++e) if (tab[GROUP_MAX_BLOCKS + e] == rank) myblk_s[n++] = e;
      *nmine_s = n;
    }
  }

  // the group barrier, one per tile (arrival counter in global memory, acquire spin, co-resident grid): everything
  // the group wrote before it -- panel, partial sums -- is visible to every rank after it, TMA reads included
  __device__ __forceinline__ void barrier(int& nbar) const {
    if (threadIdx.x == 0) {
      ++nbar;
      __threadfence();                                   // cumulative: everything this CTA wrote before the bar.sync
      atomicAdd(arrive, 1);
      const int target = nbar * gs;
      while (ld_acquire_gpu(arrive) < target) __nanosleep(40);
      __threadfence();
    }
    __syncthreads();
    fence_proxy_async();                                 // other CTAs' panel stores (generic proxy) -> our TMA reads
  }

  // Finalise my slice of the previous tile and keep this tile's complete means in mu_keep[b] (live: a tile is being
  // built).  var_of(mu, rowsum) gives the variance.
  template <class VarOf>
  __device__ __forceinline__ void finalise(const PredictParams& p, long long tile, bool live, int b,
                                           double (*mu_keep)[BM], VarOf&& var_of) const {
    const int tid = threadIdx.x;
    const int m = sl0 + tid;
    if (tid < sl1 - sl0) {
      if (live) {
        double mu = 0.0;
        for (int cb = 0; cb < nblk; ++cb) mu += __ldcg(part_mu + ((size_t)b * nblk + cb) * BM + m);
        mu_keep[b][tid] = mu;
      }
      if (tile > t_begin) {
        const long long q = (tile - 1) * BM + m;
        if (q < p.Q) {
          double tot = 0.0;
          for (int ib = 0; ib < nblk; ++ib) tot += __ldcg(part_ss + ((size_t)(b ^ 1) * nblk + ib) * BM + m);
          const double mu = p.mean + mu_keep[b ^ 1][tid];
          write_query(p, p.d, q, mu, var_of(mu, tot));
        }
      }
    }
  }
};

// Phase 1 of the grouped kernels for the tile starting at query q0: my 64-column blocks of the panel, staged up to 8
// per round (d + 1 bulk copies each) in stg, the idle operand ring of stg_doubles doubles, and each block's partial
// means into part_mu[block][BM] (the tile's buffer).  store(cb, jb, mb, e) writes the panel.
template <int BM, int BN, int NCW, class Store>
__device__ __forceinline__ void group_phase1(const PredictParams& p, long long q0, double* qs, const double* etab,
                                             double* stg, int stg_doubles, const int* myblk, int nmine,
                                             uint64_t* stagebar, uint32_t& nstaged, double* part_mu, Store&& store) {
  constexpr int NCONS = NCW * 32, R = BM / (8 * NCW);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = p.d, Npad = p.Npad;
  stage_queries<BM, NCONS>(qs, p, d, q0, tid);
  const int CAPB = min(8, (stg_doubles / (d + 1)) / BN);
  const int JCHT = CAPB * BN;                            // ring row stride
  for (int s0 = 0; s0 < nmine; s0 += CAPB) {
    const int ns = min(CAPB, nmine - s0);
    named_bar_sync(1, NCONS);
    if (tid == 0) {
      mbar_arrive_expect_tx(stagebar, (uint32_t)((d + 1) * ns * BN * 8));
      for (int sl = 0; sl < ns; ++sl) {
        const int j0 = myblk[s0 + sl] * BN;
        for (int i = 0; i < d; ++i) bulk_g2s(stg + i * JCHT + sl * BN, p.Xs + (size_t)i * Npad + j0, BN * 8, stagebar);
        bulk_g2s(stg + d * JCHT + sl * BN, p.alphaA + j0, BN * 8, stagebar);
      }
    }
    mbar_wait(stagebar, nstaged & 1u);
    ++nstaged;
    for (int sl = 0; sl < ns; ++sl) {
      const int cb = myblk[s0 + sl];
      double macc[R] = {};
      panel_columns<BM, NCW>(stg + sl * BN, JCHT, stg + d * JCHT + sl * BN, BN, qs, d, etab, warp, lane, macc,
                             [&](int jb, int mb, const double (&e)[4]) { store(cb, jb, mb, e); });
      store_row_sums<R, NCW>(macc, part_mu + (size_t)cb * BM, warp, lane);   // this block's contribution to the means
    }
  }
}

// Host side of the group scaffold: zero the groups' barrier counters and launch kernel(p, G) with one CTA per SM.  The
// group barrier spins, so every CTA of the grid must be resident at once: a cooperative launch, which is refused
// rather than left to deadlock when they cannot be.
inline int launch_grouped(const void* kernel, const PredictParams& p, int num_sms, int G, int nthreads, size_t smem,
                          cudaStream_t st, int* launches) {
  const int ngroups = (num_sms + G - 1) / G;
  cudaError_t e = cudaMemsetAsync(p.grp_arrive, 0, sizeof(int) * ngroups, st);
  if (e != cudaSuccess) return (int)e;
  PredictParams pc = p;
  int Gc = G;
  void* args[] = {(void*)&pc, (void*)&Gc};
  e = cudaLaunchCooperativeKernel(kernel, dim3(num_sms), dim3(nthreads), args, smem, st);
  if (launches) ++*launches;
  return (int)e;
}

}  // namespace apgp
