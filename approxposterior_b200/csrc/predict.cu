// Fused GP predict for sm_100a: mean, variance and acquisition utility for a batch of queries.
//
// Replaces, for a whole batch of queries at once, what the reference does one query at a time:
//   george.GP.predict(y, x, return_var=True)   called from approxposterior/utility.py:131,178,224
//   george.GP.predict(y, x, return_var=False)  called from approxposterior/approx.py:178-180
//   + the AGP/BAPE/Jones epilogues of approxposterior/utility.py:136,183,229-244
//
//   mu(q)  = m + sum_j E[q,j] * (A alpha_j)                E[q,j] = exp(-sum_i (xs_ij - qs_i)^2)
//   var(q) = A - sum_i W[q,i]^2,   W = E . (A L^{-1})^T     (lower-triangular => only k <= i)
//
// Kernel structure (persistent, one CTA per SM, 8 consumer warps + 1 TMA producer warp):
//   phase 1  the consumer warps build the K* panel E[BM x N] of the CTA's query tile on the fly
//            from the (scaled, SoA) training set staged in shared memory, accumulate the mean,
//            and park the panel -- already in DMMA A-fragment order -- in a per-CTA scratch
//            slab that lives in L2.
//   phase 2  triangular GEMM on the FP64 tensor pipe (DMMA.8x8x4): for every block-row of
//            A L^{-1} the producer warp streams 16-wide k-steps (A tile from the slab, B tile
//            from the fragment-tiled L^{-1}) through an NSTAGE mbarrier ring with 1-D bulk TMA
//            (cp.async.bulk, SASS UBLKCP); the consumer warps issue DMMAs straight from the
//            fragment-ordered tiles (conflict-free LDS.64) into register accumulators and
//            square-reduce them into per-row sums at the end of each block-row.
//   epilogue var = A - rowsum, box-prior gate, utility, coalesced stores.
// The exponentials are evaluated once per (query, training point): DMMA and DFMA share one
// FP64 pipe on B200 (profiles/r01_fp64_pipe_probe.txt), so recomputing K* per output block
// would come straight out of the GEMM's budget.
#include "predict_tile.cuh"
#include <stdio.h>
#include <stdlib.h>

namespace apgp {

namespace {

constexpr int BK = 16;

// 8 consumer warps (warp tile 32x64) + 1 TMA producer warp, one CTA per SM.  Four consumer warps (two co-resident
// 128x64 CTAs per SM, so one CTA's panel phase overlaps the other's DMMA phase) were measured: identical results,
// 0-2 % slower at every N (profiles/r01_schedules_tried/README.md).
template <int BM, int BN, int NSTAGE>
struct VarCfg {
  static constexpr int NCONS_WARPS = 8;
  static constexpr int NCONS = NCONS_WARPS * 32;
  static constexpr int NTHREADS = NCONS + 32;
  static constexpr int WARPS_M = BM / 32;
  static constexpr int WARPS_N = BN / 64;
  static_assert(WARPS_M * WARPS_N == NCONS_WARPS, "consumer warps x warp tile 32x64 must cover the CTA tile");
  static constexpr int A_TILE = BM * BK;                 // doubles
  static constexpr int B_TILE = BN * BK;
  static constexpr int STAGE = A_TILE + B_TILE;
  static constexpr int RING = NSTAGE * STAGE;            // doubles, reused as the phase-1 staging area
};

// The DMMA kernels' dynamic shared memory, in this order: the operand ring, the scaled queries qs[d][BM], the tile's
// means mu_s[BM] and per-column-warp row sums ss_s[WARPS_N][BM] (used by the one-tile kernel only), the 2^(j/64) table
// etab[64] of exp_neg, the ring's full[NSTAGE] and empty[NSTAGE] mbarriers and phase 1's stagebar.
template <int BM, int BN, int NSTAGE>
struct VarSmem {
  using C = VarCfg<BM, BN, NSTAGE>;
  double *ring, *qs, *mu_s, *ss_s, *etab;
  uint64_t *full, *empty, *stagebar;
  __device__ __forceinline__ VarSmem(unsigned char* raw, int d)
      : ring(reinterpret_cast<double*>(raw)), qs(ring + C::RING), mu_s(qs + (size_t)d * BM), ss_s(mu_s + BM),
        etab(ss_s + C::WARPS_N * BM), full(reinterpret_cast<uint64_t*>(etab + 64)), empty(full + NSTAGE),
        stagebar(empty + NSTAGE) {}
  // the carve-up above in bytes, and 128 to spare
  static constexpr size_t bytes(int d) {
    return ((size_t)C::RING + (size_t)d * BM + BM + C::WARPS_N * BM + 64) * 8 + (2 * NSTAGE + 1) * 8 + 128;
  }
};

// One block-row ib of phase 2 on the DMMA pipe: consume its (ib + 1) BN/16 k-stages from the ring, arriving on
// empty[s] once per warp, into the 32x64 tile of W of warp (wm, wn) of the WARPS_M x WARPS_N consumer warps (the n8
// fragments are interleaved over the column warps so that the diagonal block's zero skipping stays balanced), and
// return in ss[mb] the sum of W^2 over this lane's fragments of m8 block mb.
template <int BM, int BN, int NSTAGE>
__device__ __forceinline__ void dmma_block_row(const double* ring, uint64_t* full, uint64_t* empty, uint32_t& it,
                                               int ib, int wm, int wn, int lane, double (&ss)[4]) {
  using C = VarCfg<BM, BN, NSTAGE>;
  double acc[4][8][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }
  const int nk = (ib + 1) * (BN / BK);
  const int kdiag = ib * (BN / BK);
  for (int kb = 0; kb < nk; ++kb, ++it) {
    const int s = it % NSTAGE;
    const uint32_t ph = (it / NSTAGE) & 1u;
    mbar_wait(&full[s], ph);
    const double* As = ring + (size_t)s * C::STAGE + (wm * 4) * 32 + lane;
    const double* Bs = ring + (size_t)s * C::STAGE + C::A_TILE + wn * 32 + lane;
    if (kb < kdiag) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        double a[4], b[8];
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) a[mb] = As[(k4 * (BM / 8) + mb) * 32];
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) b[nb] = Bs[(k4 * (BN / 8) + nb * C::WARPS_N) * 32];
#pragma unroll
        for (int mb = 0; mb < 4; ++mb)
#pragma unroll
          for (int nb = 0; nb < 8; ++nb) dmma884(acc[mb][nb][0], acc[mb][nb][1], a[mb], b[nb]);
      }
    } else {
      // diagonal block: n8 fragment (columns n0..n0+7 of W) only sees k <= n
      const int kloc = (kb - kdiag) * BK;              // k offset inside the diagonal block
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        double a[4];
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) a[mb] = As[(k4 * (BM / 8) + mb) * 32];
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
          const int n0 = (nb * C::WARPS_N + wn) * 8;
          if (kloc + k4 * 4 <= n0 + 7) {
            const double b = Bs[(k4 * (BN / 8) + nb * C::WARPS_N) * 32];
#pragma unroll
            for (int mb = 0; mb < 4; ++mb) dmma884(acc[mb][nb][0], acc[mb][nb][1], a[mb], b);
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[s]);
  }
#pragma unroll
  for (int mb = 0; mb < 4; ++mb) {
    double sacc = 0.0;
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      sacc = fma(acc[mb][nb][0], acc[mb][nb][0], sacc);
      sacc = fma(acc[mb][nb][1], acc[mb][nb][1], sacc);
    }
    ss[mb] = sacc;
  }
}

template <int BM, int BN, int NSTAGE>
__global__ void __launch_bounds__(VarCfg<BM, BN, NSTAGE>::NTHREADS, 1)
predict_var_kernel(const __grid_constant__ PredictParams p) {
  using C = VarCfg<BM, BN, NSTAGE>;
  constexpr int NCONS_WARPS = C::NCONS_WARPS, NCONS = C::NCONS;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const VarSmem<BM, BN, NSTAGE> sm(smem_raw, p.d);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int d = p.d, Npad = p.Npad;
  const int nblk = Npad / BN;
  const long long ntiles = (p.Q + BM - 1) / BM;
  double* panel = p.scratch + (size_t)blockIdx.x * BM * Npad;
  init_tile_smem<NSTAGE>(sm.etab, sm.full, sm.empty, sm.stagebar, NCONS_WARPS);
  __syncthreads();

  uint32_t it = 0;   // ring position, identical sequence in producer and consumers
  uint32_t nstaged = 0;   // completed training-set staging copies (parity of stagebar)

  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long q0 = tile * BM;

    // ------------------------------------------------------------ phase 1: K* panel + mean
    if (warp < NCONS_WARPS) {
      stage_queries<BM, NCONS>(sm.qs, p, d, q0, tid);
      // chunk of training columns staged in the (idle) ring: xs[d][JCH] + alpha[JCH]
      int JCH = (C::RING / (d + 1)) & ~15;
      if (JCH > Npad) JCH = Npad;
      constexpr int R = BM / (8 * NCONS_WARPS);        // m8 blocks per warp
      double mu_part[R] = {};
      for (int j0 = 0; j0 < Npad; j0 += JCH) {
        const int jn = min(JCH, Npad - j0);
        named_bar_sync(1, NCONS);                      // previous chunk fully consumed / qs visible
        // TMA-staged training set: d rows of the scaled SoA inputs + the alpha row, one bulk copy each
        if (tid == 0) {
          mbar_arrive_expect_tx(sm.stagebar, (uint32_t)((d + 1) * jn * 8));
          for (int i = 0; i < d; ++i) bulk_g2s(sm.ring + i * JCH, p.Xs + (size_t)i * Npad + j0, jn * 8, sm.stagebar);
          bulk_g2s(sm.ring + d * JCH, p.alphaA + j0, jn * 8, sm.stagebar);
        }
        mbar_wait(sm.stagebar, nstaged & 1u);
        ++nstaged;
        double macc[R] = {};
        panel_columns<BM, NCONS_WARPS>(sm.ring, JCH, sm.ring + d * JCH, jn, sm.qs, d, sm.etab, warp, lane, macc,
                                       [&](int jb, int mb, const double (&e)[4]) { store_dmma_panel<BM>(panel, j0 + jb, mb, lane, e); });
#pragma unroll
        for (int r = 0; r < R; ++r) mu_part[r] += macc[r];
      }
      store_row_sums<R, NCONS_WARPS>(mu_part, sm.mu_s, warp, lane);
      fence_proxy_async();                             // panel stores -> visible to the TMA reads below
    }
    __syncthreads();

    // ------------------------------------------------------------ phase 2: triangular DMMA GEMM
    if (warp == NCONS_WARPS) {
      if (lane == 0)
        stream_operands<NSTAGE, C::A_TILE * 8, C::B_TILE * 8, BN / BK>(sm.ring, panel, p.LinvF, nblk, sm.full, sm.empty,
                                                                        it, [](int) { return true; });
    } else {
      const int wm = warp / C::WARPS_N, wn = warp % C::WARPS_N;
      double rowss[4] = {0.0, 0.0, 0.0, 0.0};
      for (int ib = 0; ib < nblk; ++ib) {
        double ss[4];
        dmma_block_row<BM, BN, NSTAGE>(sm.ring, sm.full, sm.empty, it, ib, wm, wn, lane, ss);
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) rowss[mb] += ss[mb];
      }
#pragma unroll
      for (int mb = 0; mb < 4; ++mb) {
        double v = rowss[mb];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if ((lane & 3) == 0) sm.ss_s[wn * BM + wm * 32 + mb * 8 + (lane >> 2)] = v;
      }
      named_bar_sync(1, NCONS);
      if (tid < BM) {
        const long long q = q0 + tid;
        if (q < p.Q) {
          double tot = 0.0;
#pragma unroll
          for (int w = 0; w < C::WARPS_N; ++w) tot += sm.ss_s[w * BM + tid];
          write_query(p, d, q, p.mean + sm.mu_s[tid], p.amp - tot);
        }
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// Grouped variant of predict_var_kernel (256x64 tiling): G CTAs share ONE query tile so that the K* panels
// in flight fit in L2 instead of streaming through HBM.
//
// With one tile per CTA the 148 panels in flight are 148 x 256 x Npad x 8 B (620 MB at N = 2048): every one of
// the N/(2 BN) re-reads of a panel misses the 126 MB L2 (294 GB of DRAM traffic per 2^20 queries, ncu).  Here
// the CTAs of a group (G consecutive blockIdx) split the tile's work instead:
//   phase 1  rank r builds the panel columns of ITS share of the 64-column blocks (and the partial mean);
//   barrier  one group barrier per tile (arrival counter in global memory, acquire spin, co-resident grid);
//   phase 2  rank r runs the triangular DMMA GEMM for ITS block-rows of L^-1 (longest-first balanced so that
//            every rank streams the same number of k-steps), reading the whole panel through TMA from L2;
//   epilogue the per-rank partial row sums / means meet in a small global buffer; the tile is finalised (var,
//            prior gate, utility) by the ranks, one slice of the queries each, after the NEXT tile's barrier,
//            so a single barrier per tile orders everything.  Panels and partials are double-buffered.
// Panels in flight: 2 x (grid/G) x 256 x Npad x 8 B (152 MB at N = 2048, G = 8, of which the 76 MB being read
// stay L2-resident).  Partial sums are kept per 64-column block (mean) and per block-row (variance) and added in
// block order, so a query's result does not depend on its position in the batch, on G, or on the size of the last
// group; against the one-tile-per-CTA kernel the variance agrees to ~1e-15 and the mean to the rounding of a
// length-N sum (tests/test_gpu_parity.py::test_grouped_variance_kernel_matches_one_tile_per_cta).
// ---------------------------------------------------------------------------------------------
template <int BM, int BN, int NSTAGE>
__global__ void __launch_bounds__(VarCfg<BM, BN, NSTAGE>::NTHREADS, 1)
predict_var_group_kernel(const __grid_constant__ PredictParams p, const int G) {
  using C = VarCfg<BM, BN, NSTAGE>;
  constexpr int NCW = C::NCONS_WARPS;
  static_assert(C::WARPS_N == 1, "grouped kernel is written for the 256x64 tiling");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const VarSmem<BM, BN, NSTAGE> sm(smem_raw, p.d);
  __shared__ int owner_s[GROUP_MAX_BLOCKS];             // block-row of L^-1 (phase 2) -> rank
  __shared__ int myblk_s[GROUP_MAX_BLOCKS];             // the 64-column blocks of the panel this rank builds (phase 1)
  __shared__ int nmine_s;
  __shared__ double mu_keep[2][BM];                     // my slice's complete means, per buffer

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int Npad = p.Npad;
  const GroupCtx<BM, BN> g(p, G);
  const int nblk = g.nblk, rank = g.rank;

  init_tile_smem<NSTAGE>(sm.etab, sm.full, sm.empty, sm.stagebar, NCW);
  g.load_plan(p, G, owner_s, myblk_s, &nmine_s);
  __syncthreads();
  const int nmine = nmine_s;

  uint32_t it = 0, nstaged = 0;
  int nbar = 0;                                          // group barriers passed so far

  for (long long tile = g.t_begin; tile <= g.t_end; ++tile) {
    const int b = (int)((tile - g.t_begin) & 1);
    const bool live = tile < g.t_end;                    // the extra trip only finalises the last tile
    double* panel = p.scratch + ((size_t)g.grp * 2 + b) * BM * Npad;

    // ------------------------------------------------------------ phase 1: my column blocks of the panel
    if (live && warp < NCW) {
      group_phase1<BM, BN, NCW>(p, tile * BM, sm.qs, sm.etab, sm.ring, C::RING, myblk_s, nmine, sm.stagebar, nstaged,
                                g.part_mu + (size_t)b * nblk * BM, [&](int cb, int jb, int mb, const double (&e)[4]) {
                                  store_dmma_panel<BM>(panel, cb * BN + jb, mb, lane, e);
                                });
      __threadfence();                                   // panel + partial means visible GPU-wide before we arrive
    }
    __syncthreads();

    g.barrier(nbar);
    g.finalise(p, tile, live, b, mu_keep, [&](double, double tot) { return p.amp - tot; });
    if (!live) break;

    // ------------------------------------------------------------ phase 2: my block-rows of the triangular GEMM
    if (warp == NCW) {
      if (lane == 0)
        stream_operands<NSTAGE, C::A_TILE * 8, C::B_TILE * 8, BN / BK>(sm.ring, panel, p.LinvF, nblk, sm.full, sm.empty,
                                                                        it, [&](int ib) { return owner_s[ib] == rank; });
    } else {
      for (int ib = 0; ib < nblk; ++ib) {
        if (owner_s[ib] != rank) continue;
        double ss[4];
        dmma_block_row<BM, BN, NSTAGE>(sm.ring, sm.full, sm.empty, it, ib, warp, 0, lane, ss);
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) {                 // this block-row's contribution to rowsum(W^2)
          double v = ss[mb];
          v += __shfl_xor_sync(0xffffffffu, v, 1);
          v += __shfl_xor_sync(0xffffffffu, v, 2);
          if ((lane & 3) == 0) g.part_ss[((size_t)b * nblk + ib) * BM + warp * 32 + mb * 8 + (lane >> 2)] = v;
        }
      }
      __threadfence();                                   // partial row sums visible before the next barrier's arrival
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// Mean-only predict (the emcee lnprob form, approx.py:178-180): one query per thread, training
// set streamed through shared memory in SoA chunks; exp-bound (no GEMM).
// ---------------------------------------------------------------------------------------------
constexpr int MEAN_THREADS = 256;
constexpr int MEAN_QPT = 2;                       // queries per thread
// D > 0: input dimensionality known at compile time -- the thread's scaled query coordinates live in registers and
// the dimension loop is unrolled, which halves the shared-memory wavefronts per (query, point) pair (the kernel was
// at 67 % of the DFMA peak; N=2048, d=5: 16.0 -> 14.7 ms, 72 %).  D == 0: any d, coordinates re-read from shared
// memory inside the loop.
template <int D>
__global__ void __launch_bounds__(MEAN_THREADS)
predict_mean_kernel(const __grid_constant__ PredictParams p, int JCH) {
  extern __shared__ __align__(16) double sm[];
  const int d = (D > 0) ? D : p.d, Npad = p.Npad;
  double* xs = sm;                                // [d+1][JCH]
  double* qs = sm + (size_t)(d + 1) * JCH;        // [d][MEAN_QPT*MEAN_THREADS]
  __shared__ double etab[256];
  for (int j = threadIdx.x; j < 256; j += blockDim.x) etab[j] = exp2((double)j * (1.0 / 256.0));
  constexpr int QB = MEAN_THREADS * MEAN_QPT;
  const int tid = threadIdx.x;
  const long long ntiles = (p.Q + QB - 1) / QB;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long q0 = tile * QB;
    __syncthreads();
    for (int e = tid; e < d * QB; e += MEAN_THREADS) {
      int m = e / d, i = e - m * d;               // coalesced read of Xq rows
      long long q = q0 + m;
      qs[i * QB + m] = (q < p.Q) ? p.Xq[q * d + i] * p.qscale[i] : 0.0;
    }
    double qv[MEAN_QPT][D > 0 ? D : 1];
    if (D > 0) {
      __syncthreads();
#pragma unroll
      for (int u = 0; u < MEAN_QPT; ++u)
#pragma unroll
        for (int i = 0; i < D; ++i) qv[u][i] = qs[i * QB + u * MEAN_THREADS + tid];
    }
    double acc[MEAN_QPT] = {};
    for (int j0 = 0; j0 < Npad; j0 += JCH) {
      const int jn = min(JCH, Npad - j0);
      __syncthreads();
      for (int e = tid; e < (d + 1) * jn; e += MEAN_THREADS) {
        int i = e / jn, j = e - i * jn;
        xs[i * JCH + j] = (i < d) ? p.Xs[(size_t)i * Npad + j0 + j] : p.alphaA[j0 + j];
      }
      __syncthreads();
      const double* al = xs + (size_t)d * JCH;
      for (int j = 0; j < jn; j += 4) {
        double s[MEAN_QPT][4] = {};
        if (D > 0) {
#pragma unroll
          for (int i = 0; i < D; ++i) {
            const double2 xa = *reinterpret_cast<const double2*>(xs + i * JCH + j);       // JCH, j multiples of 4
            const double2 xb = *reinterpret_cast<const double2*>(xs + i * JCH + j + 2);
#pragma unroll
            for (int u = 0; u < MEAN_QPT; ++u) {
              const double qq = qv[u][i];
              const double d0 = xa.x - qq, d1 = xa.y - qq, d2 = xb.x - qq, d3 = xb.y - qq;
              s[u][0] = fma(d0, d0, s[u][0]); s[u][1] = fma(d1, d1, s[u][1]);
              s[u][2] = fma(d2, d2, s[u][2]); s[u][3] = fma(d3, d3, s[u][3]);
            }
          }
        } else {
          for (int i = 0; i < d; ++i) {
            const double* xr = xs + i * JCH + j;
            const double x0 = xr[0], x1 = xr[1], x2 = xr[2], x3 = xr[3];
#pragma unroll
            for (int u = 0; u < MEAN_QPT; ++u) {
              const double qq = qs[i * QB + u * MEAN_THREADS + tid];
              double d0 = x0 - qq, d1 = x1 - qq, d2 = x2 - qq, d3 = x3 - qq;
              s[u][0] = fma(d0, d0, s[u][0]); s[u][1] = fma(d1, d1, s[u][1]);
              s[u][2] = fma(d2, d2, s[u][2]); s[u][3] = fma(d3, d3, s[u][3]);
            }
          }
        }
        const double2 aa = *reinterpret_cast<const double2*>(al + j);
        const double2 ab = *reinterpret_cast<const double2*>(al + j + 2);
#pragma unroll
        for (int u = 0; u < MEAN_QPT; ++u) {
          acc[u] = fma(exp_neg256(s[u][0], etab), aa.x, acc[u]);
          acc[u] = fma(exp_neg256(s[u][1], etab), aa.y, acc[u]);
          acc[u] = fma(exp_neg256(s[u][2], etab), ab.x, acc[u]);
          acc[u] = fma(exp_neg256(s[u][3], etab), ab.y, acc[u]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < MEAN_QPT; ++u) {
      const long long q = q0 + u * MEAN_THREADS + tid;
      if (q < p.Q && p.mu) p.mu[q] = p.mean + acc[u];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// A HANDFUL of queries (the reference's own scalar loops call george.GP.predict(y, x.reshape(1, -1), return_var=True) once
// per objective evaluation, utility.py:131,178,224; the lock-step optimiser rounds ask for a few points): S CTAs per query,
// k* in shared memory, v = A L^-1 k* by one warp per pair of rows of the explicit row-major inverse (rows dealt round the
// S x 8 warps so the triangle is balanced; 8 independent loads in flight per lane: the kernel is bound by the latency of
// streaming L^-1 once from L2).  Per-CTA partial sums of |v|^2 meet in a small global buffer; the CTA that arrives last adds
// them in split order (deterministic) and writes mean, variance and utility.  Pure latency path: the tiled DMMA kernels need
// 0.5 ms (N = 2048) to 2.8 ms (N = 4096) to fill and drain their pipeline for one 256-query tile.
// ---------------------------------------------------------------------------------------------
constexpr int FEW_THREADS = 256;
constexpr int FEW_WARPS = FEW_THREADS / 32;
constexpr int FEW_MAX_SPLIT = 32;
__device__ __forceinline__ double few_row_dot(const double* __restrict__ Li, const double* __restrict__ E, int i, int lane) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int j = lane;
  for (; j + 96 <= i; j += 128) {
    s0 = fma(Li[j], E[j], s0); s1 = fma(Li[j + 32], E[j + 32], s1);
    s2 = fma(Li[j + 64], E[j + 64], s2); s3 = fma(Li[j + 96], E[j + 96], s3);
  }
  for (; j <= i; j += 32) s0 = fma(Li[j], E[j], s0);
  return (s0 + s1) + (s2 + s3);
}
__global__ void __launch_bounds__(FEW_THREADS)
predict_few_kernel(const __grid_constant__ PredictParams p, const double* __restrict__ Linv, int ld, int S,
                   double* __restrict__ part /*[Q][S]*/, double* __restrict__ mu_ws /*[Q]*/, int* __restrict__ count /*[Q]*/) {
  extern __shared__ __align__(16) double E[];          // [N] k* / A
  __shared__ double red[FEW_WARPS];
  __shared__ double qs[APGP_MAXD];
  __shared__ int s_last;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = p.d, N = p.N, Npad = p.Npad;
  const int sp = blockIdx.x;
  const long long q = blockIdx.y;
  if (tid < d) qs[tid] = p.Xq[q * d + tid] * p.qscale[tid];
  __syncthreads();
  double mpart = 0.0;
  for (int j = tid; j < N; j += FEW_THREADS) {
    double s = 0.0;
    for (int i = 0; i < d; ++i) { const double t = p.Xs[(size_t)i * Npad + j] - qs[i]; s = fma(t, t, s); }
    const double e = exp(-s);
    E[j] = e;
    if (sp == 0) mpart = fma(e, p.alphaA[j], mpart);
  }
  if (sp == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mpart += __shfl_xor_sync(0xffffffffu, mpart, o);
    if (lane == 0) red[warp] = mpart;
  }
  __syncthreads();                                     // publishes E (and the mean partials)
  if (sp == 0 && tid == 0) {
    double mu = p.mean;
#pragma unroll
    for (int w = 0; w < FEW_WARPS; ++w) mu += red[w];
    mu_ws[q] = mu;
  }
  double acc = 0.0;
  const int stride = S * FEW_WARPS;
  for (int i = sp * FEW_WARPS + warp; i < N; i += 2 * stride) {       // two rows per trip: independent load streams
    const int i2 = i + stride;
    double a = few_row_dot(Linv + (size_t)i * ld, E, i, lane);
    double b = (i2 < N) ? few_row_dot(Linv + (size_t)i2 * ld, E, i2, lane) : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    const double va = p.amp * a, vb = p.amp * b;
    acc = fma(va, va, acc);                            // identical in all lanes of the warp
    acc = fma(vb, vb, acc);
  }
  __syncthreads();                                     // red is free again
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (tid == 0) {
    double tot = 0.0;
#pragma unroll
    for (int w = 0; w < FEW_WARPS; ++w) tot += red[w];
    part[q * S + sp] = tot;
    __threadfence();
    s_last = (atomicAdd(&count[q], 1) == S - 1);
  }
  __syncthreads();
  if (s_last && tid == 0) {
    __threadfence();
    double tot = 0.0;
    for (int k = 0; k < S; ++k) tot += __ldcg(part + q * S + k);
    const double mu = __ldcg(mu_ws + q);
    const double var = p.amp - tot;
    count[q] = 0;                                      // re-armed for the next launch on this stream
    write_query(p, d, q, mu, var);
  }
}

// ---------------------------------------------------------------------------------------------
// Packers (run once per factorisation)
// ---------------------------------------------------------------------------------------------
__global__ void pack_linv_kernel(const double* __restrict__ Linv, int ld, int N, int Npad, int BN, double amp,
                                 double* __restrict__ out, long total) {
  const long tile_elems = (long)BN * 16;
  for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    long t = idx / tile_elems;
    int w = (int)(idx - t * tile_elems);
    // invert t = (BN/16) * ib(ib+1)/2 + kb
    const int per = BN / 16;
    int ib = (int)((sqrt(8.0 * (double)(t / per) + 1.0) - 1.0) * 0.5);
    while ((long)per * ((long)(ib + 1) * (ib + 2) / 2) <= t) ++ib;
    while ((long)per * ((long)ib * (ib + 1) / 2) > t) --ib;
    int kb = (int)(t - (long)per * ((long)ib * (ib + 1) / 2));
    int k4 = w / (BN * 4);
    int r = w - k4 * (BN * 4);
    int n8 = r >> 5, l = r & 31;
    int n = ib * BN + n8 * 8 + (l >> 2);
    int k = kb * 16 + k4 * 4 + (l & 3);
    double v = 0.0;
    if (n < N && k <= n) v = amp * Linv[(size_t)n * ld + k];
    out[idx] = v;
  }
}

__global__ void pack_xs_kernel(const double* __restrict__ X, int N, int d, int Npad, const double* __restrict__ qscale,
                               double* __restrict__ Xs) {
  long total = (long)d * Npad;
  for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int i = (int)(idx / Npad), j = (int)(idx - (long)i * Npad);
    Xs[idx] = (j < N) ? X[(size_t)j * d + i] * qscale[i] : 0.0;
  }
}

__global__ void exp_neg_test_kernel(const double* __restrict__ s, int n, double* __restrict__ out, int variant) {
  __shared__ double tab[256];
  const int m = variant ? 256 : 64;
  for (int j = threadIdx.x; j < m; j += blockDim.x) tab[j] = exp2((double)j / (double)m);
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = variant ? exp_neg256(s[i], tab) : exp_neg(s[i], tab);
}

template <int BM, int BN, int NSTAGE>
int launch_var_t(const PredictParams& p, int num_sms, cudaStream_t st) {
  const size_t smem = VarSmem<BM, BN, NSTAGE>::bytes(p.d);
  static PerDeviceOnce attr;
  if (attr.needed()) {
    cudaError_t e = cudaFuncSetAttribute(predict_var_kernel<BM, BN, NSTAGE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         227 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr.mark();
  }
  long long ntiles = (p.Q + BM - 1) / BM;
  int grid = (int)(ntiles < num_sms ? ntiles : num_sms);
  if (grid < 1) return 0;
  predict_var_kernel<BM, BN, NSTAGE><<<grid, VarCfg<BM, BN, NSTAGE>::NTHREADS, smem, st>>>(p);
  return (int)cudaGetLastError();
}

// the grouped kernel's dynamic shared memory opt-in; its 4.6 KB of static tables (ownership, kept means) come on top
constexpr int GROUP_SMEM = 220 * 1024;

}  // namespace

// One tile per CTA: 256x64 (B fragments amortised over 8 m8 blocks, smallest diagonal-block waste, no register
// spills), or 128x128 from d = 32, where d x 256 staged queries no longer fit beside the 256x64 tile's ring.  Two other
// schedules (warp-specialised builders, inline builder) were measured slower and are archived with their profiles
// under profiles/r01_schedules_tried/.
static int tile_bm(int d) { return d > 31 ? 128 : 256; }
int predict_tile_bn(int d) { return 256 * 64 / tile_bm(d); }

size_t predict_scratch_bytes(int Npad, int num_sms, int d) { return (size_t)num_sms * tile_bm(d) * Npad * 8; }

// ---- grouped launch (256x64 tiling only) ------------------------------------------------------------
// Work split inside a group of gs ranks.  Phase 2: block-row ib of L^-1 costs ib + 1 units (one unit = 64 k-columns
// of DMMA for the 256x64 tile); longest-first onto the least loaded rank.  Phase 1: building one 64-column block of
// the panel costs (2d + 12)/64 of a unit (exp + distances on the same FP64 pipe); the blocks go, one by one, to the
// rank with the least combined load, which also evens out what phase 2 could not.  Returns max load / mean load.
// Other engines scale that phase-1 cost by their tile's phase1_scale.
// The grouped kernel takes d up to 27: from d = 28 the staged queries no longer fit beside the ring in GROUP_SMEM.
constexpr int dmma_group_max_d() {
  int d = 1;
  while (VarSmem<256, 64, 4>::bytes(d + 1) <= GROUP_SMEM) ++d;
  return d;
}
const GroupTile DMMA_GROUP_TILE = {256, 8, 1.0, dmma_group_max_d()};

double plan_group_split(int nblk, int gs, int d, int* owner2, int* owner1, const GroupTile& tile) {
  double load[64];
  for (int r = 0; r < gs; ++r) load[r] = 0.0;
  for (int ib = nblk - 1; ib >= 0; --ib) {
    int best = 0;
    for (int r = 1; r < gs; ++r) if (load[r] < load[best]) best = r;
    owner2[ib] = best; load[best] += ib + 1;
  }
  const double c1 = (2.0 * d + 12.0) / 64.0 * tile.phase1_scale;
  for (int cb = 0; cb < nblk; ++cb) {
    int best = 0;
    for (int r = 1; r < gs; ++r) if (load[r] < load[best]) best = r;
    owner1[cb] = best; load[best] += c1;
  }
  double mx = 0.0, tot = 0.0;
  for (int r = 0; r < gs; ++r) { tot += load[r]; if (load[r] > mx) mx = load[r]; }
  return mx * gs / tot;
}

int predict_group_size(int Npad, int num_sms, int requested, int d, long long Q, const GroupTile& tile) {
  if (Npad / 64 > GROUP_MAX_BLOCKS) return 1;
  if (d > tile.max_d) return 1;
  const int BM = tile.bm, EB = tile.panel_bytes;      // queries per tile, panel bytes per (query, training point)
  const int nblk = Npad / 64;
  int G = requested;
  if (G < 0) {
    int o2[GROUP_MAX_BLOCKS], o1[GROUP_MAX_BLOCKS];
    // (a) throughput regime.  Gmin = smallest group whose panels being READ (one of the two buffers per group) fit
    // ~80 MB of L2 (measured at N = 2048: G = 8 keeps the speed of one tile per CTA with 8.8x less DRAM traffic).
    // Among Gmin/2 .. 64 take the group size with the best balanced split (a group waits for its slowest rank
    // every tile: N = 1536 with G = 8 is 9 % imbalanced, G = 6 is exact); ties go to the smallest G >= Gmin.
    // Below N = 1024 the 148 one-tile panels already (nearly) fit: no grouping.
    int bestG = 1; double bestS = 1e30;
    int Gmin = 1;
    if (Npad >= 1024) {
      Gmin = 2;
      while (Gmin < 64 && (size_t)((num_sms + Gmin - 1) / Gmin) * BM * Npad * EB > ((size_t)80 << 20)) ++Gmin;
      for (int g = (Gmin / 2 > 2 ? Gmin / 2 : 2); g <= 64 && 2 * g <= nblk; ++g) {
        double imb = plan_group_split(nblk, g, d, o2, o1, tile);
        const int tail = num_sms % g;               // a smaller last group: weigh its imbalance by its share of the SMs
        if (tail > 1) imb = (imb * (num_sms - tail) + plan_group_split(nblk, tail, d, o2, o1, tile) * tail) / num_sms;
        else if (tail == 1) imb += 1.0 / num_sms;   // a lone CTA does whole tiles: fine, but it cannot share a panel
        const double score = imb + (g < Gmin ? 0.005 : 0.0) + 1e-4 * g;   // L2 fit is worth 0.5 % of balance; then small G
        if (score < bestS) { bestS = score; bestG = g; }
      }
    }
    // (b) latency regime: a call with fewer query tiles than would fill half the GPU (optimiser rounds, refinement
    // passes: a handful of queries) spreads each tile over as many CTAs as the balance allows -- one 256-query tile
    // at N = 2048 is 32 block-rows for ONE CTA otherwise.
    const long long ntiles = (Q + BM - 1) / BM;
    if (ntiles * bestG * 2 <= num_sms && nblk >= 4) {
      long long cap = num_sms / ntiles;
      if (cap > 64) cap = 64;
      if (cap > nblk / 2) cap = nblk / 2;
      int fillG = bestG; double fillS = (bestG > 1) ? plan_group_split(nblk, bestG, d, o2, o1, tile) / bestG : 1.0;
      for (int g = bestG + 1; g <= (int)cap; ++g) {
        const double t = plan_group_split(nblk, g, d, o2, o1, tile) / g;      // time per tile ~ imbalance / ranks
        if (t < fillS * 0.97) { fillS = t; fillG = g; }
      }
      bestG = fillG;
    }
    if (getenv("APGP_DEBUG_GROUP")) fprintf(stderr, "[apgp] Npad=%d nblk=%d Q=%lld Gmin=%d -> G=%d\n", Npad, nblk, Q, Gmin, bestG);
    return bestG;
  }
  while (G > 1 && 2 * G > nblk) --G;              // every rank needs block-rows from both ends to balance
  if (G > 64) G = 64;
  return G < 1 ? 1 : G;
}
// work-split tables for the kernel: [full group | last (smaller) group] x [phase-2 owner | phase-1 owner] x GROUP_MAX_BLOCKS
void predict_group_plan(int Npad, int num_sms, int G, int d, int* tab, const GroupTile& tile) {
  const int nblk = Npad / 64, tail = num_sms % G;
  for (int i = 0; i < 4 * GROUP_MAX_BLOCKS; ++i) tab[i] = 0;
  plan_group_split(nblk, G, d, tab, tab + GROUP_MAX_BLOCKS, tile);
  plan_group_split(nblk, tail > 0 ? tail : G, d, tab + 2 * GROUP_MAX_BLOCKS, tab + 3 * GROUP_MAX_BLOCKS, tile);
}
size_t predict_group_scratch_bytes(int Npad, int num_sms, int G, const GroupTile& tile) {
  return (size_t)2 * ((num_sms + G - 1) / G) * (tile.bm * tile.panel_bytes) * Npad;
}
size_t predict_group_part_bytes(int Npad, int num_sms, int G) { return (size_t)((num_sms + G - 1) / G) * 4 * (Npad / 64) * 256 * 8; }

int launch_predict_var_grouped(const PredictParams& p, int num_sms, int G, cudaStream_t st, int* launches) {
  if (p.Q <= 0) return 0;
  static PerDeviceOnce attr;
  if (attr.needed()) {
    cudaError_t e = cudaFuncSetAttribute(predict_var_group_kernel<256, 64, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GROUP_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr.mark();
  }
  return launch_grouped((const void*)predict_var_group_kernel<256, 64, 4>, p, num_sms, G, VarCfg<256, 64, 4>::NTHREADS,
                        VarSmem<256, 64, 4>::bytes(p.d), st, launches);
}

int launch_predict_var(const PredictParams& p, int num_sms, cudaStream_t st, int* launches) {
  if (p.Q <= 0) return 0;
  if (launches) ++*launches;
  if (tile_bm(p.d) == 128) return launch_var_t<128, 128, 5>(p, num_sms, st);
  return launch_var_t<256, 64, 4>(p, num_sms, st);
}

size_t predict_few_ws_bytes() { return (size_t)PREDICT_FEW_MAX * (FEW_MAX_SPLIT + 1) * 8 + PREDICT_FEW_MAX * sizeof(int); }
// ws: predict_few_ws_bytes() bytes, zeroed once when allocated (the kernel re-arms its counters itself)
int launch_predict_few(const PredictParams& p, const double* Linv, int ld, void* ws, cudaStream_t st, int* launches) {
  if (p.Q <= 0) return 0;
  const size_t smem = (size_t)p.N * 8;
  static PerDeviceOnce attr;
  if (attr.needed()) {
    cudaError_t e = cudaFuncSetAttribute(predict_few_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr.mark();
  }
  int S = p.N / 64;                                    // ~8 rows per warp and split: N = 70 -> 1, 512 -> 8, >= 2048 -> 32
  if (S < 1) S = 1;
  if (S > FEW_MAX_SPLIT) S = FEW_MAX_SPLIT;
  double* part = static_cast<double*>(ws);
  double* mu_ws = part + PREDICT_FEW_MAX * FEW_MAX_SPLIT;
  int* count = reinterpret_cast<int*>(mu_ws + PREDICT_FEW_MAX);
  predict_few_kernel<<<dim3((unsigned)S, (unsigned)p.Q), FEW_THREADS, smem, st>>>(p, Linv, ld, S, part, mu_ws, count);
  if (launches) ++*launches;
  return (int)cudaGetLastError();
}

int launch_predict_mean(const PredictParams& p, int num_sms, cudaStream_t st, int* launches) {
  if (p.Q <= 0) return 0;
  constexpr int QB = MEAN_THREADS * MEAN_QPT;
  const size_t qs_bytes = (size_t)p.d * QB * 8;
  // smem budget: 96 KB keeps 2 CTAs/SM for small d; large d needs more room for the staged queries
  const size_t budget = (qs_bytes + 16 * 1024 <= 96 * 1024) ? 96 * 1024 : 200 * 1024;
  int JCH = (int)(((budget - qs_bytes) / 8) / (p.d + 1)) & ~3;
  if (JCH > p.Npad) JCH = p.Npad;
  if (JCH < 4) return (int)cudaErrorInvalidValue;
  const size_t smem = (size_t)(p.d + 1) * JCH * 8 + qs_bytes;
  long long ntiles = (p.Q + QB - 1) / QB;
  long long cap = (long long)num_sms * 2;
  int grid = (int)(ntiles < cap ? ntiles : cap);
  cudaError_t e = cudaSuccess;
#define APGP_MEAN_LAUNCH(DD)                                                                                         \
  do {                                                                                                               \
    static PerDeviceOnce attr;                                                                                       \
    if (attr.needed()) {                                                                                             \
      e = cudaFuncSetAttribute(predict_mean_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 204 * 1024);  \
      if (e != cudaSuccess) return (int)e;                                                                           \
      attr.mark();                                                                                                   \
    }                                                                                                                \
    predict_mean_kernel<DD><<<grid, MEAN_THREADS, smem, st>>>(p, JCH);                                             \
  } while (0)
  switch (p.d) {
    // d <= 2: the exponential dominates and the generic kernel measured 2 % faster (5.85 vs 5.96 ms, N=1024, d=2)
    case 3: APGP_MEAN_LAUNCH(3); break;
    case 4: APGP_MEAN_LAUNCH(4); break;
    case 5: APGP_MEAN_LAUNCH(5); break;
    case 6: APGP_MEAN_LAUNCH(6); break;
    case 7: APGP_MEAN_LAUNCH(7); break;
    case 8: APGP_MEAN_LAUNCH(8); break;
    case 10: APGP_MEAN_LAUNCH(10); break;
    default: APGP_MEAN_LAUNCH(0); break;
  }
#undef APGP_MEAN_LAUNCH
  if (launches) ++*launches;
  return (int)cudaGetLastError();
}

int launch_pack_linv(const double* Linv, int ld, int N, int Npad, int BN, double amp, double* LinvF, cudaStream_t st) {
  long total = linvf_total_tiles(Npad, BN) * (long)BN * 16;
  int grid = (int)((total + 255) / 256); if (grid > 148 * 16) grid = 148 * 16;
  pack_linv_kernel<<<grid, 256, 0, st>>>(Linv, ld, N, Npad, BN, amp, LinvF, total);
  return (int)cudaGetLastError();
}

int launch_exp_neg_test(const double* s, int n, double* out, cudaStream_t st, int variant) {
  exp_neg_test_kernel<<<64, 256, 0, st>>>(s, n, out, variant);
  return (int)cudaGetLastError();
}

int launch_pack_xs(const double* X, int N, int d, int Npad, const double* qscale_dev, double* Xs, cudaStream_t st) {
  long total = (long)d * Npad;
  int grid = (int)((total + 255) / 256); if (grid > 148 * 8) grid = 148 * 8;
  pack_xs_kernel<<<grid, 256, 0, st>>>(X, N, d, Npad, qscale_dev, Xs);
  return (int)cudaGetLastError();
}

}  // namespace apgp
