// Fused log-likelihood of ONE hyper-parameter vector for training sets too large for one CTA's shared memory
// (N > ~220): covariance build, blocked right-looking Cholesky with look-ahead, forward substitution and the
// log-likelihood reductions in a single kernel, executed by a thread-block CLUSTER of C CTAs (C = 1, 2, 4, 8, 16) that
// keeps the matrix in L2-resident global memory and meets only at two release/acquire flags per 64-column block.
//
// Replaces, per evaluation of gpUtils._nll (reference gpUtils.py:46-80: george.GP.log_likelihood = kernel build +
// Cholesky), the 3 Np/64 + 2 dependent launches of the tiled path in factor.cu (build_K, then chol_diag / chol_panel /
// chol_update per block column, then loglik_finish), whose cost was one launch gap plus one serial 64x64 pivot chain per
// block column regardless of the batch size.
//
// Work split.  The lower triangle of K is cut into 64x64 tiles; tile (i, j) belongs to CTA  (i(i+1)/2 + j) mod C  for
// the whole factorisation (owner computes: build, every trailing update, the panel solve, and -- for diagonal tiles --
// the 64x64 factorisation).  Only PANEL results cross CTAs, so step k needs two flags:
//   A_k  "diagonal block k factored":  L_kk, its reciprocal pivots, the inverses of its eight 8x8 diagonal blocks and
//        z_k are in global memory                                                    (one writer, flagA)
//   B_k  "panel k solved":             every L_ik = A_ik L_kk^{-T} is in global memory (C writers, cntB)
// Look-ahead: after B_k a CTA first updates its tiles of column k+1 (the owner of (k+1, k+1) then factors it at once
// and raises A_{k+1}), and only then applies step k to the rest of its trailing tiles -- that deferred work overlaps
// the next block's serial pivot chain on the owner.
//
// Inside a CTA (256 threads).  The restart's matrix lives in L2-resident global memory TILE-MAJOR: every 64x64 tile is one
// contiguous [64][68] block (the shared-memory image), so an operand tile is ONE bulk TMA copy.
//   build     two workers of 4 warps, one tile each: inputs pre-scaled and transposed in shared memory, one column and
//             sixteen consecutive rows per thread and pass (16 independent chains, LDS.128 broadcasts), table exponential;
//             the next tile's inputs travel in registers meanwhile;
//   diagonal  all 256 threads (chol_small.cuh: 8-wide register-blocked, r_k riding along as a right-hand side so that
//             z_k = L_kk^{-1} r_k comes out of the same pass); 64 threads then invert the eight 8x8 diagonal blocks;
//   panel     all 8 warps on a pair of tiles (cg_panel_phase): X = P L_kk^{-T} blockwise on the tensor pipe (cg_trsm_dmma: per
//             8 rows a warp-private chain of DMMA.8x8x4 against the finished columns, the inverted 8x8 block applied by two
//             more), tile pairs fed by bulk TMA one pair ahead, rows written back by the warp that solved them;
//   updates   all 8 warps as one TMA-fed software pipeline (cg_update_phase): A, B and C tiles by bulk copies one update
//             ahead, warp tile 32x16, one CTA barrier per update; the DMMA loop itself runs at the tensor-pipe rate
//             (4.1 k cycles per 64x64x64 update).
// Measured per phase with the -DAPGP_PROF_CG build (tools/profile_chol_group_phases.py, profiles/r02_chol_group_phases.md).
//
// The flags only ever grow (epoch-based targets), so repeated evaluations by the same cluster -- the device
// optimisers call this once per objective evaluation -- need no reset.  All partial sums are added in block order:
// every CTA of the cluster returns the SAME bits, which the replicated optimiser state relies on.
// Every multiply-add is explicit (fma, or __dmul_rn / __dadd_rn / __dsub_rn where none is fused), so the routine rounds
// the same in translation units compiled with and without -fmad (loglik.cuh).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include "common.cuh"
#include "chol_small.cuh"

namespace apgp {

constexpr int CG_T = 64;                 // tile edge
constexpr int CG_LD = 68;                // padded shared leading dimension (conflict-free DMMA fragment loads)
constexpr int CG_THREADS = 256;
constexpr int CG_WT = 128;               // threads per tile worker
constexpr int CG_TILE = CG_T * CG_LD;    // doubles per staged tile
constexpr int CG_AUX = CG_T + 8 * 64;    // per worker: z_k [64] + the 8 inverted 8x8 diagonal blocks of L_kk (panel solve)
constexpr int CG_CONST = 64 + APGP_MAXD; // exponential table 2^(j/64) + per-dimension input scales sqrt(1 / (2 M_i))
constexpr int CG_NTILES = 5;             // tile buffers: 2 x (A, B) + the C tile of the update pipeline
constexpr size_t CG_SMEM_DOUBLES = (size_t)CG_NTILES * CG_TILE + 2 * CG_AUX + CG_CONST;   // + 2 x aux + constants
constexpr int CG_DIAG_LDR = CG_T + 1;
// the diagonal factorisation aliases the tile buffers: packed block + (1 + 64) right-hand sides + pivots
static_assert((size_t)(CG_T * (CG_T + 1) / 2 + (CG_T + 1) * CG_DIAG_LDR + CG_T) <= CG_SMEM_DOUBLES, "diag scratch fits");

struct CholGroup {
  int N, Np, nb, d;
  int C, rank;                           // cluster size, this CTA's rank in it
  const double* X;                       // [N][d] training inputs (global, read-only for the kernel's lifetime)
  const double* y;                       // [N]
  double* K;                             // this restart's matrix, tile-major (cg_tile_ptr): nb(nb+1)/2 tiles of [64][CG_LD]
  double* Dinv;                          // [nb][64][64]
  double* r;                             // [Np]
  double* part;                          // [2][nb][4]: per block sum z^2, sum log diag, bad pivot (double-buffered by epoch)
  unsigned long long* flagA;             // sync words of this restart (monotone)
  unsigned long long* cntB;
};

// per-restart global workspace of a batch of R problems, carved from one allocation of cg_ws_bytes(Np, R)
struct GroupWs {
  double* K; double* Dinv; double* r; double* part; unsigned long long* flags;
  size_t sK, sDinv, sR, sPart;           // strides (in doubles) between restarts; flags: 2 words per restart
};
inline size_t cg_ws_bytes(int Np, int R) {
  const size_t nb = Np / CG_T;
  return (size_t)R * (nb * (nb + 1) / 2 * CG_TILE + nb * CG_T * CG_T + Np + 2 * nb * 4) * sizeof(double) + ((size_t)R * 16 + 255) / 256 * 256 + 256;
}
inline GroupWs cg_ws_carve(void* ws_bytes, int Np, int R) {
  const size_t nb = Np / CG_T;
  GroupWs ws;
  char* base = static_cast<char*>(ws_bytes);
  ws.flags = reinterpret_cast<unsigned long long*>(base); base += ((size_t)R * 16 + 255) / 256 * 256;
  ws.K = reinterpret_cast<double*>(base); ws.sK = nb * (nb + 1) / 2 * CG_TILE; base += (size_t)R * ws.sK * 8;
  ws.Dinv = reinterpret_cast<double*>(base); ws.sDinv = nb * CG_T * CG_T; base += (size_t)R * ws.sDinv * 8;
  ws.r = reinterpret_cast<double*>(base); ws.sR = Np; base += (size_t)R * ws.sR * 8;
  ws.part = reinterpret_cast<double*>(base); ws.sPart = 2 * nb * 4;
  return ws;
}
__device__ __forceinline__ CholGroup cg_make(const GroupWs& ws, int rr, int N, int Np, int d, int C, int rank,
                                             const double* X, const double* y) {
  CholGroup g;
  g.N = N; g.Np = Np; g.nb = Np / CG_T; g.d = d; g.C = C; g.rank = rank; g.X = X; g.y = y;
  g.K = ws.K + rr * ws.sK; g.Dinv = ws.Dinv + rr * ws.sDinv; g.r = ws.r + rr * ws.sR; g.part = ws.part + rr * ws.sPart;
  g.flagA = ws.flags + 2 * (size_t)rr; g.cntB = g.flagA + 1;
  return g;
}
__device__ __forceinline__ int cg_cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r)); return (int)r; }

__device__ __forceinline__ int cg_owner(int i, int j, int C) { return (i * (i + 1) / 2 + j) & (C - 1); }   // C: power of two
// Global layout of a restart's matrix: TILE-MAJOR.  Tile (i, j), j <= i, is the contiguous block number i(i+1)/2 + j, stored
// as the shared-memory image [64][CG_LD] (padding included), so one bulk TMA copy moves a whole operand tile.
__device__ __forceinline__ double* cg_tile_ptr(const CholGroup& g, int i, int j) {
  return g.K + (size_t)(i * (i + 1) / 2 + j) * CG_TILE;
}

// ---- cross-CTA flags ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long cg_ld_acquire(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// all threads of the CTA have finished their global writes (call with the whole CTA)
__device__ __forceinline__ void cg_publish_store(unsigned long long* p, unsigned long long v) {
  __syncthreads();
  if (threadIdx.x == 0) { __threadfence(); asm volatile("st.release.gpu.global.u64 [%0], %1;\n" :: "l"(p), "l"(v) : "memory"); }
}
__device__ __forceinline__ void cg_publish_add(unsigned long long* p) {
  __syncthreads();
  if (threadIdx.x == 0) { __threadfence(); asm volatile("red.release.gpu.global.add.u64 [%0], 1;\n" :: "l"(p) : "memory"); }
}
__device__ __forceinline__ void cg_wait_ge(const unsigned long long* p, unsigned long long v) {
  if (threadIdx.x == 0) { while (cg_ld_acquire(p) < v) { } }
  __syncthreads();
}

// ---- tile staging: 64x64 doubles, global row-major (ld) -> shared [r][CG_LD], 16-byte cp.async through L2 ------
__device__ __forceinline__ void cg_stage_tile(double* dst, const double* src, int ld, int wtid) {
#pragma unroll 4
  for (int e = wtid; e < CG_T * (CG_T / 2); e += CG_WT) {
    const int r = e >> 5, c2 = (e & 31) * 2;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n"
                 :: "r"(smem_u32(dst + r * CG_LD + c2)), "l"(src + (size_t)r * ld + c2) : "memory");
  }
}
__device__ __forceinline__ void cg_stage_wait() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// -DAPGP_PROF: thread 0 of the first restart's CTAs (ranks 0 and 1) accumulates SM cycles per phase into g_cgprof
// (printed by launch_loglik_group when APGP_PROF_PRINT is set): 0 build, 1 diag load, 2 diag factor, 3 diag store +
// publish, 4 deferred updates, 5 wait A, 6 panel, 7 publish + wait B, 8 urgent updates, 9 final, 10 total;
// update pipeline: 11 wait + barrier, 12 next-tile search + staging issue + C fetch, 13 DMMA loop, 14 subtract + store;
// (21 next-tile search, 22 TMA issue, then 12 = C fetch only)
// panel: 15 staging wait (first slot also L_kk), 16 solve, 17 r update, 18 write-back; build: 19 staging, 20 entries
#ifdef APGP_PROF_CG
__device__ long long g_cgprof[2][24];
#define CGP_T(var) long long var = clock64()
#define CGP_ADD(slot, t0) do { if (threadIdx.x == 0 && blockIdx.x < 2) { const long long _n = clock64(); g_cgprof[blockIdx.x][slot] += _n - (t0); (t0) = _n; } } while (0)
#else
#define CGP_T(var) do {} while (0)
#define CGP_ADD(slot, t0) do {} while (0)
#endif


// Panel solve on the FP64 tensor pipe: X = P L^{-T} for one 64x64 panel tile P (shared, row-major, leading dimension
// CG_LD, overwritten by X), L the factored diagonal block (shared, same layout), inv the 8 inverted 8x8 diagonal blocks
// of L ([J][n][k], computed once by the block's owner).  Blocked by 8 columns, as a warp-private chain per 8 rows:
//   X_J = (P_J - sum_{I<J} X_I L_JI^T) inv_J^T
// the sum as one DMMA.8x8x4 chain over the finished columns (two accumulator pairs), the multiplication by the inverted
// block as two more DMMAs after a quad shuffle from the accumulator layout to the A-operand layout.  A warp carries the
// row block mb (rows 8 mb .. 8 mb + 7) of H different tiles side by side as independent chains; rows never cross warps, so
// __syncwarp suffices.
// The one-thread-per-row substitution this replaces (2016 dependent-ish FMAs per row, 64 registers of row, a fully
// unrolled 60 KB instruction stream) measured 25 k cycles per round of tiles; this form is ~2 k.
template <int H>
__device__ __forceinline__ void cg_trsm_dmma(double* const (&tiles)[H], const double* __restrict__ Ls,
                                             const double* __restrict__ inv, int mb, int lane) {
  const int m = lane >> 2, q = lane & 3;
  const int src0 = (lane & ~3) | (q >> 1), src1 = src0 + 2;
  const bool odd = q & 1;
  double* pr[H];
#pragma unroll
  for (int h = 0; h < H; ++h) pr[h] = tiles[h] + (mb * 8 + m) * CG_LD;
#pragma unroll
  for (int J = 0; J < CG_T / 8; ++J) {
    const double* lr = Ls + (8 * J + m) * CG_LD + q;
    double c[H][2][2];
#pragma unroll
    for (int h = 0; h < H; ++h) { c[h][0][0] = c[h][0][1] = c[h][1][0] = c[h][1][1] = 0.0; }
#pragma unroll
    for (int k4 = 0; k4 < 2 * J; ++k4) {
      const double b = lr[4 * k4];
#pragma unroll
      for (int h = 0; h < H; ++h) dmma884(c[h][k4 & 1][0], c[h][k4 & 1][1], pr[h][4 * k4 + q], b);
    }
    const double b_lo = inv[J * 64 + m * 8 + q], b_hi = inv[J * 64 + m * 8 + 4 + q];
#pragma unroll
    for (int h = 0; h < H; ++h) {
      const double2 pv = *reinterpret_cast<const double2*>(pr[h] + 8 * J + 2 * q);
      const double t0 = pv.x - (c[h][0][0] + c[h][1][0]), t1 = pv.y - (c[h][0][1] + c[h][1][1]);
      const double u0 = __shfl_sync(0xffffffffu, t0, src0), u1 = __shfl_sync(0xffffffffu, t1, src0);
      const double v0 = __shfl_sync(0xffffffffu, t0, src1), v1 = __shfl_sync(0xffffffffu, t1, src1);
      const double a_lo = odd ? u1 : u0, a_hi = odd ? v1 : v0;
      double x0 = 0.0, x1 = 0.0, y0 = 0.0, y1 = 0.0;
      dmma884(x0, x1, a_lo, b_lo);
      dmma884(y0, y1, a_hi, b_hi);
      double2 xv; xv.x = x0 + y0; xv.y = x1 + y1;
      *reinterpret_cast<double2*>(pr[h] + 8 * J + 2 * q) = xv;
    }
    __syncwarp();
  }
}

// Trailing updates  C_ij -= L_i,kc L_j,kc^T  for this CTA's tiles of the block columns [j0, j1), as ONE software
// pipeline run by all 8 warps.  Every operand arrives by bulk TMA (the global matrix is tile-major, so a tile is one
// 34 KB copy issued by one lane, completion on an mbarrier): while the tensor pipe works on update t, the A tile of
// update t + 1 -- and its B tile when the block column changes; A and B are double-buffered independently -- and the C
// tile of update t land in shared memory; one CTA barrier per update.  Warp tile 32x16 (8 DMMA chains per warp, k
// ascending: same bits as any other split of the tile).  History (cycles per update and CTA at N = 1024, against 4.1 k of
// tensor-pipe time): two workers staging, multiplying and read-modify-writing in sequence 8.3 k; this pipeline with
// per-thread cp.async staging 7.0 k (16 LDGSTS per thread block issue for 1.4 k); TMA with the C tile fetched into
// registers by LDG 6.3 k (0.6 k of LDG issue back-pressure in every warp); C by TMA as well 6.0 k; the CTA barrier per
// update replaced by an mbarrier only the issuing lane waits on 5.3 k (what is left: the two warps of a scheduler leave
// their DMMA loops together, so their C subtract/store epilogues do not hide behind each other's tensor work).
__device__ __forceinline__ bool cg_next_tile(int& i, int& j, int j1, int nb, int C, int me) {
  for (;;) {
    if (++i >= nb) { ++j; i = j; }
    if (j >= j1) return false;
    if (cg_owner(i, j, C) == me) return true;
  }
}
__device__ __forceinline__ void cg_update_phase(const CholGroup& g, double* sm, int kc, int j0, int j1) {
  const int tid = threadIdx.x, w8 = tid >> 5, lane = tid & 31;
  const int wm = w8 >> 2, wn = w8 & 3;
  const int nb = g.nb, C = g.C, me = g.rank;
  if (j1 > nb) j1 = nb;
  __shared__ __align__(8) uint64_t full[4];            // operand pairs 0 / 1, C tile; [3]: "update t - 1 finished" (8 warps)
  int i = j0 - 1, j = j0;
  bool have = (j0 < j1) && cg_next_tile(i, j, j1, nb, C, me);
  if (!have) return;                                   // uniform across the CTA
  if (tid == 0) { mbar_init(&full[0], 1); mbar_init(&full[1], 1); mbar_init(&full[2], 1); mbar_init(&full[3], 8); mbar_fence_init(); }
  fence_proxy_async();                                 // tiles written through the generic proxy (here, or by peers and
  __syncthreads();                                     // already acquired) and the buffers' last contents -> bulk copies
  double* const Cb = sm + 4 * CG_TILE;
  if (tid == 0) {
    mbar_arrive_expect_tx(&full[0], 2u * CG_TILE * 8u);
    bulk_g2s(sm, cg_tile_ptr(g, i, kc), CG_TILE * 8, &full[0]);
    bulk_g2s(sm + CG_TILE, cg_tile_ptr(g, j, kc), CG_TILE * 8, &full[0]);
  }
  int abuf = 0, bsel = 0;
  uint32_t ph0 = 0, ph1 = 0, phc = 0;
  int t = 0;
  CGP_T(t_u);
  while (have) {
    const int ci = i, cj = j;
    // No CTA barrier inside the pipeline: a warp only waits for its operands; the ISSUING lane alone waits until all 8
    // warps have finished update t - 1 (whose buffers the copies below refill).  The duty rotates over the warps: a bulk
    // copy holds its issuing lane for a few hundred cycles, which the warp makes up while its neighbours issue.
    if (abuf == 0) { mbar_wait(&full[0], ph0); ph0 ^= 1u; } else { mbar_wait(&full[1], ph1); ph1 ^= 1u; }
    CGP_ADD(11, t_u);
    have = cg_next_tile(i, j, j1, nb, C, me);
    const bool newB = have && (j != cj);
    double* Ct = cg_tile_ptr(g, ci, cj);
    if (lane == 0 && w8 == (t & 7)) {
      if (t > 0) mbar_wait(&full[3], (uint32_t)(t - 1) & 1u);
      mbar_arrive_expect_tx(&full[2], CG_TILE * 8u);
      bulk_g2s(Cb, Ct, CG_TILE * 8, &full[2]);
      if (have) {
        mbar_arrive_expect_tx(&full[abuf ^ 1], (newB ? 2u : 1u) * CG_TILE * 8u);
        bulk_g2s(sm + (size_t)(abuf ^ 1) * 2 * CG_TILE, cg_tile_ptr(g, i, kc), CG_TILE * 8, &full[abuf ^ 1]);
        if (newB) bulk_g2s(sm + (size_t)(bsel ^ 1) * 2 * CG_TILE + CG_TILE, cg_tile_ptr(g, j, kc), CG_TILE * 8, &full[abuf ^ 1]);
      }
    }
    CGP_ADD(12, t_u);
    const double* As = sm + (size_t)abuf * 2 * CG_TILE;
    const double* Bs = sm + (size_t)bsel * 2 * CG_TILE + CG_TILE;
    double acc[4][2][2];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }
    const double* ap = As + (wm * 32 + (lane >> 2)) * CG_LD + (lane & 3);
    const double* bp = Bs + (wn * 16 + (lane >> 2)) * CG_LD + (lane & 3);
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
    CGP_ADD(13, t_u);
    mbar_wait(&full[2], phc); phc ^= 1u;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const int off = (wm * 32 + a * 8 + (lane >> 2)) * CG_LD + wn * 16 + b * 8 + 2 * (lane & 3);
        double2 o = *reinterpret_cast<const double2*>(Cb + off);
        o.x -= acc[a][b][0]; o.y -= acc[a][b][1];
        *reinterpret_cast<double2*>(Ct + off) = o;
      }
    CGP_ADD(14, t_u);
    __syncwarp();
    if (lane == 0) mbar_arrive(&full[3]);
    ++t;
    abuf ^= 1;
    if (newB) bsel ^= 1;
  }
  __syncthreads();
  if (tid == 0) {                                      // every phase of the barriers has been waited for: hand the words back
#pragma unroll
    for (int b = 0; b < 4; ++b) asm volatile("mbarrier.inval.shared::cta.b64 [%0];\n" :: "r"(smem_u32(&full[b])) : "memory");
  }
}

// Panel k: this CTA's tiles (i, k), i > k:  L_ik = A_ik L_kk^{-T},  r_i -= L_ik z_k.  All 8 warps work on a PAIR of tiles
// at a time (warp w owns rows 8w .. 8w+7 of both: the solve is a warp-private dependent chain of ~4 k cycles, so two
// independent chains per warp and eight warps side by side finish two tiles in little more than the latency of one), the
// pairs pass through two buffer pairs fed by bulk TMA one pair ahead, and every warp writes its own rows back as soon as
// they are solved; one CTA barrier per pair.  History (cycles per tile at N = 1024): two workers of four warps, a tile each,
// staged by cp.async and written back after a worker barrier 7.0 k (staging 2.4 k + solve 6.7 k + r update 1.9 k +
// write-back 1.4 k per round of two tiles, in sequence); one tile at a time on 8 warps with TMA prefetch 6.7 k.
template <int H>
__device__ __forceinline__ void cg_panel_tiles(const CholGroup& g, double* const (&Ts)[H], const int (&ti)[H], const double* Lk,
                                               const double* aux, int k, int w8, int lane) {
  const int row = w8 * 8 + (lane >> 2), q = lane & 3;
  double rold[H];                                      // r_i of this lane's rows: in flight during the solve
#pragma unroll
  for (int h = 0; h < H; ++h) rold[h] = (q == 0) ? __ldcg(g.r + ti[h] * CG_T + row) : 0.0;
  cg_trsm_dmma<H>(Ts, Lk, aux + CG_T, w8, lane);
  fence_proxy_async();                                 // the solved rows (st.shared) before a later bulk copy refills the buffer
#pragma unroll
  for (int h = 0; h < H; ++h) {                        // r_i -= L_ik z_k: four lanes per row, 16 columns each, fixed order
    const double* xr = Ts[h] + row * CG_LD;
    double s0 = 0.0;
#pragma unroll
    for (int m = 0; m < CG_T / 4; ++m) s0 = fma(xr[q + 4 * m], aux[q + 4 * m], s0);
    s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
    s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
    if (q == 0) g.r[ti[h] * CG_T + row] = rold[h] - s0;
  }
#pragma unroll
  for (int h = 0; h < H; ++h) {                        // the warp's 8 rows of L_ik back to global (512 B per row)
    double* At = cg_tile_ptr(g, ti[h], k);
#pragma unroll
    for (int rr = 0; rr < 8; ++rr) {
      const int off = (w8 * 8 + rr) * CG_LD + 2 * lane;
      *reinterpret_cast<double2*>(At + off) = *reinterpret_cast<const double2*>(Ts[h] + off);
    }
  }
}
__device__ __forceinline__ void cg_panel_phase(const CholGroup& g, double* sm, int k) {
  const int tid = threadIdx.x, w8 = tid >> 5, lane = tid & 31;
  const int nb = g.nb, C = g.C, me = g.rank;
  int i = k;
  auto next_mine = [&]() -> int { while (++i < nb) if (cg_owner(i, k, C) == me) return i; return -1; };
  int ia = next_mine();
  if (ia < 0) return;                                  // uniform across the CTA
  int ib = next_mine();
  __shared__ __align__(8) uint64_t pfull[3];           // L_kk, tile pairs 0 / 1
  double* const Lk = sm;
  double* const aux = sm + CG_NTILES * CG_TILE;        // z_k [64], inverted 8x8 diagonal blocks [8][8][8]
  if (tid == 0) { mbar_init(&pfull[0], 1); mbar_init(&pfull[1], 1); mbar_init(&pfull[2], 1); mbar_fence_init(); }
  fence_proxy_async();
  __syncthreads();
  if (tid == 0) {
    mbar_arrive_expect_tx(&pfull[0], CG_TILE * 8u);
    bulk_g2s(Lk, cg_tile_ptr(g, k, k), CG_TILE * 8, &pfull[0]);
    mbar_arrive_expect_tx(&pfull[1], (ib >= 0 ? 2u : 1u) * CG_TILE * 8u);
    bulk_g2s(sm + CG_TILE, cg_tile_ptr(g, ia, k), CG_TILE * 8, &pfull[1]);
    if (ib >= 0) bulk_g2s(sm + 2 * CG_TILE, cg_tile_ptr(g, ib, k), CG_TILE * 8, &pfull[1]);
  }
  {
    const double* Dg = g.Dinv + (size_t)k * CG_T * CG_T;
    if (tid < CG_T) aux[tid] = __ldcg(g.r + k * CG_T + tid);
    for (int e = tid; e < 8 * 64; e += CG_THREADS) aux[CG_T + e] = __ldcg(Dg + CG_T + e);
  }
  mbar_wait(&pfull[0], 0u);
  int buf = 0;
  uint32_t ph[2] = {0u, 0u};
  CGP_T(t_p);
  while (ia >= 0) {
    const int ca = ia, cb = ib;
    double* const T0 = sm + (size_t)(1 + 2 * buf) * CG_TILE;
    if (buf == 0) { mbar_wait(&pfull[1], ph[0]); ph[0] ^= 1u; } else { mbar_wait(&pfull[2], ph[1]); ph[1] ^= 1u; }
    __syncthreads();                                   // aux staged (first trip); everyone is done with the previous pair
    ia = (cb >= 0) ? next_mine() : -1;
    ib = (ia >= 0) ? next_mine() : -1;
    if (ia >= 0 && tid == 0) {
      double* const N0 = sm + (size_t)(1 + 2 * (buf ^ 1)) * CG_TILE;
      mbar_arrive_expect_tx(&pfull[1 + (buf ^ 1)], (ib >= 0 ? 2u : 1u) * CG_TILE * 8u);
      bulk_g2s(N0, cg_tile_ptr(g, ia, k), CG_TILE * 8, &pfull[1 + (buf ^ 1)]);
      if (ib >= 0) bulk_g2s(N0 + CG_TILE, cg_tile_ptr(g, ib, k), CG_TILE * 8, &pfull[1 + (buf ^ 1)]);
    }
    CGP_ADD(15, t_p);
    if (cb >= 0) {
      double* const Ts[2] = {T0, T0 + CG_TILE};
      const int ti[2] = {ca, cb};
      cg_panel_tiles<2>(g, Ts, ti, Lk, aux, k, w8, lane);
    } else {
      double* const Ts[1] = {T0};
      const int ti[1] = {ca};
      cg_panel_tiles<1>(g, Ts, ti, Lk, aux, k, w8, lane);
    }
    CGP_ADD(16, t_p);
    buf ^= 1;
  }
  __syncthreads();
  if (tid == 0) {
#pragma unroll
    for (int b = 0; b < 3; ++b) asm volatile("mbarrier.inval.shared::cta.b64 [%0];\n" :: "r"(smem_u32(&pfull[b])) : "memory");
  }
}

// One evaluation.  hyp (shared or global, [3 + d]): mean, amplitude, noise variance, 1/M_0 .. 1/M_{d-1}.
// sm: CG_SMEM_DOUBLES doubles of dynamic shared memory (16-byte aligned).  epoch: number of evaluations this cluster
// has completed on these flags (identical in every CTA).  Returns the log-likelihood (-inf when not positive definite
// or not finite) to every thread of every CTA of the cluster.  Ends with a CTA barrier.
template <bool FAST_PIVOT>
__device__ double chol_group_loglik(const CholGroup& g, const double* hyp, double* sm, unsigned long long epoch) {
  const int tid = threadIdx.x, w = tid >> 7, wtid = tid & 127;
  const int nb = g.nb, C = g.C, me = g.rank, d = g.d;
  double* As = sm + (size_t)w * 2 * CG_TILE;
  double* Bs = As + CG_TILE;
  const unsigned long long baseA = epoch * (unsigned long long)(nb + 1);
  const unsigned long long baseB = epoch * (unsigned long long)(nb - 1) * C;       // one increment per CTA per panel
  double* part = g.part + (size_t)(epoch & 1ull) * nb * 4;
  const double mean = hyp[0], amp = hyp[1], noise = hyp[2];
  __shared__ int s_bad;
  CGP_T(t_all);
  CGP_T(t_ph);

  // ---- build: every CTA forms its own tiles; the owner of (i, 0) also initialises r_i = y_i - mean --------------
  // K_ij = amp exp(-sum_c (xs_ic - xs_jc)^2) with the inputs pre-scaled by sqrt(1 / (2 M_c)) while they are staged and
  // the table exponential of the predict kernels (<= 2 ulp): 2 d + 12 FP64 operations per entry.
  double* etab = sm + CG_NTILES * CG_TILE + 2 * CG_AUX;     // [64] 2^(j/64)
  double* scl = etab + 64;                          // [d]
  if (tid < 64) etab[tid] = exp2((double)tid * (1.0 / 64.0));
  else if (tid < 64 + d) scl[tid - 64] = sqrt(0.5 * hyp[3 + tid - 64]);
  __syncthreads();
  {
    // this worker's tiles in column-major order (the first block columns are needed first).  The raw inputs of the NEXT
    // tile's row block travel in registers while the current tile is evaluated (staging them at the top of each tile cost
    // 3.5 k cycles of exposed global-memory latency per tile)
    int t = 0, staged_j = -1, i = -1, j = 0;
    auto next_mine = [&]() -> bool {
      for (;;) {
        if (++i >= nb) { ++j; i = j; }
        if (j >= nb) return false;
        if (cg_owner(i, j, C) == me && (t++ & 1) == w) return true;
      }
    };
    constexpr int NPRE = CG_T * APGP_MAXD / CG_WT;                 // 16 values per thread at d = 32
    double pre[NPRE];
    auto fetch = [&](int ib) {                                     // rows ib*64.. of X are one contiguous run of 64 d values
      const int lim = min(CG_T, g.N - ib * CG_T) * d;
#pragma unroll
      for (int m = 0; m < NPRE; ++m) {
        const int e = wtid + m * CG_WT;
        pre[m] = (e < lim) ? g.X[(size_t)ib * CG_T * d + e] : 0.0;
      }
    };
    bool have = next_mine();
    if (have) fetch(i);
    while (have) {
      const int ci = i, cj = j;
      {
        CGP_T(t_b);
        // both row blocks TRANSPOSED and pre-scaled: rows ci*64.. in As ([d][64]: a thread reads 16 consecutive rows of
        // one dimension as 8 warp-wide LDS.128 broadcasts), rows cj*64.. in Bs ([d][64]: the 64 columns of the tile read
        // conflict-free; kept while the worker stays in block column cj)
        {
          int rr = wtid / d, c = wtid - rr * d;
          const int drr = CG_WT / d, dc = CG_WT - drr * d;
#pragma unroll
          for (int m = 0; m < NPRE; ++m) {
            if (wtid + m * CG_WT < CG_T * d) As[c * CG_T + rr] = pre[m] * scl[c];
            rr += drr; c += dc;
            if (c >= d) { c -= d; ++rr; }
          }
        }
        if (staged_j != cj) {
          staged_j = cj;
          for (int e = wtid; e < CG_T * d; e += CG_WT) {
            const int c2 = e >> 6, r2 = e & 63;
            const int gj = cj * CG_T + r2;
            Bs[e] = (gj < g.N) ? g.X[(size_t)gj * d + c2] * scl[c2] : 0.0;
          }
        }
        have = next_mine();
        if (have) fetch(i);
        named_bar_sync(1 + w, CG_WT);
        CGP_ADD(19, t_b);
        double* Kt = cg_tile_ptr(g, ci, cj);
        {
          // one column per thread, sixteen consecutive rows per pass: sixteen independent distance / exponential chains
          // (the one-entry-per-pass loop with libdevice exp was bound by its own dependent latency: 27 k cycles per tile)
          const int cc = wtid & 63, rh = wtid >> 6;
          const int gj = cj * CG_T + cc;
#pragma unroll 1
          for (int pass = 0; pass < 2; ++pass) {
            const int rbase = rh * 32 + pass * 16;
            double s16[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) s16[u] = 0.0;
            for (int c = 0; c < d; ++c) {
              const double bv = Bs[c * CG_T + cc];
              const double2* ar = reinterpret_cast<const double2*>(As + c * CG_T + rbase);
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const double2 av = ar[u];
                const double d0 = av.x - bv, d1 = av.y - bv;
                s16[2 * u] = fma(d0, d0, s16[2 * u]); s16[2 * u + 1] = fma(d1, d1, s16[2 * u + 1]);
              }
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) {
              const int rr = rbase + u, gi = ci * CG_T + rr;
              double v;
              if (gi < g.N && gj < g.N) {
                v = __dmul_rn(amp, exp_neg(s16[u], etab));
                if (gi == gj) v = __dadd_rn(v, noise);
              } else {
                v = (gi == gj) ? 1.0 : 0.0;
              }
              Kt[rr * CG_LD + cc] = v;
            }
          }
        }
        if (cj == 0 && wtid < CG_T) {
          const int gi = ci * CG_T + wtid;
          g.r[gi] = (gi < g.N) ? (g.y[gi] - mean) : 0.0;
        }
        named_bar_sync(1 + w, CG_WT);
        CGP_ADD(20, t_b);
      }
    }
  }
  __syncthreads();
  CGP_ADD(0, t_ph);

  for (int k = 0; k < nb; ++k) {
    // ---- (1) diagonal block k: factor, invert, z_k, partial sums -- by its owner, all 256 threads -------------------
    if (cg_owner(k, k, C) == me) {
      double* S = sm;                                   // packed lower triangle
      double* R = S + CG_T * (CG_T + 1) / 2;            // [CG_DIAG_LDR]: r_k -> z_k
      double* dg = R + CG_DIAG_LDR;                     // [64] pivots
      double* A = cg_tile_ptr(g, k, k);
      double* rk = g.r + k * CG_T;
      if (tid == 0) s_bad = 0;
      for (int e = tid; e < CG_T * CG_T; e += CG_THREADS) {
        const int i = e >> 6, j = e & 63;
        if (j <= i) S[i * (i + 1) / 2 + j] = A[i * CG_LD + j];          // own tile: written by this CTA only
      }
      if (tid < CG_T) R[tid] = __ldcg(rk + tid);                              // r_k was updated by other CTAs' panels
      __syncthreads();
      CGP_ADD(1, t_ph);
      chol_packed_blocked<CG_THREADS, FAST_PIVOT>(S, R, dg, CG_T, &s_bad, true, 1, CG_DIAG_LDR);
      CGP_ADD(2, t_ph);
      // the factored block goes back row-major (the panel solves read it); its reciprocal pivots and the inverses of
      // its eight 8x8 diagonal blocks go into the block's slot of Dinv ([0, 64): 1 / L_cc; [64, 576): inv[J][n][k]) --
      // the panel tiles are solved blockwise on the tensor pipe (cg_trsm_dmma), never through a full 64x64 inverse
      double* Dg = g.Dinv + (size_t)k * CG_T * CG_T;
      for (int e = tid; e < CG_T * CG_T; e += CG_THREADS) {
        const int i = e >> 6, j = e & 63;
        A[i * CG_LD + j] = (j <= i) ? S[i * (i + 1) / 2 + j] : 0.0;
      }
      if (tid < CG_T) { Dg[tid] = 1.0 / dg[tid]; rk[tid] = R[tid]; }
      else if (tid < 2 * CG_T) {
        // thread (J, col): column col of the inverse of diagonal block J by forward substitution (uniform trip counts:
        // the entries above col are exact zeros)
        const int J = (tid - CG_T) >> 3, col = tid & 7;
        double x[8], rinv[8];
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) rinv[rr] = 1.0 / dg[8 * J + rr];
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          const int gr = 8 * J + rr;
          double acc = (rr == col) ? 1.0 : 0.0;
#pragma unroll
          for (int mm = 0; mm < rr; ++mm) acc = fma(-S[gr * (gr + 1) / 2 + 8 * J + mm], x[mm], acc);
          x[rr] = acc * rinv[rr];
          Dg[CG_T + J * 64 + rr * 8 + col] = x[rr];
        }
      }
      if (tid < 32) {                                                          // block partials, fixed order
        double zz = __dadd_rn(__dmul_rn(R[tid], R[tid]), __dmul_rn(R[tid + 32], R[tid + 32]));
        double lg = log(dg[tid]) + log(dg[tid + 32]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { zz += __shfl_xor_sync(0xffffffffu, zz, o); lg += __shfl_xor_sync(0xffffffffu, lg, o); }
        if (tid == 0) { part[k * 4 + 0] = zz; part[k * 4 + 1] = lg; part[k * 4 + 2] = s_bad ? 1.0 : 0.0; }
      }
      if (C > 1) cg_publish_store(g.flagA, baseA + k + 1); else __syncthreads();
      CGP_ADD(3, t_ph);
    }
    // ---- (2) deferred trailing work of step k-1 (columns >= k+1) and (3) panel k: L_ik = A_ik L_kk^{-T} on the tensor pipe,
    //      r_i -= L_ik z_k.  They touch different tiles, so their order is free: the CTA that has just factored block k
    //      solves its panel tiles FIRST (the rest of the cluster needs them to pass flag B) and catches up on the deferred
    //      work afterwards; everyone else does the deferred work under the owner's pivot chain and the panel after flag A.
    if (C > 1 && k < nb - 1 && cg_owner(k, k, C) == me) {
      cg_panel_phase(g, sm, k);
      CGP_ADD(6, t_ph);
      cg_publish_add(g.cntB);
      if (k > 0) cg_update_phase(g, sm, k - 1, k + 1, nb);
      CGP_ADD(4, t_ph);
      cg_wait_ge(g.cntB, baseB + (unsigned long long)(k + 1) * C);
      CGP_ADD(7, t_ph);
    } else {
      if (k > 0) {
        cg_update_phase(g, sm, k - 1, k + 1, nb);
        CGP_ADD(4, t_ph);
      }
      if (k == nb - 1) break;
      if (C > 1) cg_wait_ge(g.flagA, baseA + k + 1);
      CGP_ADD(5, t_ph);
      cg_panel_phase(g, sm, k);
      CGP_ADD(6, t_ph);
      if (C > 1) { cg_publish_add(g.cntB); cg_wait_ge(g.cntB, baseB + (unsigned long long)(k + 1) * C); } else __syncthreads();
      CGP_ADD(7, t_ph);
    }
    // ---- (4) urgent part of step k: column k+1 (the next diagonal block and the next panel's inputs) --------------
    cg_update_phase(g, sm, k, k + 1, k + 2);
    CGP_ADD(8, t_ph);
  }

  // ---- log-likelihood: block partials in block order (identical bits in every CTA) -----------------------------------
  if (C > 1) cg_wait_ge(g.flagA, baseA + nb);
  double zz = 0.0, lg = 0.0, bad = 0.0;
  for (int k = 0; k < nb; ++k) { zz += __ldcg(part + k * 4); lg += __ldcg(part + k * 4 + 1); bad += __ldcg(part + k * 4 + 2); }
  double ll = __dsub_rn(__dsub_rn(__dmul_rn(-0.5, zz), lg), __dmul_rn(__dmul_rn(0.5, (double)g.N), 1.8378770664093454836));
  if (bad != 0.0 || !(ll == ll) || !(fabs(ll) < INFINITY)) ll = -INFINITY;
  __syncthreads();
  CGP_ADD(9, t_ph);
  CGP_ADD(10, t_all);
  return ll;
}

}  // namespace apgp
