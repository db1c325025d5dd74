// Grouped variance predict on the int8 tensor cores (tcgen05.mma.kind::i8): the triangular product
// W = E . (A L^{-1})^T of predict.cu's grouped kernel, computed exactly in integer arithmetic (Ozaki split).
//
//   E[q,k] in [0,1]  -> fixed 2^-55 grid, 7 unsigned base-256 digits e_p (top digit <= 128)
//   B = A L^{-1}     -> per row i a power-of-two scale 2^(ex_i - 55), 7 balanced signed digits b_r in [-127,127]
//                       at the top, [-128,127] below
//   W[q,i] = 2^(ex_i - 14) * sum_{s=0..7} 2^(-8 s) * acc_s,   acc_s = sum_k sum_{p+r=s} e_p[q,k] b_r[i,k]
// The 34 digit products with p + r <= 7 are kept (the dropped levels 8..12 weigh 2^-64 and less against level 0).
// Each level accumulates in int32 in tensor memory: <= 7 pairs x N x 255 x 128 < 2^31 for N <= 8192.  The integer sums are exact, so a
// query's variance does not depend on the accumulation order, its position in the batch or the group size.
//
// Tile: 128 queries x 64 rows of B per block-row, K staged 64 at a time; 8 levels x 64 int32 columns fill the 512
// TMEM columns, level s at columns 64 s.  Operands use the no-swizzle K-major canonical layout of 8-row x 16-byte
// core matrices.  A (panel) stages are [plane][k16 chunk][8-row group][8 rows][16 bytes]; B (LinvI8) stages are
// [k16 chunk][plane][8-row group][8 rows][16 bytes], so B's planes r0, r0+1, ... follow each other along N and one
// MMA of N = 64 n multiplies A plane p by n of them into n adjacent levels (i8_sched: 11 MMAs per 32-wide k-step
// instead of one 128 x 64 x 32 MMA per digit pair, which read the 4 KB A tile once per 64 output columns and left
// the MMAs bound by shared-memory operand reads).  Inside a 16-wide k chunk byte c holds k = c/4 + 4 (c%4): one
// phase-1 thread builds k = l, l+4, l+8, l+12 (the DMMA kernel's order, so the mean is bit-identical) and stores
// them as one 32-bit word.  A and B use the same permutation; an exact integer sum does not see it.
//
// Warps: 0-7 build the panel (phase 1) and run the per-block-row epilogue (tcgen05.ld, combine, W^2 row sums);
// warp 8 lane 0 streams digit tiles with 1-D bulk TMA; warp 9 owns the TMEM allocation and its lane 0 issues MMAs.
#include "predict_tile.cuh"
#include <stdio.h>
#include <stdlib.h>

namespace apgp {

namespace {

constexpr int I8_BM = 128, I8_BN = 64, I8_BK = 64, I8_NST = 2;
constexpr int I8_DIG = 7, I8_LEVELS = 8;
constexpr int I8_A_STAGE = I8_DIG * I8_BM * I8_BK;      // bytes: 57344
constexpr int I8_B_STAGE = I8_DIG * I8_BN * I8_BK;      // bytes: 28672
constexpr int I8_STAGE = I8_A_STAGE + I8_B_STAGE;
constexpr int I8_RING = I8_NST * I8_STAGE;
constexpr int I8_NTHREADS = 10 * 32;

// -DAPGP_PROF: SM cycles per phase for the first I8_PROF_CTAS CTAs, summed over the tiles of a call and printed by
// launch_predict_var_i8 when APGP_PROF_PRINT is set (tools/profile_var_i8_phases.py).  Thread 0: 0 phase 1 (panel
// build, to the end-of-phase barrier), 1 group-barrier wait, 2 finaliser, 7 phase 2 (epilogue warps' view, to the
// end-of-tile barrier), 8 whole kernel.  MMA lane: 3 waiting on full[] (operands late), 4 waiting on accempty (the
// epilogue still reads the previous block-row), 5 MMA issue, 6 waiting for the last block-row's epilogue.  Counts:
// 9 tiles, 10 panel blocks built, 11 phase-2 units (64-wide k-stages) issued.
#ifdef APGP_PROF
constexpr int I8_PROF_CTAS = 4, I8_PROF_SLOTS = 12;
__device__ long long g_i8prof[I8_PROF_CTAS][I8_PROF_SLOTS];
#define I8P_T(var) long long var = clock64()
#define I8P_SET(var) ((var) = clock64())
#define I8P_CNT(slot, n) do { if (blockIdx.x < I8_PROF_CTAS) g_i8prof[blockIdx.x][slot] += (n); } while (0)
#define I8P_ADD(slot, t0) do { if (blockIdx.x < I8_PROF_CTAS) { const long long _n = clock64(); g_i8prof[blockIdx.x][slot] += _n - (t0); (t0) = _n; } } while (0)
#else
#define I8P_T(var) do {} while (0)
#define I8P_SET(var) do {} while (0)
#define I8P_CNT(slot, n) do {} while (0)
#define I8P_ADD(slot, t0) do {} while (0)
#endif

size_t i8_smem_bytes(int d) { return (size_t)I8_RING + (size_t)d * I8_BM * 8 + 64 * 8 + 8 * 8 + 128; }

// no-swizzle K-major shared-memory matrix descriptor (sm_100: version bits 46-48 = 0b001)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
         (1ull << 46);
}
// kind::i8 instruction descriptor: D s32, A u8, B s8, both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t i8_idesc(int n) {
  return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(I8_BM >> 4) << 24);
}

// The MMAs of one 32-wide k-step.  B's digit planes are stacked along N inside a k16 chunk, so one MMA multiplies A
// plane p by B planes r0 .. r0 + n - 1 (N = 64 n) into the contiguous level accumulators p + r0 .. p + r0 + n - 1,
// TMEM columns 64 (p + r0) onward: 11 MMAs for the 34 digit products with p + r <= 7, each 4 KB A tile read once per
// up to 256 output columns.  The accumulate flag covers a whole MMA, so the order is chosen such that on a
// block-row's first k-step each MMA either writes only levels no earlier MMA has written (it overwrites: level 7
// first comes from {3, 4, 1}) or only levels some earlier MMA has (it accumulates).
struct I8Mma { int p, r0, n; };
constexpr int I8_NMMA = 11;
__host__ __device__ constexpr I8Mma i8_sched(int j) {
  constexpr I8Mma t[I8_NMMA] = {{0, 0, 4}, {0, 4, 3}, {3, 4, 1}, {1, 0, 4}, {1, 4, 3}, {2, 0, 4},
                                {2, 4, 2}, {3, 0, 4}, {4, 0, 4}, {5, 0, 3}, {6, 0, 2}};
  return t[j];
}

// how many of the levels of MMA j an earlier MMA of the step has written
__host__ __device__ constexpr int i8_levels_written_before(int j) {
  const I8Mma m = i8_sched(j);
  int cnt = 0;
  for (int l = m.p + m.r0; l < m.p + m.r0 + m.n; ++l) {
    bool w = false;
    for (int i = 0; i < j; ++i) {
      const I8Mma e = i8_sched(i);
      w = w || (l >= e.p + e.r0 && l < e.p + e.r0 + e.n);
    }
    cnt += w;
  }
  return cnt;
}
__host__ __device__ constexpr bool i8_sched_ok() {
  int covered[I8_DIG][I8_DIG] = {};
  for (int j = 0; j < I8_NMMA; ++j) {
    const I8Mma m = i8_sched(j);
    if (m.p < 0 || m.p >= I8_DIG || m.r0 < 0 || m.n < 1 || m.n > 4 || m.r0 + m.n > I8_DIG) return false;
    if ((m.p + m.r0 + m.n) * I8_BN > 512) return false;                        // inside the TMEM allocation
    const int w = i8_levels_written_before(j);
    if (w != 0 && w != m.n) return false;                                       // one accumulate flag serves all its levels
    for (int r = m.r0; r < m.r0 + m.n; ++r) ++covered[m.p][r];
  }
  for (int pa = 0; pa < I8_DIG; ++pa)
    for (int rb = 0; rb < I8_DIG; ++rb)
      if (covered[pa][rb] != (pa + rb < I8_LEVELS ? 1 : 0)) return false;       // every kept product exactly once
  return true;
}
static_assert(i8_sched_ok(), "i8_sched must cover each digit product with p + r <= 7 exactly once, inside 512 TMEM "
                             "columns, with all of an MMA's levels fresh or all already written");

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
               :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// round(e * 2^55) for 0 <= e <= 1 from the bits of e (integer pipe only); ties round up
__device__ __forceinline__ unsigned long long fixed55(double e) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(e);
  const int ex = (int)(b >> 52);
  const int sh = 1023 - ex;
  if (ex == 0 || sh > 56) return 0ull;
  const unsigned long long m = ((b & 0xFFFFFFFFFFFFFull) | (1ull << 52)) << 3;
  return sh <= 0 ? m : ((m >> (sh - 1)) + 1ull) >> 1;
}
// byte `byte` (0 = least significant) of four 64-bit values, packed into one word (value j -> byte j)
__device__ __forceinline__ uint32_t gather_byte(const uint32_t (&lo)[4], const uint32_t (&hi)[4], int byte) {
  const uint32_t* w = byte >= 4 ? hi : lo;
  const uint32_t bb = (uint32_t)(byte & 3);
  const uint32_t sel = bb | ((bb + 4u) << 4);
  return __byte_perm(__byte_perm(w[0], w[1], sel), __byte_perm(w[2], w[3], sel), 0x5410);
}

// phase 1's store (panel_columns): the four kernel values of m8 query block mg at columns jb + lane % 4 + {0, 4, 8, 12}
// of 64-column block cb, as round(E 2^55) in the 7 digit planes of the block's A stage, most significant first; the
// four values form one 32-bit word of each plane
__device__ __forceinline__ void store_i8_panel(unsigned char* panel, int cb, int jb, int mg, int lane, const double (&e)[4]) {
  uint32_t lo[4], hi[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const unsigned long long v = fixed55(e[j]);
    lo[j] = (uint32_t)v; hi[j] = (uint32_t)(v >> 32);
  }
  uint32_t* dst = reinterpret_cast<uint32_t*>(panel + (size_t)cb * I8_A_STAGE + ((size_t)(jb >> 4) * 16 + mg) * 128 +
                                              (lane >> 2) * 16 + (lane & 3) * 4);
#pragma unroll
  for (int pl = 0; pl < I8_DIG; ++pl) dst[pl * (4 * 16 * 128 / 4)] = gather_byte(lo, hi, 6 - pl);
}

__global__ void __launch_bounds__(I8_NTHREADS, 1)
predict_var_i8_kernel(const __grid_constant__ PredictParams p, const int G) {
  constexpr int BM = I8_BM, BN = I8_BN, NCW = 8, NCONS = NCW * 32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* ring = smem_raw;
  double* qs = reinterpret_cast<double*>(smem_raw + I8_RING);   // [d][BM] scaled queries
  double* etab = qs + (size_t)p.d * BM;                          // [64]
  uint64_t* full = reinterpret_cast<uint64_t*>(etab + 64);
  uint64_t* empty = full + I8_NST;
  uint64_t* stagebar = empty + I8_NST;
  uint64_t* accfull = stagebar + 1;
  uint64_t* accempty = accfull + 1;
  __shared__ int owner_s[GROUP_MAX_BLOCKS];
  __shared__ int myblk_s[GROUP_MAX_BLOCKS];
  __shared__ int nmine_s;
  __shared__ double mu_keep[2][BM];
  __shared__ double ss_s[BM];
  __shared__ uint32_t tmem_base_s;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  I8P_T(tk);
  I8P_T(tp);
  I8P_T(tm);
  const int Npad = p.Npad;
  const GroupCtx<BM, BN> g(p, G);
  const int nblk = g.nblk, rank = g.rank;
  unsigned char* scratch8 = reinterpret_cast<unsigned char*>(p.scratch);

  if (tid == 0) {                                        // before init_tile_smem, whose fence covers these too
    mbar_init(accfull, 1);
    mbar_init(accempty, NCONS);
  }
  init_tile_smem<I8_NST>(etab, full, empty, stagebar, 1);   // empty[s]: one tcgen05.commit per stage
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n"
                 :: "r"(smem_u32(&tmem_base_s)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  g.load_plan(p, G, owner_s, myblk_s, &nmine_s);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const int nmine = nmine_s;
  const uint32_t tmem = tmem_base_s;

  uint32_t it = 0, nstaged = 0, nacc = 0;
  int nbar = 0;

  for (long long tile = g.t_begin; tile <= g.t_end; ++tile) {
    const int b = (int)((tile - g.t_begin) & 1);
    const bool live = tile < g.t_end;
    unsigned char* panel = scratch8 + ((size_t)g.grp * 2 + b) * BM * (size_t)Npad * I8_DIG;
    if (tid == 0 && live) { I8P_CNT(9, 1); I8P_CNT(10, nmine); }

    // ------------------------------------------------------------ phase 1: my column blocks of the digit panel
    if (live && warp < NCW) {
      group_phase1<BM, BN, NCW>(p, tile * BM, qs, etab, reinterpret_cast<double*>(ring), I8_RING / 8, myblk_s, nmine,
                                stagebar, nstaged, g.part_mu + (size_t)b * nblk * BM,
                                [&](int cb, int jb, int mg, const double (&e)[4]) { store_i8_panel(panel, cb, jb, mg, lane, e); });
      __threadfence();
    }
    __syncthreads();
    if (tid == 0) I8P_ADD(0, tp);

    g.barrier(nbar);
    if (tid == 0) I8P_ADD(1, tp);
    // a NaN query has NaN kernel values, which reach the mean but not the panel (fixed55 has no NaN digits)
    g.finalise(p, tile, live, b, mu_keep, [&](double mu, double tot) { return isnan(mu) ? mu : p.amp - tot; });
    if (tid == 0) I8P_ADD(2, tp);
    if (!live) break;

    // ------------------------------------------------------------ phase 2: my block-rows on the int8 tensor cores
    if (warp == NCW) {
      if (lane == 0)
        stream_operands<I8_NST, I8_A_STAGE, I8_B_STAGE, 1>(ring, panel, p.LinvI8, nblk, full, empty, it,
                                                           [&](int ib) { return owner_s[ib] == rank; });
    } else if (warp == NCW + 1) {
      if (lane == 0) {
        I8P_SET(tm);
        for (int ib = 0; ib < nblk; ++ib) {
          if (owner_s[ib] != rank) continue;
          mbar_wait(accempty, (nacc & 1u) ^ 1u);         // the epilogue has read the previous block-row
          I8P_ADD(4, tm);
          tc_fence_after();
          for (int kb = 0; kb <= ib; ++kb, ++it) {
            const int s = it % I8_NST;
            const uint32_t ph = (it / I8_NST) & 1u;
            mbar_wait(&full[s], ph);
            I8P_ADD(3, tm);
            tc_fence_after();
            const uint32_t sa = smem_u32(ring + (size_t)s * I8_STAGE);
            const uint32_t sb = sa + I8_A_STAGE;
#pragma unroll
            for (int kk = 0; kk < I8_BK / 32; ++kk) {
#pragma unroll
              for (int j = 0; j < I8_NMMA; ++j) {
                const I8Mma m = i8_sched(j);
                const uint64_t da = umma_desc(sa + (m.p * 4 + 2 * kk) * 2048, 2048, 128);
                const uint64_t db = umma_desc(sb + (2 * kk * I8_DIG + m.r0) * 1024, I8_DIG * 1024, 128);
                const bool first = kb == 0 && kk == 0 && i8_levels_written_before(j) == 0;
                umma_i8(tmem + (m.p + m.r0) * BN, da, db, i8_idesc(m.n * BN), first ? 0u : 1u);
              }
            }
            umma_commit(&empty[s]);                       // stage free once these MMAs have read it
            I8P_ADD(5, tm);
            I8P_CNT(11, 1);
          }
          umma_commit(accfull);
          ++nacc;
        }
        I8P_ADD(5, tm);
      }
    } else {
      // epilogue: warp w reads TMEM lanes 32 (w % 4) .. + 31 (its queries), columns 32 (w / 4) .. + 31 of each level
      const int quarter = warp & 3, half = warp >> 2;
      const int m = quarter * 32 + lane;
      const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16) + half * 32;
      for (int ib = 0; ib < nblk; ++ib) {
        if (owner_s[ib] != rank) continue;
        mbar_wait(accfull, nacc & 1u);
        ++nacc;
        tc_fence_after();
        const double* sc = p.i8scale + ib * BN + half * 32;
        double ss = 0.0;
#pragma unroll 1
        for (int c0 = 0; c0 < 32; c0 += 8) {
          uint32_t v[I8_LEVELS][8];
#pragma unroll
          for (int lev = 0; lev < I8_LEVELS; ++lev) tmem_ld8(tl + lev * BN + c0, v[lev]);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            long long hi = (int)v[0][j], lo = (int)v[4][j];
#pragma unroll
            for (int lev = 1; lev < 4; ++lev) {
              hi = hi * 256 + (int)v[lev][j];
              lo = lo * 256 + (int)v[4 + lev][j];
            }
            const double w = fma((double)lo, 0x1p-32, (double)hi) * __ldg(sc + c0 + j);
            ss = fma(w, w, ss);
          }
        }
        tc_fence_before();
        if (half == 1) ss_s[m] = ss;
        named_bar_sync(1, NCONS);
        if (half == 0) g.part_ss[((size_t)b * nblk + ib) * BM + m] = ss + ss_s[m];
        mbar_arrive(accempty);
      }
      __threadfence();
    }
    __syncthreads();
    if (tid == 0) I8P_ADD(7, tp);
    if (warp == NCW + 1 && lane == 0) I8P_ADD(6, tm);
  }

  if (tid == 0) I8P_ADD(8, tk);
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// Operand pack: one CTA per padded row i of B = A L^{-1}.  Row scale 2^(ex_i - 38) (the combine's 2^(ex_i - 14) and
// the hi/lo split's 2^-24), zero for padding rows; digits of round(B[i,k] 2^(55 - ex_i)) with |.| <= 127 * 2^48.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pack_linv_i8_kernel(const double* __restrict__ Linv, int ld, int N, double amp, unsigned char* __restrict__ out,
                    double* __restrict__ rowscale) {
  __shared__ double red[8];
  const int i = blockIdx.x, tid = threadIdx.x;
  const int ib = i / I8_BN, ng = (i / 8) % 8, row = i % 8;
  double mx = 0.0;
  if (i < N)
    for (int k = tid; k <= i; k += blockDim.x) mx = fmax(mx, fabs(amp * Linv[(size_t)i * ld + k]));
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((tid & 31) == 0) red[tid >> 5] = mx;
  __syncthreads();
  mx = 0.0;
  for (int w = 0; w < 8; ++w) mx = fmax(mx, red[w]);
  int ex = 0;
  if (mx > 0.0) {
    ex = ilogb(mx) + 1;                                  // mx < 2^ex
    if (mx > ldexp(127.0 / 128.0, ex)) ++ex;             // top digit <= 127 after balanced rounding
  }
  if (tid == 0) rowscale[i] = mx > 0.0 ? ldexp(1.0, ex - 38) : 0.0;
  unsigned char* tile0 = out + ((size_t)ib * (ib + 1) / 2) * I8_B_STAGE;
  for (int kk = tid; kk < (ib + 1) * I8_BK; kk += blockDim.x) {
    const int kb = kk / I8_BK, kc = (kk / 16) % 4, c = kk % 16;
    const int k = kb * I8_BK + kc * 16 + (c >> 2) + 4 * (c & 3);
    long long X = 0;
    if (i < N && k <= i && mx > 0.0) X = llrint(ldexp(amp * Linv[(size_t)i * ld + k], 55 - ex));
    unsigned char* t = tile0 + (size_t)kb * I8_B_STAGE + ((kc * I8_DIG) * 8 + ng) * 128 + row * 16 + c;
    for (int r = I8_DIG - 1; r >= 1; --r) {
      const int dg = (int)(signed char)(X & 0xff);
      X = (X - dg) >> 8;
      t[r * (8 * 128)] = (unsigned char)dg;
    }
    t[0] = (unsigned char)(signed char)X;
  }
}

}  // namespace

// The planner's unit for this engine is one 64-wide k-stage of a 128-query block-row on the int8 pipe; a panel block is
// estimated at ~0.86 units at d = 5 (2.5 times the DMMA tile's estimate).  The -DAPGP_PROF phase profile
// (profiles/r04_i8_phases_after.txt, cfg3) measures 3.5 units (a factor of 10); that value moves G at many padded
// sizes that are not powers of two and has not been timed there, so the estimate stays until it has (DESIGN 4.1a)
// The largest d is the DMMA tile's 27, the engine's range since it was introduced: its own shared memory would take d up
// to 31 (predict_i8_fits), but the engine has not been tested or timed beyond 27.
const GroupTile I8_GROUP_TILE = {I8_BM, I8_DIG, 2.5, 27};

size_t linv_i8_bytes(int Npad) {
  const size_t nblk = (size_t)Npad / I8_BN;
  return nblk * (nblk + 1) / 2 * I8_B_STAGE;
}

int launch_pack_linv_i8(const double* Linv, int ld, int N, int Npad, double amp, unsigned char* out, double* rowscale,
                        cudaStream_t st) {
  pack_linv_i8_kernel<<<Npad, 256, 0, st>>>(Linv, ld, N, amp, out, rowscale);
  return (int)cudaGetLastError();
}

bool predict_i8_fits(int Npad, int d) {
  return Npad % I8_BN == 0 && Npad / I8_BN <= GROUP_MAX_BLOCKS && i8_smem_bytes(d) <= 200 * 1024;
}

int launch_predict_var_i8(const PredictParams& p, int num_sms, int G, cudaStream_t st, int* launches) {
  if (p.Q <= 0) return 0;
  const size_t smem = i8_smem_bytes(p.d);
  static PerDeviceOnce attr;
  if (attr.needed()) {
    cudaError_t e = cudaFuncSetAttribute(predict_var_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         200 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr.mark();
  }
  const int e = launch_grouped((const void*)predict_var_i8_kernel, p, num_sms, G, I8_NTHREADS, smem, st, launches);
#ifdef APGP_PROF
  if (getenv("APGP_PROF_PRINT")) {
    cudaStreamSynchronize(st);
    long long h[I8_PROF_CTAS][I8_PROF_SLOTS];
    cudaMemcpyFromSymbol(h, g_i8prof, sizeof(h));
    for (int c = 0; c < I8_PROF_CTAS; ++c) {
      fprintf(stderr, "[i8prof] Npad=%d Q=%lld G=%d cta=%d cycles:", p.Npad, p.Q, G, c);
      for (int i = 0; i < I8_PROF_SLOTS; ++i) fprintf(stderr, " %lld", h[c][i]);
      fprintf(stderr, "\n");
    }
    long long z[I8_PROF_CTAS][I8_PROF_SLOTS] = {};
    cudaMemcpyToSymbol(g_i8prof, z, sizeof(z));
  }
#endif
  return e;
}

}  // namespace apgp
