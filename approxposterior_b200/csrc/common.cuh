// Shared device helpers for the sm_100a GP-surrogate kernels (libapgp).
//   * DMMA.8x8x4 wrapper (the only FP64 tensor instruction on sm_100a: every
//     mma.sync f64 shape lowers to it -- see profiles/r01_fp64_pipe_probe.txt)
//   * mbarrier + 1-D bulk TMA (cp.async.bulk -> SASS UBLKCP) wrappers
//   * fragment-order index helpers shared by the packers and the consumers
//   * fixed-order CTA sum
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define APGP_MAXD 32          // max input dimensionality carried in kernel params

namespace apgp {

// ---------------------------------------------------------------------------------
// FP64 tensor-core MMA: C(8x8) += A(8x4) * B(4x8).
//   lane l holds A[row=l/4][k=l%4], B[k=l%4][n=l/4], C[row=l/4][col=2*(l%4)+{0,1}]
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// fixed-order sum over a CTA of NT threads, the same bits in every thread; red: NT / 32 doubles of shared memory
template <int NT>
__device__ __forceinline__ double cta_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();                      // red free to overwrite
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < NT / 32; ++w) t += red[w];
  return t;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------------------------
// mbarrier (shared::cta) + bulk async copy
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
               :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk TMA: global -> shared, completion counted in bytes on `bar`.
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
               :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// generic-proxy writes -> async-proxy (TMA) reads ordering
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async;\n" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;\n" :: "r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------
// Fragment-tiled storage of A * L^{-1} for the predict GEMM  W = K* . (A L^{-1})^T
//   block-row ib (BN rows) x k-step kb (16 columns), only kb*16 < (ib+1)*BN stored: tile (ib, kb) is tile
//   (BN/16) ib(ib+1)/2 + kb (stream_operands, pack_linv_kernel).
//   inside a tile: [k4 (4)][n8 (BN/8)][lane (32)],  lane <-> (n = n8*8 + lane/4, k = k4*4 + lane%4)
// ---------------------------------------------------------------------------------
__host__ __device__ __forceinline__ long linvf_total_tiles(int Npad, int BN) {
  int nb = Npad / BN;
  return (long)(BN / 16) * ((long)nb * (nb + 1) / 2);
}

// ---------------------------------------------------------------------------------
// Acquisition utilities on (mu, var): reference approxposterior/utility.py
//   logsubexp :69-89 (naive log(1-exp), kept), AGP :136, BAPE :183, Jones :229-244
// kind: 0 none, 1 AGP, 2 BAPE, 3 Jones
// ---------------------------------------------------------------------------------
__device__ __forceinline__ double logsubexp_ref(double x1, double x2) {
  if (x1 <= x2) return -INFINITY;
  return x1 + log(1.0 - exp(x2 - x1));
}
__device__ __forceinline__ double utility_eval(int kind, double mu, double var, double ybest, double zeta) {
  if (kind == 1) {
    return -(mu + 0.5 * log(2.0 * 3.14159265358979323846 * 2.71828182845904523536 * var));
  } else if (kind == 2) {
    return -((2.0 * mu + var) + logsubexp_ref(var, 0.0));
  } else if (kind == 3) {
    double sd = sqrt(var);
    if (!(sd > 0.0)) return 0.0;
    double imp = mu - ybest - zeta;
    double z = imp / sd;
    double cdf = 0.5 * erfc(-z * 0.70710678118654752440);
    double pdf = exp(-0.5 * z * z) * 0.39894228040143267794;
    return -(imp * cdf + sd * pdf);
  }
  return 0.0;
}

// ---------------------------------------------------------------------------------
// exp(-s) for s >= 0: 2^(n/64) table + degree-5 polynomial, ~1 ulp; 10 FP64 ops instead of libdevice's 16.
__device__ __forceinline__ double exp_neg(double s, const double* __restrict__ tab) {
  const double x = -s;
  const double t = fma(x, 92.33248261689366 /*64/ln2*/, 6755399441055744.0);
  const int n = __double2loint(t);
  const double nf = t - 6755399441055744.0;
  double r = fma(nf, -0.010830424696249145 /*ln2/64 hi*/, x);    // fma: x - nf*hi is a single rounding
  r = fma(nf, -3.623510646634843e-19 /*ln2/64 lo*/, r);
  const double r2 = r * r;
  double q = fma(r, 8.3333333333333332e-03, 4.1666666666666664e-02);
  q = fma(r, q, 1.6666666666666666e-01);
  q = fma(r, q, 0.5);
  const double pm1 = fma(r2, q, r);                         // e^r - 1
  const double T = tab[n & 63];
  double res = fma(T, pm1, T);
  const int k = n >> 6;
  res = __hiloint2double(__double2hiint(res) + (k << 20), __double2loint(res));
  return (s >= 700.0) ? 0.0 : res;                            // exp(-700) ~ 1e-304: flush (keeps 2^k normal); NaN propagates
}

// exp(-s) for s >= 0 with a 256-entry table 2^(j/256) and a degree-4 polynomial: 9 FP64 operations (the 64-entry form
// above needs 10 plus an FP64 compare for the range check, done here on the integer pipe), <= 2 ulp.  Used where the
// exponential IS the work and the kernel is bound by instruction issue next to the FP64 pipe (sampler, mean-only
// predict); |r| <= ln2/512, so the first dropped term r^5/120 is below 4e-17.
// RANGE_CHECK = false (callers whose arguments are finite by construction, i.e. prior-gated sampler proposals): the
// exponent is clamped at 2^-1022 with one integer max instead of the four-instruction range test, so arguments beyond
// ~708 return a positive number below 4.5e-308 instead of an exact 0.
template <bool RANGE_CHECK = true>
__device__ __forceinline__ double exp_neg256(double s, const double* __restrict__ tab) {
  const double x = -s;
  const double t = fma(x, 369.32993046757464 /*256/ln2*/, 6755399441055744.0);
  const int n = __double2loint(t);
  const double nf = t - 6755399441055744.0;
  double r = fma(nf, -0.0027076061740622863 /*ln2/256 hi*/, x);
  r = fma(nf, -9.0587766165871075e-20 /*ln2/256 lo*/, r);
  double q = fma(r, 4.1666666666666664e-02, 1.6666666666666666e-01);
  q = fma(r, q, 0.5);
  const double pm1 = fma(r * r, q, r);                      // e^r - 1
  const double T = tab[n & 255];
  double res = fma(T, pm1, T);
  if (!RANGE_CHECK) return __hiloint2double(__double2hiint(res) + (max(n >> 8, -1022) << 20), __double2loint(res));
  res = __hiloint2double(__double2hiint(res) + ((n >> 8) << 20), __double2loint(res));
  // s in [700, +inf] -> 0 (keeps 2^k normal); NaN has a larger high word and falls through to propagate
  const unsigned hs = (unsigned)__double2hiint(s);
  return (hs - 0x4085E000u <= 0x7FF00000u - 0x4085E000u) ? 0.0 : res;
}

// Philox4x32-10 counter-based RNG (Salmon et al. 2011), for the device sampler.
struct Philox {
  uint32_t k0, k1;
  __device__ __forceinline__ void round(uint32_t* c, uint32_t ka, uint32_t kb) const {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
    uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
    uint32_t n0 = hi1 ^ c[1] ^ ka, n1 = lo1, n2 = hi0 ^ c[3] ^ kb, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
  }
  __device__ __forceinline__ void gen(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out) const {
    uint32_t c[4] = {c0, c1, c2, c3};
    uint32_t ka = k0, kb = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) { round(c, ka, kb); ka += 0x9E3779B9u; kb += 0xBB67AE85u; }
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
  }
};
// uniform in the OPEN interval (0,1) from 52 random bits: (x + 1/2) 2^-52 is exact for x < 2^52, so neither end is
// reachable (with 53 bits the +1/2 is not representable above 2^52 and the largest value rounded to exactly 1.0)
__device__ __forceinline__ double u01_from_bits(uint32_t hi, uint32_t lo) {
  uint64_t x = (((uint64_t)hi << 32) | lo) >> 12;
  return ((double)x + 0.5) * (1.0 / 4503599627370496.0);
}

}  // namespace apgp
