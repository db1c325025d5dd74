// int8 tensor-core rate against the MMA's N on sm_100a: one CTA per SM, one lane issuing a long accumulating stream of
// tcgen05.mma.cta_group::1.kind::i8 (M = 128, K = 32, A and B from shared memory, D in tensor memory) at N = 64, 128,
// 192 and 256.  Reports MAC per clock per SM (SM cycles of the issuing lane, clock64) and TOPS (CUDA events), with the
// card's name, power limit and SM clock read while the probe runs.  Operand bytes read per MAC fall with N:
// A (4 KB) is read once per MMA whatever N is, so a shared-memory-bound stream shows a lower rate at small N.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/i8_mma_probe tools/i8_mma_probe.cu
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>

#define CK(x) do{cudaError_t e=(x); if(e!=cudaSuccess){printf("CUDA error %s at %d\n",cudaGetErrorString(e),__LINE__); exit(1);} }while(0)

constexpr int NTILE = 8;                 // distinct A and B tiles, cycled so successive MMAs read different addresses
constexpr int A_TILE = 128 * 32;         // bytes
constexpr int B_TILE_MAX = 256 * 32;
constexpr int SMEM = NTILE * (A_TILE + B_TILE_MAX) + 16;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// no-swizzle K-major descriptor: LBO = K-direction core-matrix stride, SBO = M/N-direction 8-row-group stride
__device__ __forceinline__ uint64_t desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}

template <int N>
__global__ void __launch_bounds__(128, 1) probe(int iters, long long* cyc) {
  extern __shared__ __align__(128) unsigned char sm[];
  unsigned char* A = sm;
  unsigned char* B = sm + NTILE * A_TILE;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sm + NTILE * (A_TILE + B_TILE_MAX));
  __shared__ uint32_t tmem_s;
  for (int i = threadIdx.x; i < NTILE * (A_TILE + B_TILE_MAX) / 4; i += blockDim.x)
    reinterpret_cast<uint32_t*>(sm)[i] = 0x9E3779B9u * (uint32_t)(i + 1);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" :: "r"(smem_u32(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" :: "r"(smem_u32(&tmem_s)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem = tmem_s;
  if (threadIdx.x == 0) {
    // D s32, A u8, B s8, both K-major, M = 128
    constexpr uint32_t idesc = (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr int NREG = 512 / N < 8 ? 512 / N : 8;    // accumulators rotated like the level sums of predict_i8.cu
    const uint32_t sa = smem_u32(A), sb = smem_u32(B);
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) {
      const int t = i % NTILE, rg = i % NREG;
      const uint64_t da = desc(sa + t * A_TILE, 2048, 128);
      const uint64_t db = desc(sb + t * (N * 32), N * 16, 128);
      const uint32_t acc = i >= NREG;
      asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                   "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n"
                   :: "r"(tmem + rg * (512 / NREG)), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
    }
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" :: "r"(smem_u32(bar)) : "memory");
    asm volatile("{\n\t.reg .pred P1;\n\tW:\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n\t@!P1 bra W;\n\t}\n"
                 :: "r"(smem_u32(bar)) : "memory");
    cyc[blockIdx.x] = clock64() - t0;
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem) : "memory");
  }
}

static void smi(const char* tag) {
  FILE* f = popen("nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.max.sm,power.draw --format=csv,noheader -i 0", "r");
  char buf[512];
  if (f && fgets(buf, sizeof buf, f)) printf("%s nvidia-smi (name, power limit, SM clock, max SM clock, power draw): %s", tag, buf);
  else printf("%s nvidia-smi: not read\n", tag);
  if (f) pclose(f);
}

template <int N>
static void run(int nsm, long long* dcyc, long long* hcyc, cudaEvent_t e0, cudaEvent_t e1) {
  CK(cudaFuncSetAttribute(probe<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
  const long long macs_per_mma = 128LL * N * 32;
  const int iters = (int)((1LL << 36) / macs_per_mma);     // same MAC count per CTA for every N (~8.4 M clk at 8 K MAC/clk)
  probe<N><<<nsm, 128, SMEM>>>(iters / 16, dcyc);          // warm-up
  CK(cudaDeviceSynchronize());
  float best = 1e30f; double cyc_best = 0;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0));
    probe<N><<<nsm, 128, SMEM>>>(iters, dcyc);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    CK(cudaGetLastError());
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaMemcpy(hcyc, dcyc, sizeof(long long) * nsm, cudaMemcpyDeviceToHost));
    double c = 0; for (int i = 0; i < nsm; ++i) c += (double)hcyc[i]; c /= nsm;
    if (ms < best) { best = ms; cyc_best = c; }
  }
  const double macs = (double)iters * macs_per_mma;
  printf("N=%3d  MMAs/CTA %8d  %.3f ms  %.0f MAC/clk/SM  %.1f TOPS  %.1f clk per MMA  (SM clock from cycles/time %.0f MHz)  "
         "smem operand bytes per MAC %.4f\n",
         N, iters, best, macs / cyc_best, 2.0 * macs * nsm / (best * 1e-3) / 1e12, cyc_best / iters,
         cyc_best / (best * 1e-3) / 1e6, (double)(A_TILE + N * 32) / macs_per_mma);
  for (int rep = 0; rep < 100; ++rep) probe<N><<<nsm, 128, SMEM>>>(iters, dcyc);   // keep the card busy while it is read
  smi("  while running:");
  CK(cudaDeviceSynchronize());
}

int main() {
  cudaDeviceProp p; CK(cudaGetDeviceProperties(&p, 0));
  printf("device %s SMs %d\n", p.name, p.multiProcessorCount);
  smi("idle:");
  const int nsm = p.multiProcessorCount;
  long long* dcyc; CK(cudaMalloc(&dcyc, sizeof(long long) * nsm));
  long long* hcyc = (long long*)malloc(sizeof(long long) * nsm);
  cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
  run<64>(nsm, dcyc, hcyc, e0, e1);
  run<128>(nsm, dcyc, hcyc, e0, e1);
  run<192>(nsm, dcyc, hcyc, e0, e1);
  run<256>(nsm, dcyc, hcyc, e0, e1);
  free(hcyc);
  return 0;
}
