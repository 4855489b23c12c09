// f16_kernels_common.cuh -- pieces shared by the kernel translation units (f16_kernels.cu, f16_step_fast.cu):
// TMA table staging, per-aircraft model selection, the trim start point and the persistent-launch helper.
#pragma once
#include <stdint.h>

#include "f16_kernels.cuh"

namespace f16 {

extern __shared__ __align__(128) unsigned char f16_smem[];

// ------------------------------------------------------------------------------------------------------
// table staging: global -> shared with TMA bulk copies completing on one mbarrier
// ------------------------------------------------------------------------------------------------------
static __device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int BYTES>
__device__ __forceinline__ void stage_tables_tma(void* dst, const void* src, unsigned long long* bar) {
  static_assert(BYTES % 16 == 0, "bulk copies move multiples of 16 bytes");
  const uint32_t bar_a = smem_u32(bar);
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(BYTES) : "memory");
    constexpr int CHUNK = 32768;
#pragma unroll 1
    for (int off = 0; off < BYTES; off += CHUNK) {
      const int n = (BYTES - off) < CHUNK ? (BYTES - off) : CHUNK;
      asm volatile(
          "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
              smem_u32(static_cast<char*>(dst) + off)),
          "l"(static_cast<const char*>(src) + off), "r"(n), "r"(bar_a)
          : "memory");
    }
  }
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar_a), "r"(0)
        : "memory");
  }
}

// which aircraft does the FI instantiation own?  (per-aircraft flags other than 0/1 are reported by FI == 1)
template <int FI>
__device__ __forceinline__ int owns(const BatchSel& s, long long n) {
  const int f = s.fi ? (int)s.fi[n] : s.fi_default;
  if (f == FI) return 1;
  if (FI == 1 && f != 0) return -1;
  return 0;
}

// does a batch hold aircraft of fidelity FI?  (per-aircraft flags: the launch for each fidelity picks its own)
static bool wants(const BatchSel& s, int FI) { return s.fi != nullptr || s.fi_default == FI || (FI == 1 && s.fi_default != 0); }

// start point of the trim search, and whether it may leave at a bitwise fixed point (trim kernels of both builds)
struct TrimGuess {
  double ux[5];
  int fixed_point_exit;
};

__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000LL); }

static int grid_for(long long work_items, int per_block, int resident) {
  long long b = (work_items + per_block - 1) / per_block;
  if (b < 1) b = 1;
  if (b > resident) b = resident;
  return (int)b;
}

template <typename Kern>
static cudaError_t prepare(Kern kern, int threads, int smem, int sm_count, int* resident) {
  cudaError_t e = cudaSuccess;
  if (smem > 48 * 1024) {
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
  }
  int per_sm = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorLaunchOutOfResources;
  *resident = per_sm * sm_count;
  return cudaSuccess;
}

// persistent launch: grid = min(ceil(items / per_block), resident CTAs)
template <typename Kern, typename... Args>
static cudaError_t launch_persistent(const LaunchCfg& cfg, Kern kern, int threads, int smem, long long items,
                                     int per_block, Args... args) {
  int resident = 0;
  cudaError_t e = prepare(kern, threads, smem, cfg.sm_count, &resident);
  if (e != cudaSuccess) return e;
  kern<<<grid_for(items, per_block, resident), threads, smem, cfg.stream>>>(args...);
  if (cfg.launch_counter) ++*cfg.launch_counter;
  return cudaGetLastError();
}

}  // namespace f16
