// common.cuh — error plumbing, options and small device helpers shared by the
// kernels of libcozo_gpu.so (sm_100a only).
#pragma once
// Two test-only build modes exist besides nvcc (tests/emu is test infrastructure; the product is always
// built by nvcc): COZO_CPU_EMU = a harness compiles device headers only; COZO_CPU_EMU_LIB = the whole library is
// compiled against a fake CUDA runtime (tests/emu/fake_cuda/cuda_runtime.h, which defines COZO_CPU_EMU itself).
#if defined(COZO_CPU_EMU) && !defined(COZO_CPU_EMU_LIB)
#include <stdint.h>

#include "../../include/cozo_gpu.h"
namespace cozo {
constexpr uint32_t NONE = 0xFFFFFFFFu;
inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }
#else
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>
#include <string>

#include "../../include/cozo_gpu.h"

namespace cozo {

// thread-local last error (cozo_gpu_last_error)
std::string& last_error();
int set_error(int code, const char* fmt, ...);
int64_t get_option(const char* name, int64_t dflt);

#define COZO_CUDA(call)                                                                              \
  do {                                                                                               \
    cudaError_t _e = (call);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return ::cozo::set_error(_e == cudaErrorMemoryAllocation ? COZO_GPU_ENOMEM : COZO_GPU_ECUDA,    \
                               "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct DeviceInfo {
  int device = -1;
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  size_t smem_optin = 0;
  bool ok = false;
};
const DeviceInfo& device_info();
int ensure_init();

constexpr uint32_t NONE = 0xFFFFFFFFu;

__host__ __device__ inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }

#endif

// ---- device helpers ----------------------------------------------------------
#if defined(COZO_CPU_EMU)
// CPU SIMT emulation: mbarrier / bulk copy come from cuda_emu.hpp, the rest are plain loads
inline float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
inline float4 ldg_nc_f4(const float4* p) { return *p; }
inline void prefetch_l2(const void*) {}
#elif defined(__CUDACC__)
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// mbarrier + 1-D bulk async copy (TMA engine, no tensor map): PTX ISA
// cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();  // never hang the GPU on a protocol bug
  }
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ float4 ldg_nc_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
#endif

// Key order of every sorted distance list (search beams, per-shard top-k lists), the reference's OrderedFloat:
// NaN sorts after every number, +inf included, and equal keys keep arrival order.  A raw `<=` is false for NaN, so
// a NaN key (0/0 of a zero-norm Cosine row) would go first and break the sorted prefix behind it.
template <typename T>
__device__ __forceinline__ bool precedes(T a, T b) {
  return a < b || (isnan(b) && !isnan(a));
}

}  // namespace cozo
