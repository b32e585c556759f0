// Shared helpers for liboffk (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "offk.h"

namespace offk {

// ---- per-thread last-error string (offk_last_error_string) -----------------
extern thread_local char g_err[512];
inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
inline int cuda_check(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return (int)e;
}
#define OFFK_LAUNCH_CHECK(what) ::offk::cuda_check(cudaGetLastError(), what)
#define OFFK_REQUIRE(cond, ...) \
  do {                          \
    if (!(cond)) return ::offk::fail(OFFK_E_BADARG, __VA_ARGS__); \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- counter-hash dropout (OFFK_DROP_SEED) ----------------------------------
// One 64-bit hash (two 32-bit lowbias mixers) serves FOUR consecutive elements (a channel quad of a channels-last
// tensor): keep(idx) = 16-bit field (idx & 3) of hash(seed, idx >> 2) >= p * 2^16.
// Same on host and device so tests can regenerate the mask and the backward kernels never need it in memory.
__host__ __device__ __forceinline__ uint32_t drop_mix32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x21F0AAADu;
  x ^= x >> 15;
  x *= 0x735A2D97u;
  x ^= x >> 15;
  return x;
}
__host__ __device__ __forceinline__ uint64_t drop_hash64(uint64_t seed, uint64_t quad) {
  // fold the whole 64-bit seed into BOTH 32-bit keys (a multiply carries the low seed bits into the high word, the
  // xor-shift brings the high word down): small seeds (1, 2, 3, ...) must change all four keep decisions of a quad
  uint64_t k = (seed + 0x9E3779B97F4A7C15ull) * 0xBF58476D1CE4E5B9ull;
  k ^= k >> 31;
  const uint32_t k0 = (uint32_t)k, k1 = (uint32_t)(k >> 32);
  const uint32_t q = (uint32_t)quad ^ ((uint32_t)(quad >> 32) * 0x9E3779B1u);
  const uint32_t lo = drop_mix32(q * 0x9E3779B1u + k0);
  const uint32_t hi = drop_mix32((q ^ 0x85EBCA77u) * 0xC2B2AE3Du + k1);
  return ((uint64_t)hi << 32) | lo;
}
__host__ __device__ __forceinline__ uint32_t drop_threshold16(float p) {
  float t = p * 65536.0f;
  return t <= 0.f ? 0u : (t >= 65536.0f ? 65536u : (uint32_t)t);
}
// bit i = keep decision of element 4*quad + i
__host__ __device__ __forceinline__ uint32_t drop_keep4(uint64_t seed, uint64_t quad, uint32_t thr16) {
  const uint64_t h = drop_hash64(seed, quad);
  const uint32_t lo = (uint32_t)h, hi = (uint32_t)(h >> 32);
  return ((lo & 0xFFFFu) >= thr16 ? 1u : 0u) | ((lo >> 16) >= thr16 ? 2u : 0u) |
         ((hi & 0xFFFFu) >= thr16 ? 4u : 0u) | ((hi >> 16) >= thr16 ? 8u : 0u);
}
__host__ __device__ __forceinline__ bool drop_keep(uint64_t seed, uint64_t idx, uint32_t thr16) {
  return (drop_keep4(seed, idx >> 2, thr16) >> (idx & 3u)) & 1u;
}

// ---- vector / cache-hinted global access ------------------------------------
__device__ __forceinline__ float4 ldg_stream4(const float* p) {  // read-once data: keep it out of L1
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream4(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}
// fp32 accumulation into global memory WITHOUT a return value: always the fire-and-forget RED instruction.  (atomicAdd
// with an unused result is normally lowered to RED too, but ptxas keeps the round-trip ATOM form once the kernel also
// contains a fence / a value-returning atomic -- measured: the unit weight-gradient GEMMs ran 2x slower.)
__device__ __forceinline__ void red_add_f32(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

int sm_count();  // cached multiprocessor count of the current device

// ---- programmatic dependent launch ---------------------------------------------
// Kernels call pdl_sync() before their first global access: it waits until the previous kernel in the stream has
// completed and its writes are visible, then lets the NEXT kernel be scheduled (whose own pdl_sync() blocks until this
// grid is done).  Launch latency and kernel prologues thereby overlap the predecessor's tail.  Without the launch
// attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_sync() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace offk
