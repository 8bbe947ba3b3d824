// Shared helpers for libmrfp_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stddef.h>
#include <stdlib.h>
#include <utility>
#include <atomic>
#include "../../include/mrfp_b200.h"

#define MRFP_CUDA_TRY(expr)                          \
  do {                                               \
    cudaError_t _e = (expr);                         \
    if (_e != cudaSuccess) return (int)_e;           \
  } while (0)

namespace mrfp {

struct DeviceInfo {
  int device;
  int sm_count;
  int max_smem_optin;
};
// cached per device; thread-safe (function-local statics + idempotent fill)
int get_device_info(DeviceInfo* out);

__host__ __device__ inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Programmatic dependent launch: every kernel of the HRFP chain is launched with the stream-serialisation attribute and
// starts with pdl_sync().  The trigger lets the NEXT kernel be scheduled (block launch, barrier / TMEM set-up,
// descriptor fetch) while this one is still running; the wait returns only when all prerequisite grids have
// completed and flushed, so every global access behind it sees the same ordering as a plain stream launch.  The trigger
// is ptx::pdl_trigger() (ptx.cuh).
__device__ __forceinline__ void pdl_sync() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device): `flag` is a static of the call site
#define MRFP_SMEM_OPT_IN(kern, bytes, device)                                                              \
  do {                                                                                                     \
    static std::atomic<unsigned long long> _done{0};                                                       \
    const unsigned long long _bit = 1ull << ((device) & 63);                                               \
    if (!(_done.load(std::memory_order_acquire) & _bit)) {                                                 \
      MRFP_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
      _done.fetch_or(_bit, std::memory_order_release);                                                     \
    }                                                                                                      \
  } while (0)

template <typename... Exp, typename... Act>
inline cudaError_t launch_k(void (*kern)(Exp...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Act&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Act>(args)...);
}

__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f4(float4* p, const float4& v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float ld_stream_f1(const float* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f1(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// BatchNorm + ReLU of two bf16 values in one register: one packed fp32 FMA, one rounding to bf16x2, ReLU on the pair.
// max(round(x), 0) == round(max(x, 0)): the same results as fmaxf(fmaf(s, x, b), 0) rounded afterwards, in 5 instructions
// (shift, mask, FFMA2, F2FP, HMNMX2) instead of 7.
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint32_t bn_relu_x2(uint32_t v, uint64_t scale2, uint64_t shift2) {
  uint64_t x, y;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "r"(v << 16), "r"(v & 0xffff0000u));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(y) : "l"(x), "l"(scale2), "l"(shift2));
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(y));
  uint32_t p;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(p) : "f"(hi), "f"(lo));
  asm("max.bf16x2 %0, %1, %2;" : "=r"(p) : "r"(p), "r"(0u));
  return p;
}

// 8 consecutive bf16 values in a uint4 (value 2i in the low half of word i) <-> 8 floats; packing rounds to nearest even
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace mrfp
