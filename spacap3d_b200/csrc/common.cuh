// common.cuh -- shared helpers for libspacap3d_ops.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/spacap3d_ops.h"

#ifndef __CUDA_ARCH_LIST__
#define __CUDA_ARCH_LIST__ 1000
#endif

namespace spc {

constexpr int kNumSMs = 148;  // B200

// thread-local error text (spc_last_error)
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);

#define SPC_CHECK_ARG(cond, ...)        \
  do {                                  \
    if (!(cond)) {                      \
      spc::set_error(__VA_ARGS__);      \
      return SPC_ERR_INVALID_ARG;       \
    }                                   \
  } while (0)

#define SPC_CUDA(expr)                                   \
  do {                                                   \
    cudaError_t _e = (expr);                             \
    if (_e != cudaSuccess) return spc::cuda_fail(_e, #expr); \
  } while (0)

#define SPC_LAUNCH_CHECK(name)                                      \
  do {                                                              \
    cudaError_t _e = cudaGetLastError();                            \
    if (_e != cudaSuccess) return spc::cuda_fail(_e, name);         \
  } while (0)

// Squared distance in the reference's exact rounding order (SURVEY F3; SASS of
// ball_query_gpu.cu:31-32 / sampling_gpu.cu:103-104 / interpolate_gpu.cu:33):
//   t = dy*dy (FMUL);  t = fma(dx,dx,t);  d = fma(dz,dz,t)
// Intrinsics pin the contraction so a compiler change cannot re-associate it.
__device__ __forceinline__ float sqdist_ref(float ax, float ay, float az, float bx, float by,
                                            float bz) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- storage types of the training-path kernels -----------------------------------------------------------------
// The large operands of grouping, interpolation and BatchNorm + ReLU are stored as float or as bf16 (torch.autocast
// with dtype=torch.bfloat16); arithmetic is fp32 either way and every stored value is rounded once (to nearest even).
// For T = float every helper below is the plain fp32 load / store, so the fp32 instantiations are the same code.
using bf16 = __nv_bfloat16;

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(bf16 v) { return __bfloat162float(v); }

template <class T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

// v as it reads back after a store to T: itself for float, rounded to bf16 for bf16
template <class T> __device__ __forceinline__ float stored(float v) { return to_f32(from_f32<T>(v)); }

__device__ __forceinline__ unsigned bf16_pair_bits(bf16 lo, bf16 hi) {
  return (unsigned)__bfloat16_as_ushort(lo) | ((unsigned)__bfloat16_as_ushort(hi) << 16);
}

// four consecutive elements, 4 * sizeof(T)-byte aligned, through the read-only path
__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }
__device__ __forceinline__ float4 ldg4(const bf16 *p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                     __uint_as_float(u.y & 0xffff0000u));
}

// four consecutive elements, 4 * sizeof(T)-byte aligned
__device__ __forceinline__ void st4(float *p, float4 v) { *reinterpret_cast<float4 *>(p) = v; }
__device__ __forceinline__ void st4(bf16 *p, float4 v) {
  *reinterpret_cast<uint2 *>(p) = make_uint2(bf16_pair_bits(__float2bfloat16_rn(v.x), __float2bfloat16_rn(v.y)),
                                             bf16_pair_bits(__float2bfloat16_rn(v.z), __float2bfloat16_rn(v.w)));
}

// the same with a streaming (evict-first) store, for outputs that are not read again soon
__device__ __forceinline__ void st_cs4(float *p, float a, float b, float c, float d) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void st_cs4(bf16 *p, bf16 a, bf16 b, bf16 c, bf16 d) {
  asm volatile("st.global.cs.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(bf16_pair_bits(a, b)), "r"(bf16_pair_bits(c, d))
               : "memory");
}

// opt_n_threads of the reference (include/cuda_utils.h:15-19): largest power of two <= n,
// capped at 512 -- it defines the FPS tie-break order, so it is part of the numerical contract.
static inline int ref_opt_n_threads(int work_size) {
  int t = 1;
  while (t * 2 <= work_size && t * 2 <= 512) t *= 2;
  return t;
}

}  // namespace spc
