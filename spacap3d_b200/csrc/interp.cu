// interp.cu -- three_nn, three_interpolate and its backward (sm_100a).
//
// Replaces three_nn_kernel, three_interpolate_kernel, three_interpolate_grad_kernel (reference
// interpolate_gpu.cu:9-154), each of which runs one block per scene.  These ops are small
// (FP1: 512x256, FP2: 1024x512 per scene) and launch/latency bound, so the design goal is a
// wide grid with on-chip reuse: `known` is staged once per CTA in shared memory for three_nn;
// three_interpolate keeps (idx, weight) of a point in registers and sweeps channels with
// coalesced stores, the small feature rows being served by L1.
// three_interpolate and its backward are instantiated for float and bf16 storage of the features (common.cuh): the
// forward reads bf16 rows and writes bf16, the backward reads a bf16 grad_out and writes an fp32 gradient.  idx and
// weight stay fp32 / int32, and the arithmetic is fp32 either way.
#include "common.cuh"
#include "ptx.cuh"

namespace spc {

constexpr int NN_THREADS = 128;
constexpr int NN_TILE = 1024;  // known points staged per tile (12 KB)

// unknown (B,n,3), known (B,m,3) -> dist2 (B,n,3), idx (B,n,3).
// The reference keeps its running bests in double initialised to 1e40 (interpolate_gpu.cu:27);
// since d is a float promoted for the compare, float bests initialised to +inf order every
// candidate identically (d < 1e40 <=> d < +inf for every float d incl. +inf/NaN), and the
// final (float)1e40 store is +inf as well.
__global__ void __launch_bounds__(NN_THREADS) three_nn_kernel(const float *__restrict__ unknown,
                                                              const float *__restrict__ known,
                                                              int n, int m,
                                                              float *__restrict__ dist2,
                                                              int32_t *__restrict__ idx) {
  __shared__ float sx[NN_TILE], sy[NN_TILE], sz[NN_TILE];
  const int b = blockIdx.y;
  const int j = blockIdx.x * NN_THREADS + threadIdx.x;
  const float *U = unknown + (size_t)b * n * 3;
  const float *K = known + (size_t)b * m * 3;
  const bool ok = j < n;
  const float ux = ok ? __ldg(U + 3 * j + 0) : 0.f, uy = ok ? __ldg(U + 3 * j + 1) : 0.f,
              uz = ok ? __ldg(U + 3 * j + 2) : 0.f;
  float b1 = INFINITY, b2 = INFINITY, b3 = INFINITY;
  int i1 = 0, i2 = 0, i3 = 0;
  for (int base = 0; base < m; base += NN_TILE) {
    const int tile = min(NN_TILE, m - base);
    __syncthreads();
    for (int e = threadIdx.x; e < tile * 3; e += NN_THREADS) {
      const float v = __ldg(K + (size_t)base * 3 + e);
      const int pt = e / 3, comp = e - pt * 3;
      (comp == 0 ? sx : comp == 1 ? sy : sz)[pt] = v;
    }
    __syncthreads();
    for (int k = 0; k < tile; ++k) {
      const float d = sqdist_ref(ux, uy, uz, sx[k], sy[k], sz[k]);   // smem broadcast reads
      if (d < b1) { b3 = b2; i3 = i2; b2 = b1; i2 = i1; b1 = d; i1 = base + k; }
      else if (d < b2) { b3 = b2; i3 = i2; b2 = d; i2 = base + k; }
      else if (d < b3) { b3 = d; i3 = base + k; }
    }
  }
  if (ok) {
    float *od = dist2 + ((size_t)b * n + j) * 3;
    int32_t *oi = idx + ((size_t)b * n + j) * 3;
    od[0] = b1; od[1] = b2; od[2] = b3;
    oi[0] = i1; oi[1] = i2; oi[2] = i3;
  }
}

// ------------------------------------------------------------------------------------------------
// three_interpolate / three_interpolate_grad
//
// Both are streams of a (B,C,*) tensor with a 3-entry gather / scatter per point, i.e. HBM-bound once the clouds
// are large (config 5: n = 4096, m = 2048 per scene) and launch-bound at the detector's own sizes.
//  * forward: a CTA stages CT whole rows of `points` (contiguous in (B,C,m)) in shared memory with ONE bulk-TMA
//    copy, keeps (idx, weight) of FOUR consecutive output positions per thread in registers (three 16-byte loads
//    each) and writes 16-byte streaming stores; the reference's contraction order fma(p3,w3, fma(p1,w1, p2*w2)) is
//    kept, so the result stays bit-equal to the golden vectors.
//  * backward: a CTA owns TI_CT whole rows of grad_points in shared memory, sweeps all n positions and flushes the
//    rows once -- no global atomics, no pre-zeroing.  Measured and NOT kept (round 2): inverting the relation into
//    per-known-point lists (atomic-free, bit-reproducible) -- list build 39 us + gather kernel 105 us at config 5's
//    x4 shape against 96 us for this kernel, and 29 vs 16 us at FP1's; and warp-owned channels with
//    __match_any pre-combining and plain load-add-store (no atomics at all): 42 / 75 / 265 us against 16 / 28 / 96 --
//    one dependent shared-memory round trip per update and warp is slower than 256 independent CAS chains.
// ------------------------------------------------------------------------------------------------
constexpr int TI_THREADS = 256;

// one bulk-TMA copy global -> shared (bytes % 16 == 0, 16-byte aligned) or a plain copy; all threads call it
template <class T>
__device__ __forceinline__ void ti_stage(T *dst, const T *src, size_t count, uint64_t *bar, int tid, int nthr) {
  const size_t bytes = count * sizeof(T);
  if (((reinterpret_cast<uintptr_t>(src) & 15) == 0) && bytes % 16 == 0 && bytes < (1u << 20)) {
    if (tid == 0) {
      mbarrier_init(bar, 1);
      fence_mbarrier_init();
    }
    __syncthreads();
    if (tid == 0) {
      mbarrier_arrive_expect_tx(bar, (unsigned)bytes);
      bulk_g2s(dst, src, (unsigned)bytes, bar);
    }
    mbarrier_wait(bar, 0);
  } else {
    for (size_t e = tid; e < count; e += nthr) dst[e] = __ldg(src + e);
    __syncthreads();
  }
}

// points (B,C,m), idx/weight (B,n,3) -> out (B,C,n).   grid = (ceil(n/1024), ceil(C/CT), B)
template <class T, bool STAGED>
__global__ void __launch_bounds__(TI_THREADS) three_interpolate_kernel(
    const T *__restrict__ points, const int32_t *__restrict__ idx,
    const float *__restrict__ weight, int C, int m, int n, int CT, T *__restrict__ out) {
  extern __shared__ __align__(128) float s_smem[];
  T *s_rows = reinterpret_cast<T *>(s_smem);        // [CT][m]
  __shared__ __align__(8) uint64_t bar;
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * CT;
  const int ct = min(CT, C - c0);
  const T *src = points + ((size_t)b * C + c0) * m;
  if (STAGED) ti_stage(s_rows, src, (size_t)ct * m, &bar, threadIdx.x, TI_THREADS);
  const int j0 = (blockIdx.x * TI_THREADS + threadIdx.x) * 4;
  if (j0 >= n) return;
  const int32_t *ix = idx + ((size_t)b * n + j0) * 3;
  const float *w = weight + ((size_t)b * n + j0) * 3;
  int a[12];
  float ww[12];
  if (j0 + 4 <= n && (((size_t)b * n + j0) * 3) % 4 == 0) {       // 48 contiguous bytes each: three 16-byte loads
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const int4 i4 = __ldg(reinterpret_cast<const int4 *>(ix) + q);
      const float4 w4 = __ldg(reinterpret_cast<const float4 *>(w) + q);
      a[4 * q + 0] = i4.x; a[4 * q + 1] = i4.y; a[4 * q + 2] = i4.z; a[4 * q + 3] = i4.w;
      ww[4 * q + 0] = w4.x; ww[4 * q + 1] = w4.y; ww[4 * q + 2] = w4.z; ww[4 * q + 3] = w4.w;
    }
  } else {
#pragma unroll
    for (int e = 0; e < 12; ++e) {
      const bool ok = j0 + e / 3 < n;
      a[e] = ok ? __ldg(ix + e) : 0;
      ww[e] = ok ? __ldg(w + e) : 0.f;
    }
  }
  const bool vec = j0 + 4 <= n && n % 4 == 0;
  for (int c = 0; c < ct; ++c) {
    const T *row = STAGED ? s_rows + (size_t)c * m : src + (size_t)c * m;
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float p1 = to_f32(STAGED ? row[a[3 * q]] : __ldg(row + a[3 * q]));
      const float p2 = to_f32(STAGED ? row[a[3 * q + 1]] : __ldg(row + a[3 * q + 1]));
      const float p3 = to_f32(STAGED ? row[a[3 * q + 2]] : __ldg(row + a[3 * q + 2]));
      v[q] = __fmaf_rn(p3, ww[3 * q + 2], __fmaf_rn(p1, ww[3 * q], __fmul_rn(p2, ww[3 * q + 1])));
    }
    T *o = out + ((size_t)b * C + c0 + c) * n + j0;
    if (vec) st_cs4(o, from_f32<T>(v[0]), from_f32<T>(v[1]), from_f32<T>(v[2]), from_f32<T>(v[3]));
    else
#pragma unroll
      for (int q = 0; q < 4; ++q) if (j0 + q < n) o[q] = from_f32<T>(v[q]);
  }
}

// grad_out (B,C,n) -> grad_points (B,C,m): a CTA owns TI_CT whole output rows (all n positions), accumulates them
// in shared memory and stores them once.
constexpr int TI_CT = 8;
template <class T>
__global__ void __launch_bounds__(TI_THREADS) three_interpolate_grad_kernel(
    const T *__restrict__ grad_out, const int32_t *__restrict__ idx,
    const float *__restrict__ weight, int C, int n, int m, float *__restrict__ grad_points) {
  extern __shared__ float s_acc[];  // [TI_CT][m]
  const int b = blockIdx.y;
  const int c0 = blockIdx.x * TI_CT;
  const int ct = min(TI_CT, C - c0);
  for (int e = threadIdx.x; e < ct * m; e += TI_THREADS) s_acc[e] = 0.f;
  __syncthreads();
  for (int j = threadIdx.x; j < n; j += TI_THREADS) {
    const int32_t *ix = idx + ((size_t)b * n + j) * 3;
    const float *w = weight + ((size_t)b * n + j) * 3;
    const int a1 = __ldg(ix), a2 = __ldg(ix + 1), a3 = __ldg(ix + 2);
    const float w1 = __ldg(w), w2 = __ldg(w + 1), w3 = __ldg(w + 2);
    for (int c = 0; c < ct; ++c) {
      const float g = to_f32(__ldg(grad_out + ((size_t)b * C + c0 + c) * n + j));
      float *row = s_acc + (size_t)c * m;
      atomicAdd(row + a1, g * w1);
      atomicAdd(row + a2, g * w2);
      atomicAdd(row + a3, g * w3);
    }
  }
  __syncthreads();
  float *dst = grad_points + ((size_t)b * C + c0) * m;
  for (int e = threadIdx.x; e < ct * m; e += TI_THREADS) dst[e] = s_acc[e];
}

// fallback for rows that do not fit in shared memory: global atomics into a zeroed buffer
template <class T>
__global__ void three_interpolate_grad_global_kernel(const T *__restrict__ grad_out,
                                                     const int32_t *__restrict__ idx,
                                                     const float *__restrict__ weight, int C,
                                                     int n, int m,
                                                     float *__restrict__ grad_points) {
  const int b = blockIdx.z;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int32_t *ix = idx + ((size_t)b * n + j) * 3;
  const float *w = weight + ((size_t)b * n + j) * 3;
  const int a1 = __ldg(ix), a2 = __ldg(ix + 1), a3 = __ldg(ix + 2);
  const float w1 = __ldg(w), w2 = __ldg(w + 1), w3 = __ldg(w + 2);
  for (int c = blockIdx.y; c < C; c += gridDim.y) {
    const float g = to_f32(__ldg(grad_out + ((size_t)b * C + c) * n + j));
    float *row = grad_points + ((size_t)b * C + c) * m;
    atomicAdd(row + a1, g * w1);
    atomicAdd(row + a2, g * w2);
    atomicAdd(row + a3, g * w3);
  }
}

}  // namespace spc

using namespace spc;

extern "C" int spc_three_nn(const float *unknown, const float *known, int B, int n, int m,
                            float *dist2, int32_t *idx, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && n >= 0 && m >= 0, "three_nn: bad sizes");
  if (B == 0 || n == 0) return SPC_OK;
  SPC_CHECK_ARG(unknown && dist2 && idx && (known || m == 0), "three_nn: null pointer");
  SPC_CHECK_ARG(B <= 65535, "three_nn: B too large");
  dim3 grid(ceil_div(n, NN_THREADS), B);
  three_nn_kernel<<<grid, NN_THREADS, 0, (cudaStream_t)stream_>>>(unknown, known, n, m, dist2, idx);
  SPC_LAUNCH_CHECK("three_nn_kernel");
  return SPC_OK;
}

template <class T>
static int three_interpolate(const T *points, const int32_t *idx, const float *weight, int B, int C, int m, int n,
                             T *out, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && m >= 0 && n >= 0, "three_interpolate: bad sizes");
  if (B == 0 || C == 0 || n == 0) return SPC_OK;
  SPC_CHECK_ARG(points && idx && weight && out, "three_interpolate: null pointer");
  SPC_CHECK_ARG(B <= 65535, "three_interpolate: B too large");
  cudaStream_t stream = (cudaStream_t)stream_;
  // rows staged per CTA: as many fp32 rows as fit in ~64 KB (re-reading idx / weight once per channel tile costs
  // 24 B per point and tile against 4*CT B of output), but enough CTAs to fill the machine; bf16 rows take the same
  // tiling in half the shared memory
  int CT = m > 0 ? (int)((64 * 1024) / ((size_t)m * sizeof(float))) : 0;
  if (CT > 32) CT = 32;
  if (CT > C) CT = C;
  const int xchunks = ceil_div(n, TI_THREADS * 4);
  while (CT > 4 && (long long)xchunks * ceil_div(C, CT) * B < 2 * kNumSMs) CT /= 2;
  if (CT >= 1) {
    SPC_CHECK_ARG(ceil_div(C, CT) <= 65535, "three_interpolate: C too large");
    const size_t smem = (size_t)CT * m * sizeof(T);
    SPC_CUDA(cudaFuncSetAttribute(three_interpolate_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(xchunks, ceil_div(C, CT), B);
    three_interpolate_kernel<T, true><<<grid, TI_THREADS, smem, stream>>>(points, idx, weight, C, m, n, CT, out);
  } else {                                         // a single row exceeds the budget: read-only-cache gathers
    CT = 8;
    SPC_CHECK_ARG(ceil_div(C, CT) <= 65535, "three_interpolate: C too large");
    dim3 grid(xchunks, ceil_div(C, CT), B);
    three_interpolate_kernel<T, false><<<grid, TI_THREADS, 0, stream>>>(points, idx, weight, C, m, n, CT, out);
  }
  SPC_LAUNCH_CHECK("three_interpolate_kernel");
  return SPC_OK;
}

// the accumulators are fp32 rows for either storage type of grad_out
template <class T>
static int three_interpolate_grad(const T *grad_out, const int32_t *idx, const float *weight, int B, int C, int n,
                                  int m, float *grad_points, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && m >= 0 && n >= 0, "three_interpolate_grad: bad sizes");
  if (B == 0 || C == 0 || m == 0) return SPC_OK;
  SPC_CHECK_ARG(grad_points && (n == 0 || (grad_out && idx && weight)), "three_interpolate_grad: null pointer");
  SPC_CHECK_ARG(B <= 65535, "three_interpolate_grad: B too large");
  cudaStream_t stream = (cudaStream_t)stream_;
  const size_t smem = (size_t)TI_CT * m * sizeof(float);
  if (smem <= 96 * 1024) {
    if (smem > 40 * 1024)
      SPC_CUDA(cudaFuncSetAttribute(three_interpolate_grad_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    three_interpolate_grad_kernel<<<dim3(ceil_div(C, TI_CT), B), TI_THREADS, smem, stream>>>(grad_out, idx, weight, C, n, m,
                                                                                         grad_points);
    SPC_LAUNCH_CHECK("three_interpolate_grad_kernel");
    return SPC_OK;
  }
  SPC_CUDA(cudaMemsetAsync(grad_points, 0, (size_t)B * C * m * sizeof(float), stream));
  if (n == 0) return SPC_OK;
  dim3 grid(ceil_div(n, 256), min(C, 64), B);
  three_interpolate_grad_global_kernel<<<grid, 256, 0, stream>>>(grad_out, idx, weight, C, n, m, grad_points);
  SPC_LAUNCH_CHECK("three_interpolate_grad_global_kernel");
  return SPC_OK;
}

// ---- C entry points: fp32 storage, and bf16 storage (points / out / grad_out are __nv_bfloat16 tensors) ------------
extern "C" int spc_three_interpolate(const float *points, const int32_t *idx, const float *weight,
                                     int B, int C, int m, int n, float *out, void *stream) {
  return three_interpolate(points, idx, weight, B, C, m, n, out, stream);
}
extern "C" int spc_three_interpolate_bf16(const void *points, const int32_t *idx, const float *weight,
                                          int B, int C, int m, int n, void *out, void *stream) {
  return three_interpolate(static_cast<const bf16 *>(points), idx, weight, B, C, m, n, static_cast<bf16 *>(out),
                           stream);
}

extern "C" int spc_three_interpolate_grad(const float *grad_out, const int32_t *idx,
                                          const float *weight, int B, int C, int n, int m,
                                          float *grad_points, void *stream) {
  return three_interpolate_grad(grad_out, idx, weight, B, C, n, m, grad_points, stream);
}
extern "C" int spc_three_interpolate_grad_bf16(const void *grad_out, const int32_t *idx,
                                               const float *weight, int B, int C, int n, int m,
                                               float *grad_points, void *stream) {
  return three_interpolate_grad(static_cast<const bf16 *>(grad_out), idx, weight, B, C, n, m, grad_points, stream);
}
