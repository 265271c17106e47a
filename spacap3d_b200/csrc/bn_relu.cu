// bn_relu.cu -- training-mode BatchNorm + ReLU over (B, C, S) fp32 or bf16 activations, forward and backward (sm_100a).
//
// Replaces, for the shared-MLP blocks in TRAINING mode, the reference's
//     nn.BatchNorm2d (pytorch_utils.py:39-64, cuDNN bn_fw_tr / bn_bw kernels) followed by nn.ReLU(inplace=True)
//     (pytorch_utils.py:11-36) on the (B, C, npoint, nsample) tensors produced by the 1x1 convolutions.
// Profiled on B200 (batch 4 x 40k points, forward+backward): cuDNN's bn_bw_1C11_kernel_new is 30 % of the
// step and bn_fw_tr 11 %, both at < 20 % of HBM bandwidth; together with the separate ReLU forward and
// backward passes the block makes ~14 full passes over tensors of up to 134 MB.  Here:
//   forward : one statistics pass (read y) + one normalise+ReLU pass (read y, write z)
//   backward: one reduction pass (read dz, y; the ReLU mask is recomputed from y) + one apply pass
//             (read dz, y; write dy)
// All four are streaming kernels: float4 loads with UNR independent loads in flight per thread, grids sized in
// multiples of the SM count, fp32 per-thread partial sums of SHIFTED data (x - K, K = first element of the
// channel: no cancellation), per-CTA and cross-CTA combination in fp64.
// Semantics = torch.nn.functional.batch_norm(training=True) + relu: biased variance for normalisation,
// running_mean/var updated with `momentum` and the unbiased variance, save_mean / save_invstd for backward,
// gradient of ReLU taken where the OUTPUT is > 0.
// Every kernel is instantiated for float and bf16 storage of y, z, dz, dy, dpool, pooled and ymax (common.cuh):
// arithmetic, partial sums and per-channel tensors stay fp32 / fp64, and a bf16 pass compares and masks the
// bf16-ROUNDED relu(bn(y)), as torch's own bf16 sequence (batch_norm -> relu -> max_pool2d) sees it.
#include <initializer_list>
#include <type_traits>

#include "common.cuh"

namespace spc {

constexpr int BN_THREADS = 256;
constexpr int BN_MAX_SPLITS = 64;
constexpr int BN_UNR = 4;
constexpr int BN_SYNC_K = 3;      // fp64 values per channel in a rank's synced-BatchNorm row (see below)

__device__ __forceinline__ double block_sum_double(double v, double *s_red) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  double t = 0.0;
  if (warp == 0) {
    t = lane < BN_THREADS / 32 ? s_red[lane] : 0.0;
#pragma unroll
    for (int o = 4; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  return t;   // valid in thread 0
}

// grid (splits, C): CTA (s, c) reduces positions [p0, p1) of every batch row of channel c.
// MODE 0: sums of (x-K), (x-K)^2.   MODE 1 (backward): sums of dzm, dzm * xhat.
template <class T, int MODE, bool VEC>
__global__ void __launch_bounds__(BN_THREADS) bn_reduce_kernel(const T *__restrict__ y, const T *__restrict__ dz,
                                                                const float *__restrict__ gamma,
                                                                const float *__restrict__ beta,
                                                                const float *__restrict__ mean,
                                                                const float *__restrict__ invstd, int B, int C, int S,
                                                                int chunk, double *__restrict__ partial) {
  __shared__ double s_red[BN_THREADS / 32];
  const int c = blockIdx.y, s = blockIdx.x, splits = gridDim.x;
  const int p0 = s * chunk, p1 = min(S, p0 + chunk);
  float a0 = 0.f, a1 = 0.f;
  float K = 0.f, mu = 0.f, is = 0.f, g = 0.f, bt = 0.f;
  if (MODE == 0) K = to_f32(__ldg(y + (size_t)c * S));
  else { mu = __ldg(mean + c); is = __ldg(invstd + c); g = __ldg(gamma + c); bt = __ldg(beta + c); }
  auto acc = [&](float yv, float dv) {
    if (MODE == 0) {
      const float d = yv - K;
      a0 += d;
      a1 = fmaf(d, d, a1);
    } else {
      const float xh = (yv - mu) * is;
      const float z = fmaf(xh, g, bt);
      const float dm = stored<T>(z) > 0.f ? dv : 0.f;
      a0 += dm;
      a1 = fmaf(dm, xh, a1);
    }
  };
  for (int b = 0; b < B; ++b) {
    const T *row = y + ((size_t)b * C + c) * S;
    const T *drow = MODE == 1 ? dz + ((size_t)b * C + c) * S : nullptr;
    if (VEC) {
      int p = p0 + threadIdx.x * 4;
      for (; p + (BN_UNR - 1) * BN_THREADS * 4 < p1; p += BN_UNR * BN_THREADS * 4) {
        float4 v[BN_UNR], d[BN_UNR];
#pragma unroll
        for (int u = 0; u < BN_UNR; ++u) {
          v[u] = ldg4(row + p + u * BN_THREADS * 4);
          if (MODE == 1) d[u] = ldg4(drow + p + u * BN_THREADS * 4);
        }
#pragma unroll
        for (int u = 0; u < BN_UNR; ++u) {
          acc(v[u].x, MODE == 1 ? d[u].x : 0.f); acc(v[u].y, MODE == 1 ? d[u].y : 0.f);
          acc(v[u].z, MODE == 1 ? d[u].z : 0.f); acc(v[u].w, MODE == 1 ? d[u].w : 0.f);
        }
      }
      for (; p < p1; p += BN_THREADS * 4) {
        const float4 v = ldg4(row + p);
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
        if (MODE == 1) d = ldg4(drow + p);
        acc(v.x, d.x); acc(v.y, d.y); acc(v.z, d.z); acc(v.w, d.w);
      }
    } else {
      for (int p = p0 + threadIdx.x; p < p1; p += BN_THREADS)
        acc(to_f32(__ldg(row + p)), MODE == 1 ? to_f32(__ldg(drow + p)) : 0.f);
    }
  }
  const double t0 = block_sum_double((double)a0, s_red);
  const double t1 = block_sum_double((double)a1, s_red);
  if (threadIdx.x == 0) {
    partial[((size_t)c * splits + s) * 2 + 0] = t0;
    partial[((size_t)c * splits + s) * 2 + 1] = t1;
  }
}

// channel c's two sums over the splits of bn_reduce_kernel, in split order
__device__ __forceinline__ void sum_partials(const double *__restrict__ partial, int c, int splits, double &s1,
                                             double &s2) {
  s1 = 0.0;
  s2 = 0.0;
  for (int s = 0; s < splits; ++s) { s1 += partial[((size_t)c * splits + s) * 2]; s2 += partial[((size_t)c * splits + s) * 2 + 1]; }
}

template <class T>
__global__ void bn_finalize_forward_kernel(const T *__restrict__ y, const double *__restrict__ partial, int C, int S,
                                           int splits, double M, float eps, float momentum,
                                           float *__restrict__ running_mean, float *__restrict__ running_var,
                                           float *__restrict__ save_mean, float *__restrict__ save_invstd) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1, s2;
  sum_partials(partial, c, splits, s1, s2);
  const double K = (double)to_f32(__ldg(y + (size_t)c * S));
  const double m1 = s1 / M;
  const double mean = K + m1;
  double var = s2 / M - m1 * m1;
  if (var < 0.0) var = 0.0;
  save_mean[c] = (float)mean;
  save_invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
  if (running_var) {
    const double unbiased = M > 1.0 ? var * M / (M - 1.0) : var;
    running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
  }
}

// dgamma / dbeta; ROW (synced backward) also writes this rank's row (n, sum dm, sum dm * xhat) with n = M
template <bool ROW>
__global__ void bn_finalize_backward_kernel(const double *__restrict__ partial, int C, int splits,
                                            float *__restrict__ dgamma, float *__restrict__ dbeta, double M,
                                            double *__restrict__ row) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1, s2;
  sum_partials(partial, c, splits, s1, s2);
  dbeta[c] = (float)s1;
  dgamma[c] = (float)s2;
  if (ROW) {
    row[(size_t)c * BN_SYNC_K + 0] = M;
    row[(size_t)c * BN_SYNC_K + 1] = s1;
    row[(size_t)c * BN_SYNC_K + 2] = s2;
  }
}

// grid (position tiles, B*C).  MODE 0: z = relu(bn(y)).  MODE 1: dy from dz, y and the channel sums.
template <class T, int MODE, bool VEC>
__global__ void __launch_bounds__(BN_THREADS) bn_apply_kernel(const T *__restrict__ y, const T *__restrict__ dz,
                                                               const float *__restrict__ gamma, const float *__restrict__ beta,
                                                               const float *__restrict__ mean, const float *__restrict__ invstd,
                                                               const float *__restrict__ dgamma, const float *__restrict__ dbeta,
                                                               int C, int S, float inv_M, T *__restrict__ out) {
  const int rowi = blockIdx.y;
  const int c = rowi % C;
  const float mu = __ldg(mean + c), is = __ldg(invstd + c), g = __ldg(gamma + c), bt = __ldg(beta + c);
  float k0 = 0.f, k1 = 0.f, gs = 0.f;
  if (MODE == 1) { k0 = __ldg(dbeta + c) * inv_M; k1 = __ldg(dgamma + c) * inv_M; gs = g * is; }
  const T *row = y + (size_t)rowi * S;
  const T *drow = MODE == 1 ? dz + (size_t)rowi * S : nullptr;
  T *orow = out + (size_t)rowi * S;
  auto f = [&](float yv, float dv) -> float {
    const float xh = (yv - mu) * is;
    const float z = fmaf(xh, g, bt);
    if (MODE == 0) return fmaxf(z, 0.f);
    const float dm = stored<T>(z) > 0.f ? dv : 0.f;
    return gs * ((dm - k0) - xh * k1);
  };
  const int tile = BN_THREADS * 4 * BN_UNR;
  if (VEC) {
    const int base = blockIdx.x * tile + threadIdx.x * 4;
    float4 v[BN_UNR], d[BN_UNR];
#pragma unroll
    for (int u = 0; u < BN_UNR; ++u) {
      const int p = base + u * BN_THREADS * 4;
      if (p < S) {
        v[u] = ldg4(row + p);
        if (MODE == 1) d[u] = ldg4(drow + p);
      }
    }
#pragma unroll
    for (int u = 0; u < BN_UNR; ++u) {
      const int p = base + u * BN_THREADS * 4;
      if (p < S) {
        float4 o;
        o.x = f(v[u].x, MODE == 1 ? d[u].x : 0.f); o.y = f(v[u].y, MODE == 1 ? d[u].y : 0.f);
        o.z = f(v[u].z, MODE == 1 ? d[u].z : 0.f); o.w = f(v[u].w, MODE == 1 ? d[u].w : 0.f);
        st4(orow + p, o);
      }
    }
  } else {
    for (int p = blockIdx.x * tile + threadIdx.x; p < min(S, (int)(blockIdx.x + 1) * tile); p += BN_THREADS)
      orow[p] = from_f32<T>(f(to_f32(__ldg(row + p)), MODE == 1 ? to_f32(__ldg(drow + p)) : 0.f));
  }
}

struct BnPlan {
  int splits, chunk;
  bool vec;
};

// the vector kernels move four elements of T per access: S % 4 == 0 and 4 * sizeof(T)-byte aligned rows
template <class T>
static BnPlan plan_bn(const void *a, const void *b, const void *c, int C, int S) {
  BnPlan p;
  p.vec = (S % 4 == 0) && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
                            reinterpret_cast<uintptr_t>(c)) & (4 * sizeof(T) - 1)) == 0;
  int splits = ceil_div(4 * kNumSMs, C);                       // ~4 CTAs per SM in total
  splits = max(1, min(min(splits, BN_MAX_SPLITS), ceil_div(S, BN_THREADS * 4)));
  int chunk = ceil_div(S, splits);
  chunk = (chunk + 3) & ~3;
  p.chunk = chunk;
  p.splits = ceil_div(S, chunk);
  return p;
}

// ----------------------------------------------------------------------------------------------------
// Last block of a set-abstraction MLP: BatchNorm + ReLU + max over the nsample neighbours
// (pointnet2_modules.py:256-259: F.max_pool2d(kernel=[1, nsample])).  The (B,C,npoint,nsample) activation is
// never written: the forward emits the pooled (B,C,npoint) tensor, the winning slot and the pre-BN value at
// that slot; the backward needs one pass (read y, write dy) because the incoming gradient is non-zero at one
// slot per group only, so the channel sums come from (B,C,npoint) data.
// A group of NS contiguous elements is handled by NS/4 adjacent lanes (four each): fully coalesced.
// Ties keep the lowest slot, like ATen's max_pool2d (strict '>'), which matters because ball-query padding
// repeats the first neighbour.  With bf16 storage the candidates are compared after rounding to bf16, so two slots
// that differ only below bf16 resolution tie and the lower one wins, as in max_pool2d on the rounded tensor.
// ----------------------------------------------------------------------------------------------------
constexpr int BP_UNR = 4;

template <class T, int NS>
__global__ void __launch_bounds__(BN_THREADS) bn_relu_pool_fwd_kernel(const T *__restrict__ y,
                                                                       const float *__restrict__ gamma,
                                                                       const float *__restrict__ beta,
                                                                       const float *__restrict__ mean,
                                                                       const float *__restrict__ invstd, int C, int np,
                                                                       T *__restrict__ pooled,
                                                                       uint8_t *__restrict__ argmax,
                                                                       T *__restrict__ ymax) {
  constexpr int LPG = NS / 4;                 // lanes per group
  constexpr int GPW = 32 / LPG;               // groups per warp per step
  const int rowi = blockIdx.y, c = rowi % C;
  const float mu = __ldg(mean + c), is = __ldg(invstd + c), g = __ldg(gamma + c), bt = __ldg(beta + c);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane % LPG, gl = lane / LPG;
  const int j0 = (blockIdx.x * (BN_THREADS / 32) + warp) * GPW * BP_UNR + gl;
  const T *row = y + (size_t)rowi * np * NS;
  float4 v[BP_UNR];
#pragma unroll
  for (int u = 0; u < BP_UNR; ++u) {
    const int j = j0 + u * GPW;
    if (j < np) v[u] = ldg4(row + (size_t)j * NS + sub * 4);
  }
#pragma unroll
  for (int u = 0; u < BP_UNR; ++u) {
    const int j = j0 + u * GPW;             // uniform across the LPG lanes of a group
    const bool ok = j < np;
    const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
    float bz = -INFINITY, by = 0.f;
    int bi = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float z = ok ? stored<T>(fmaf((e[q] - mu) * is, g, bt)) : 0.f;
      if (z > bz) { bz = z; bi = sub * 4 + q; by = e[q]; }
    }
#pragma unroll
    for (int o = 1; o < LPG; o <<= 1) {
      const float oz = __shfl_xor_sync(0xffffffffu, bz, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      const float oy = __shfl_xor_sync(0xffffffffu, by, o);
      if (oz > bz || (oz == bz && oi < bi)) { bz = oz; bi = oi; by = oy; }
    }
    if (ok && sub == 0) {
      const size_t o = (size_t)rowi * np + j;
      pooled[o] = from_f32<T>(fmaxf(bz, 0.f));
      argmax[o] = (uint8_t)bi;
      ymax[o] = from_f32<T>(by);
    }
  }
}

// one CTA per channel: dbeta = sum dm, dgamma = sum dm * xhat over the (B, npoint) winners; ROW as in
// bn_finalize_backward_kernel
template <class T, bool ROW>
__global__ void __launch_bounds__(BN_THREADS) bn_pool_bwd_reduce_kernel(
    const T *__restrict__ dpool, const T *__restrict__ ymax, const float *__restrict__ gamma,
    const float *__restrict__ beta, const float *__restrict__ mean, const float *__restrict__ invstd, int B, int C,
    int np, float *__restrict__ dgamma, float *__restrict__ dbeta, double M, double *__restrict__ row) {
  __shared__ double s_red[BN_THREADS / 32];
  const int c = blockIdx.x;
  const float mu = __ldg(mean + c), is = __ldg(invstd + c), g = __ldg(gamma + c), bt = __ldg(beta + c);
  float a0 = 0.f, a1 = 0.f;
  for (int b = 0; b < B; ++b) {
    const size_t base = ((size_t)b * C + c) * np;
    for (int j = threadIdx.x; j < np; j += BN_THREADS) {
      const float xh = (to_f32(__ldg(ymax + base + j)) - mu) * is;
      const float dm = stored<T>(fmaf(xh, g, bt)) > 0.f ? to_f32(__ldg(dpool + base + j)) : 0.f;
      a0 += dm;
      a1 = fmaf(dm, xh, a1);
    }
  }
  const double t0 = block_sum_double((double)a0, s_red);
  const double t1 = block_sum_double((double)a1, s_red);
  if (threadIdx.x == 0) {
    dbeta[c] = (float)t0;
    dgamma[c] = (float)t1;
    if (ROW) {
      row[(size_t)c * BN_SYNC_K + 0] = M;
      row[(size_t)c * BN_SYNC_K + 1] = t0;
      row[(size_t)c * BN_SYNC_K + 2] = t1;
    }
  }
}

template <class T, int NS>
__global__ void __launch_bounds__(BN_THREADS) bn_pool_bwd_apply_kernel(
    const T *__restrict__ y, const T *__restrict__ dpool, const uint8_t *__restrict__ argmax,
    const T *__restrict__ ymax, const float *__restrict__ gamma, const float *__restrict__ beta,
    const float *__restrict__ mean, const float *__restrict__ invstd, const float *__restrict__ dgamma,
    const float *__restrict__ dbeta, int C, int np, float inv_M, T *__restrict__ dy) {
  constexpr int LPG = NS / 4;
  constexpr int GPW = 32 / LPG;
  const int rowi = blockIdx.y, c = rowi % C;
  const float mu = __ldg(mean + c), is = __ldg(invstd + c), g = __ldg(gamma + c), bt = __ldg(beta + c);
  const float k0 = __ldg(dbeta + c) * inv_M, k1 = __ldg(dgamma + c) * inv_M, gs = g * is;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane % LPG, gl = lane / LPG;
  const int j0 = (blockIdx.x * (BN_THREADS / 32) + warp) * GPW * BP_UNR + gl;
  const T *row = y + (size_t)rowi * np * NS;
  T *orow = dy + (size_t)rowi * np * NS;
  float4 v[BP_UNR];
  float dp[BP_UNR], ym[BP_UNR];
  int am[BP_UNR];
#pragma unroll
  for (int u = 0; u < BP_UNR; ++u) {
    const int j = j0 + u * GPW;
    if (j < np) {
      v[u] = ldg4(row + (size_t)j * NS + sub * 4);
      const size_t o = (size_t)rowi * np + j;
      dp[u] = to_f32(__ldg(dpool + o));
      ym[u] = to_f32(__ldg(ymax + o));
      am[u] = (int)__ldg(argmax + o);
    }
  }
#pragma unroll
  for (int u = 0; u < BP_UNR; ++u) {
    const int j = j0 + u * GPW;
    if (j >= np) continue;
    const float dwin = stored<T>(fmaf((ym[u] - mu) * is, g, bt)) > 0.f ? dp[u] : 0.f;
    const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
    float o4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float xh = (e[q] - mu) * is;
      const float dm = (sub * 4 + q == am[u]) ? dwin : 0.f;
      o4[q] = gs * ((dm - k0) - xh * k1);
    }
    st4(orow + (size_t)j * NS + sub * 4, make_float4(o4[0], o4[1], o4[2], o4[3]));
  }
}

// ----------------------------------------------------------------------------------------------------
// Synchronised BatchNorm (torch.nn.SyncBatchNorm semantics) over the ranks of a process group.  The entry points
// split each pass at its one cross-channel reduction: a rank writes its per-channel fp64 row of BN_SYNC_K values,
//   forward : (n, mean, M2)                  n = B*S elements, M2 = sum (x - mean)^2,
//   backward: (n, sum dm, sum dm * xhat),
// the caller gathers the rows of all ranks into a (world, C, BN_SYNC_K) buffer, and the next entry point combines
// them in rank order on the device, so every rank derives bit-identical statistics and nothing depends on the
// collective's reduction order.  The global count comes from the rows, so ranks may hold different batch sizes.
// The reduction, normalise, pool and apply kernels are the ones above; the backward reductions write the row when
// ROW.  The finalisations below are kept apart from the plain ones on purpose: the plain variance s2/M - m1^2 and
// the merged M2 = s2 - s1*m1 can round differently, and so can the plain fp32(sum dm) * fp32(1/M) and the synced
// fp32(sum dm / n), so running the plain pass as a synced one of one rank would change its results (and add two
// launches per pass).
// ----------------------------------------------------------------------------------------------------

// forward, local: (n, mean, M2) from the shifted partial sums s1 = sum (x-K), s2 = sum (x-K)^2 of bn_reduce_kernel<0>
template <class T>
__global__ void bn_sync_moments_kernel(const T *__restrict__ y, const double *__restrict__ partial, int C, int S,
                                       int splits, double M, double *__restrict__ row) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s1, s2;
  sum_partials(partial, c, splits, s1, s2);
  const double K = (double)to_f32(__ldg(y + (size_t)c * S));
  const double m1 = s1 / M;
  double m2 = s2 - s1 * m1;
  if (m2 < 0.0) m2 = 0.0;
  row[(size_t)c * BN_SYNC_K + 0] = M;
  row[(size_t)c * BN_SYNC_K + 1] = K + m1;
  row[(size_t)c * BN_SYNC_K + 2] = m2;
}

// forward, global: Chan's pairwise merge of the ranks' (n, mean, M2) in rank order, then what
// bn_finalize_forward_kernel does with the merged moments.  Empty rows (n = 0) are skipped.
__global__ void bn_sync_finalize_forward_kernel(const double *__restrict__ rows, int world, int C, float eps,
                                                float momentum, float *__restrict__ running_mean,
                                                float *__restrict__ running_var, float *__restrict__ save_mean,
                                                float *__restrict__ save_invstd) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int r = 0; r < world; ++r) {
    const double *q = rows + ((size_t)r * C + c) * BN_SYNC_K;
    const double nb = q[0];
    if (!(nb > 0.0)) continue;
    const double nn = n + nb, d = q[1] - mean;
    mean += d * (nb / nn);
    m2 += q[2] + d * d * (n * nb / nn);
    n = nn;
  }
  const double var = n > 0.0 ? m2 / n : 0.0;
  save_mean[c] = (float)mean;
  save_invstd[c] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) running_mean[c] = (float)((1.0 - momentum) * running_mean[c] + momentum * mean);
  if (running_var) {
    const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
    running_var[c] = (float)((1.0 - momentum) * running_var[c] + momentum * unbiased);
  }
}

// backward, global: k0 = sum dm / n and k1 = sum dm * xhat / n over all ranks, rounded once to fp32.  The apply
// kernels read them in place of dbeta / dgamma with inv_M = 1, which leaves them unchanged.
__global__ void bn_sync_combine_backward_kernel(const double *__restrict__ rows, int world, int C,
                                                float *__restrict__ k0, float *__restrict__ k1) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double n = 0.0, s1 = 0.0, s2 = 0.0;
  for (int r = 0; r < world; ++r) {
    const double *q = rows + ((size_t)r * C + c) * BN_SYNC_K;
    n += q[0];
    s1 += q[1];
    s2 += q[2];
  }
  k0[c] = n > 0.0 ? (float)(s1 / n) : 0.f;
  k1[c] = n > 0.0 ? (float)(s2 / n) : 0.f;
}

}  // namespace spc

using namespace spc;

extern "C" size_t spc_bn_relu_workspace_bytes(int C) {
  return C > 0 ? (size_t)C * BN_MAX_SPLITS * 2 * sizeof(double) : 0;
}

// ---- checks and launchers shared by the plain and the synced entry points ----------------------------------------
// Sizes and pointers of a pass over y (B, C, np * ns); the passes without max-pool give ns = 1.  The plain passes need
// B >= 1; the synced ones take B = 0 (min_B = 0): a rank with an empty shard still takes part in every exchange, so
// the other ranks are not left waiting, and its per-sample tensors may then be NULL.  Per-channel tensors never.
static int check_bn(const char *what, int B, int min_B, int C, int np, int ns, int world,
                    std::initializer_list<const void *> samples, std::initializer_list<const void *> channels) {
  SPC_CHECK_ARG(B >= min_B && C >= 1 && C <= 65535 && np >= 1 && ns >= 1 && (long long)np * ns < (1LL << 31) && world >= 1,
                "%s: bad sizes B=%d C=%d S=%d*%d world=%d", what, B, C, np, ns, world);
  bool ok = true;
  for (const void *q : channels) ok = ok && q;
  if (B > 0) for (const void *q : samples) ok = ok && q;
  SPC_CHECK_ARG(ok, "%s: null pointer", what);
  return SPC_OK;
}

static int check_workspace(const char *what, const void *workspace, size_t workspace_bytes, int C) {
  SPC_CHECK_ARG(workspace && workspace_bytes >= spc_bn_relu_workspace_bytes(C) && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0,
                "%s: workspace of spc_bn_relu_workspace_bytes(C) bytes required", what);
  return SPC_OK;
}

// the pool kernels exist for nsample 16, 32 and 64, and read y and write dy four elements of T at a time
template <class T>
static int check_pool(const char *what, int nsample, const void *y, const void *dy) {
  if (!(nsample == 16 || nsample == 32 || nsample == 64) ||
      ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(dy)) & (4 * sizeof(T) - 1))) {
    set_error("%s: nsample=%d not in {16,32,64} or tensors not %d-byte aligned", what, nsample, (int)(4 * sizeof(T)));
    return SPC_ERR_UNSUPPORTED;
  }
  return SPC_OK;
}

// The reductions take any B.  The normalise / apply / pool kernels put B*C rows on grid.y, so they are launched once
// per slice of at most 65535 / C batch rows: one launch whenever B*C <= 65535.
static int sync_batch_slice(int C) { return max(1, 65535 / C); }

template <int MODE, class T>
static void launch_reduce(const BnPlan &p, const T *y, const T *dz, const float *gamma, const float *beta,
                          const float *mean, const float *invstd, int B, int C, int S, double *partial,
                          cudaStream_t stream) {
  const dim3 grid(p.splits, C);
  if (p.vec) bn_reduce_kernel<T, MODE, true><<<grid, BN_THREADS, 0, stream>>>(y, dz, gamma, beta, mean, invstd, B, C, S, p.chunk, partial);
  else bn_reduce_kernel<T, MODE, false><<<grid, BN_THREADS, 0, stream>>>(y, dz, gamma, beta, mean, invstd, B, C, S, p.chunk, partial);
}

// MODE 0: out = z (dz, dgamma, dbeta unused).  MODE 1: out = dy with k0 = dbeta * inv_M, k1 = dgamma * inv_M.
template <int MODE, class T>
static void launch_apply(bool vec, const T *y, const T *dz, const float *gamma, const float *beta,
                         const float *mean, const float *invstd, const float *dgamma, const float *dbeta, int B, int C,
                         int S, float inv_M, T *out, cudaStream_t stream) {
  const int slice = sync_batch_slice(C);
  for (int b0 = 0; b0 < B; b0 += slice) {
    const size_t off = (size_t)b0 * C * S;
    const T *dzs = MODE == 1 ? dz + off : nullptr;
    const dim3 grid(ceil_div(S, BN_THREADS * 4 * BN_UNR), min(slice, B - b0) * C);
    if (vec) bn_apply_kernel<T, MODE, true><<<grid, BN_THREADS, 0, stream>>>(y + off, dzs, gamma, beta, mean, invstd, dgamma, dbeta, C, S, inv_M, out + off);
    else bn_apply_kernel<T, MODE, false><<<grid, BN_THREADS, 0, stream>>>(y + off, dzs, gamma, beta, mean, invstd, dgamma, dbeta, C, S, inv_M, out + off);
  }
}

// calls launch(std::integral_constant<int, NS>) for the nsample check_pool accepted
template <class F>
static void dispatch_nsample(int nsample, F &&launch) {
  if (nsample == 16) launch(std::integral_constant<int, 16>());
  else if (nsample == 32) launch(std::integral_constant<int, 32>());
  else launch(std::integral_constant<int, 64>());
}

// grid.x of the pool kernels: BN_THREADS / 32 warps, each over 32 / (nsample / 4) groups BP_UNR times
static int pool_tiles(int npoint, int nsample) {
  return ceil_div(npoint, (BN_THREADS / 32) * (32 / (nsample / 4)) * BP_UNR);
}

template <class T>
static void launch_pool_fwd(const T *y, const float *gamma, const float *beta, const float *mean,
                            const float *invstd, int B, int C, int npoint, int nsample, T *pooled, uint8_t *argmax,
                            T *ymax, cudaStream_t stream) {
  const int slice = sync_batch_slice(C);
  for (int b0 = 0; b0 < B; b0 += slice) {
    const size_t po = (size_t)b0 * C * npoint, yo = po * nsample;
    const dim3 grid(pool_tiles(npoint, nsample), min(slice, B - b0) * C);
    dispatch_nsample(nsample, [&](auto ns) {
      bn_relu_pool_fwd_kernel<T, decltype(ns)::value><<<grid, BN_THREADS, 0, stream>>>(
          y + yo, gamma, beta, mean, invstd, C, npoint, pooled + po, argmax + po, ymax + po);
    });
  }
}

// dy from dpool, with k0 = dbeta * inv_M, k1 = dgamma * inv_M
template <class T>
static void launch_pool_bwd(const T *y, const T *dpool, const uint8_t *argmax, const T *ymax,
                            const float *gamma, const float *beta, const float *mean, const float *invstd,
                            const float *dgamma, const float *dbeta, int B, int C, int npoint, int nsample, float inv_M,
                            T *dy, cudaStream_t stream) {
  const int slice = sync_batch_slice(C);
  for (int b0 = 0; b0 < B; b0 += slice) {
    const size_t po = (size_t)b0 * C * npoint, yo = po * nsample;
    const dim3 grid(pool_tiles(npoint, nsample), min(slice, B - b0) * C);
    dispatch_nsample(nsample, [&](auto ns) {
      bn_pool_bwd_apply_kernel<T, decltype(ns)::value><<<grid, BN_THREADS, 0, stream>>>(
          y + yo, dpool + po, argmax + po, ymax + po, gamma, beta, mean, invstd, dgamma, dbeta, C, npoint, inv_M, dy + yo);
    });
  }
}

// ---- plain passes -------------------------------------------------------------------------------------------------
template <class T>
static int bn_relu_train_forward(const T *y, const float *gamma, const float *beta, int B, int C, int S, float eps,
                                 float momentum, float *running_mean, float *running_var, T *z, float *save_mean,
                                 float *save_invstd, void *workspace, size_t workspace_bytes, void *stream_) {
  if (const int e = check_bn("bn_relu_forward", B, 1, C, S, 1, 1, {y, z}, {gamma, beta, save_mean, save_invstd})) return e;
  if (const int e = check_workspace("bn_relu_forward", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  double *partial = reinterpret_cast<double *>(workspace);
  const BnPlan p = plan_bn<T>(y, z, y, C, S);
  launch_reduce<0>(p, y, (const T *)nullptr, gamma, beta, nullptr, nullptr, B, C, S, partial, stream);
  bn_finalize_forward_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(y, partial, C, S, p.splits, (double)B * S, eps, momentum,
                                                                   running_mean, running_var, save_mean, save_invstd);
  launch_apply<0>(p.vec, y, (const T *)nullptr, gamma, beta, save_mean, save_invstd, nullptr, nullptr, B, C, S, 0.f, z, stream);
  SPC_LAUNCH_CHECK("bn_relu_train_forward");
  return SPC_OK;
}

template <class T>
static int bn_relu_train_backward(const T *dz, const T *y, const float *gamma, const float *beta, const float *save_mean,
                                  const float *save_invstd, int B, int C, int S, T *dy, float *dgamma, float *dbeta,
                                  void *workspace, size_t workspace_bytes, void *stream_) {
  if (const int e = check_bn("bn_relu_backward", B, 1, C, S, 1, 1, {dz, y, dy},
                             {gamma, beta, save_mean, save_invstd, dgamma, dbeta})) return e;
  if (const int e = check_workspace("bn_relu_backward", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  double *partial = reinterpret_cast<double *>(workspace);
  const BnPlan p = plan_bn<T>(y, dz, dy, C, S);
  launch_reduce<1>(p, y, dz, gamma, beta, save_mean, save_invstd, B, C, S, partial, stream);
  bn_finalize_backward_kernel<false><<<ceil_div(C, 128), 128, 0, stream>>>(partial, C, p.splits, dgamma, dbeta, 0.0, nullptr);
  const float inv_M = (float)(1.0 / ((double)B * S));
  launch_apply<1>(p.vec, y, dz, gamma, beta, save_mean, save_invstd, dgamma, dbeta, B, C, S, inv_M, dy, stream);
  SPC_LAUNCH_CHECK("bn_relu_train_backward");
  return SPC_OK;
}

template <class T>
static int bn_relu_maxpool_train_forward(const T *y, const float *gamma, const float *beta, int B, int C, int npoint,
                                         int nsample, float eps, float momentum, float *running_mean,
                                         float *running_var, T *pooled, uint8_t *argmax, T *ymax, float *save_mean,
                                         float *save_invstd, void *workspace, size_t workspace_bytes, void *stream_) {
  if (const int e = check_bn("bn_relu_maxpool_forward", B, 1, C, npoint, nsample, 1, {y, pooled, argmax, ymax},
                             {gamma, beta, save_mean, save_invstd})) return e;
  if (const int e = check_pool<T>("bn_relu_maxpool_forward", nsample, y, nullptr)) return e;
  if (const int e = check_workspace("bn_relu_maxpool_forward", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  const int S = npoint * nsample;
  double *partial = reinterpret_cast<double *>(workspace);
  const BnPlan p = plan_bn<T>(y, y, y, C, S);     // vector: y is aligned (check_pool) and S a multiple of 16
  launch_reduce<0>(p, y, (const T *)nullptr, gamma, beta, nullptr, nullptr, B, C, S, partial, stream);
  bn_finalize_forward_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(y, partial, C, S, p.splits, (double)B * S, eps, momentum,
                                                                   running_mean, running_var, save_mean, save_invstd);
  launch_pool_fwd(y, gamma, beta, save_mean, save_invstd, B, C, npoint, nsample, pooled, argmax, ymax, stream);
  SPC_LAUNCH_CHECK("bn_relu_maxpool_train_forward");
  return SPC_OK;
}

template <class T>
static int bn_relu_maxpool_train_backward(const T *dpool, const uint8_t *argmax, const T *ymax, const T *y,
                                          const float *gamma, const float *beta, const float *save_mean,
                                          const float *save_invstd, int B, int C, int npoint, int nsample, T *dy,
                                          float *dgamma, float *dbeta, void *stream_) {
  if (const int e = check_bn("bn_relu_maxpool_backward", B, 1, C, npoint, nsample, 1, {dpool, argmax, ymax, y, dy},
                             {gamma, beta, save_mean, save_invstd, dgamma, dbeta})) return e;
  if (const int e = check_pool<T>("bn_relu_maxpool_backward", nsample, y, dy)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  bn_pool_bwd_reduce_kernel<T, false><<<C, BN_THREADS, 0, stream>>>(dpool, ymax, gamma, beta, save_mean, save_invstd, B, C,
                                                                    npoint, dgamma, dbeta, 0.0, nullptr);
  const float inv_M = (float)(1.0 / ((double)B * npoint * nsample));
  launch_pool_bwd(y, dpool, argmax, ymax, gamma, beta, save_mean, save_invstd, dgamma, dbeta, B, C, npoint, nsample,
                  inv_M, dy, stream);
  SPC_LAUNCH_CHECK("bn_relu_maxpool_train_backward");
  return SPC_OK;
}

// ---- synchronised passes (see BN_SYNC_K above) --------------------------------------------------------------------
// Each takes any local B >= 0; a rank with B = 0 contributes a row with n = 0, which the combinations skip.
template <class T>
static int bn_relu_sync_stats(const T *y, int B, int C, int S, double *stats, void *workspace, size_t workspace_bytes,
                              void *stream_) {
  if (const int e = check_bn("bn_relu_sync_stats", B, 0, C, S, 1, 1, {y}, {stats})) return e;
  if (const int e = check_workspace("bn_relu_sync_stats", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  if (B == 0) {                                   // (n, mean, M2) = 0: an empty shard
    SPC_CUDA(cudaMemsetAsync(stats, 0, (size_t)C * BN_SYNC_K * sizeof(double), stream));
    return SPC_OK;
  }
  double *partial = reinterpret_cast<double *>(workspace);
  const BnPlan p = plan_bn<T>(y, y, y, C, S);
  launch_reduce<0>(p, y, (const T *)nullptr, nullptr, nullptr, nullptr, nullptr, B, C, S, partial, stream);
  bn_sync_moments_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(y, partial, C, S, p.splits, (double)B * S, stats);
  SPC_LAUNCH_CHECK("bn_relu_sync_stats");
  return SPC_OK;
}

template <class T>
static int bn_relu_sync_forward(const T *y, const float *gamma, const float *beta, int B, int C, int S, int world,
                                const double *stats_all, float eps, float momentum, float *running_mean,
                                float *running_var, T *z, float *save_mean, float *save_invstd, void *stream_) {
  if (const int e = check_bn("bn_relu_sync_forward", B, 0, C, S, 1, world, {y, z},
                             {gamma, beta, stats_all, save_mean, save_invstd})) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  bn_sync_finalize_forward_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(stats_all, world, C, eps, momentum, running_mean,
                                                                        running_var, save_mean, save_invstd);
  const BnPlan p = plan_bn<T>(y, z, y, C, S);
  launch_apply<0>(p.vec, y, (const T *)nullptr, gamma, beta, save_mean, save_invstd, nullptr, nullptr, B, C, S, 0.f, z, stream);
  SPC_LAUNCH_CHECK("bn_relu_sync_forward");
  return SPC_OK;
}

template <class T>
static int bn_relu_sync_backward_reduce(const T *dz, const T *y, const float *gamma, const float *beta,
                                        const float *save_mean, const float *save_invstd, int B, int C, int S,
                                        float *dgamma, float *dbeta, double *stats, void *workspace,
                                        size_t workspace_bytes, void *stream_) {
  if (const int e = check_bn("bn_relu_sync_backward_reduce", B, 0, C, S, 1, 1, {dz, y},
                             {gamma, beta, save_mean, save_invstd, dgamma, dbeta, stats})) return e;
  if (const int e = check_workspace("bn_relu_sync_backward_reduce", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  if (B == 0) {                                   // empty shard: zero local sums and an n = 0 row
    SPC_CUDA(cudaMemsetAsync(stats, 0, (size_t)C * BN_SYNC_K * sizeof(double), stream));
    SPC_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)C * sizeof(float), stream));
    SPC_CUDA(cudaMemsetAsync(dbeta, 0, (size_t)C * sizeof(float), stream));
    return SPC_OK;
  }
  double *partial = reinterpret_cast<double *>(workspace);
  const BnPlan p = plan_bn<T>(y, dz, dz, C, S);
  launch_reduce<1>(p, y, dz, gamma, beta, save_mean, save_invstd, B, C, S, partial, stream);
  bn_finalize_backward_kernel<true><<<ceil_div(C, 128), 128, 0, stream>>>(partial, C, p.splits, dgamma, dbeta,
                                                                          (double)B * S, stats);
  SPC_LAUNCH_CHECK("bn_relu_sync_backward_reduce");
  return SPC_OK;
}

template <class T>
static int bn_relu_sync_backward(const T *dz, const T *y, const float *gamma, const float *beta, const float *save_mean,
                                 const float *save_invstd, int B, int C, int S, int world, const double *stats_all,
                                 T *dy, void *workspace, size_t workspace_bytes, void *stream_) {
  if (const int e = check_bn("bn_relu_sync_backward", B, 0, C, S, 1, world, {dz, y, dy},
                             {gamma, beta, save_mean, save_invstd, stats_all})) return e;
  if (const int e = check_workspace("bn_relu_sync_backward", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  float *k0 = reinterpret_cast<float *>(workspace), *k1 = k0 + C;
  bn_sync_combine_backward_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(stats_all, world, C, k0, k1);
  const BnPlan p = plan_bn<T>(y, dz, dy, C, S);
  launch_apply<1>(p.vec, y, dz, gamma, beta, save_mean, save_invstd, k1, k0, B, C, S, 1.f, dy, stream);
  SPC_LAUNCH_CHECK("bn_relu_sync_backward");
  return SPC_OK;
}

// Max-pool variant.  Its statistics phase is bn_relu_sync_stats with S = npoint * nsample.
template <class T>
static int bn_relu_maxpool_sync_forward(const T *y, const float *gamma, const float *beta, int B, int C, int npoint,
                                        int nsample, int world, const double *stats_all, float eps, float momentum,
                                        float *running_mean, float *running_var, T *pooled, uint8_t *argmax, T *ymax,
                                        float *save_mean, float *save_invstd, void *stream_) {
  if (const int e = check_bn("bn_relu_maxpool_sync_forward", B, 0, C, npoint, nsample, world, {y, pooled, argmax, ymax},
                             {gamma, beta, stats_all, save_mean, save_invstd})) return e;
  if (const int e = check_pool<T>("bn_relu_maxpool_sync_forward", nsample, y, nullptr)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  bn_sync_finalize_forward_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(stats_all, world, C, eps, momentum, running_mean,
                                                                        running_var, save_mean, save_invstd);
  launch_pool_fwd(y, gamma, beta, save_mean, save_invstd, B, C, npoint, nsample, pooled, argmax, ymax, stream);
  SPC_LAUNCH_CHECK("bn_relu_maxpool_sync_forward");
  return SPC_OK;
}

template <class T>
static int bn_relu_maxpool_sync_backward_reduce(const T *dpool, const T *ymax, const float *gamma, const float *beta,
                                                const float *save_mean, const float *save_invstd, int B, int C,
                                                int npoint, int nsample, float *dgamma, float *dbeta, double *stats,
                                                void *stream_) {
  if (const int e = check_bn("bn_relu_maxpool_sync_backward_reduce", B, 0, C, npoint, nsample, 1, {dpool, ymax},
                             {gamma, beta, save_mean, save_invstd, dgamma, dbeta, stats})) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  bn_pool_bwd_reduce_kernel<T, true><<<C, BN_THREADS, 0, stream>>>(dpool, ymax, gamma, beta, save_mean, save_invstd, B, C,
                                                                   npoint, dgamma, dbeta, (double)B * npoint * nsample, stats);
  SPC_LAUNCH_CHECK("bn_relu_maxpool_sync_backward_reduce");
  return SPC_OK;
}

template <class T>
static int bn_relu_maxpool_sync_backward(const T *dpool, const uint8_t *argmax, const T *ymax, const T *y,
                                         const float *gamma, const float *beta, const float *save_mean,
                                         const float *save_invstd, int B, int C, int npoint, int nsample, int world,
                                         const double *stats_all, T *dy, void *workspace, size_t workspace_bytes,
                                         void *stream_) {
  if (const int e = check_bn("bn_relu_maxpool_sync_backward", B, 0, C, npoint, nsample, world,
                             {dpool, argmax, ymax, y, dy}, {gamma, beta, save_mean, save_invstd, stats_all})) return e;
  if (const int e = check_pool<T>("bn_relu_maxpool_sync_backward", nsample, y, dy)) return e;
  if (const int e = check_workspace("bn_relu_maxpool_sync_backward", workspace, workspace_bytes, C)) return e;
  cudaStream_t stream = (cudaStream_t)stream_;
  float *k0 = reinterpret_cast<float *>(workspace), *k1 = k0 + C;
  bn_sync_combine_backward_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(stats_all, world, C, k0, k1);
  launch_pool_bwd(y, dpool, argmax, ymax, gamma, beta, save_mean, save_invstd, k1, k0, B, C, npoint, nsample, 1.f, dy,
                  stream);
  SPC_LAUNCH_CHECK("bn_relu_maxpool_sync_backward");
  return SPC_OK;
}

// ---- C entry points: fp32 storage, and bf16 storage (the void pointers are __nv_bfloat16 tensors) ------------------
#define BF(p) static_cast<const bf16 *>(p)
#define BFW(p) static_cast<bf16 *>(p)

extern "C" int spc_bn_relu_train_forward(const float *y, const float *gamma, const float *beta, int B, int C, int S,
                                         float eps, float momentum, float *running_mean, float *running_var,
                                         float *z, float *save_mean, float *save_invstd, void *workspace,
                                         size_t workspace_bytes, void *stream) {
  return bn_relu_train_forward(y, gamma, beta, B, C, S, eps, momentum, running_mean, running_var, z, save_mean,
                               save_invstd, workspace, workspace_bytes, stream);
}
extern "C" int spc_bn_relu_train_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C, int S,
                                              float eps, float momentum, float *running_mean, float *running_var,
                                              void *z, float *save_mean, float *save_invstd, void *workspace,
                                              size_t workspace_bytes, void *stream) {
  return bn_relu_train_forward(BF(y), gamma, beta, B, C, S, eps, momentum, running_mean, running_var, BFW(z), save_mean,
                               save_invstd, workspace, workspace_bytes, stream);
}

extern "C" int spc_bn_relu_train_backward(const float *dz, const float *y, const float *gamma, const float *beta,
                                          const float *save_mean, const float *save_invstd, int B, int C, int S,
                                          float *dy, float *dgamma, float *dbeta, void *workspace,
                                          size_t workspace_bytes, void *stream) {
  return bn_relu_train_backward(dz, y, gamma, beta, save_mean, save_invstd, B, C, S, dy, dgamma, dbeta, workspace,
                                workspace_bytes, stream);
}
extern "C" int spc_bn_relu_train_backward_bf16(const void *dz, const void *y, const float *gamma, const float *beta,
                                               const float *save_mean, const float *save_invstd, int B, int C, int S,
                                               void *dy, float *dgamma, float *dbeta, void *workspace,
                                               size_t workspace_bytes, void *stream) {
  return bn_relu_train_backward(BF(dz), BF(y), gamma, beta, save_mean, save_invstd, B, C, S, BFW(dy), dgamma, dbeta,
                                workspace, workspace_bytes, stream);
}

extern "C" int spc_bn_relu_maxpool_train_forward(const float *y, const float *gamma, const float *beta, int B, int C,
                                                 int npoint, int nsample, float eps, float momentum,
                                                 float *running_mean, float *running_var, float *pooled,
                                                 uint8_t *argmax, float *ymax, float *save_mean, float *save_invstd,
                                                 void *workspace, size_t workspace_bytes, void *stream) {
  return bn_relu_maxpool_train_forward(y, gamma, beta, B, C, npoint, nsample, eps, momentum, running_mean, running_var,
                                       pooled, argmax, ymax, save_mean, save_invstd, workspace, workspace_bytes, stream);
}
extern "C" int spc_bn_relu_maxpool_train_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C,
                                                      int npoint, int nsample, float eps, float momentum,
                                                      float *running_mean, float *running_var, void *pooled,
                                                      uint8_t *argmax, void *ymax, float *save_mean, float *save_invstd,
                                                      void *workspace, size_t workspace_bytes, void *stream) {
  return bn_relu_maxpool_train_forward(BF(y), gamma, beta, B, C, npoint, nsample, eps, momentum, running_mean,
                                       running_var, BFW(pooled), argmax, BFW(ymax), save_mean, save_invstd, workspace,
                                       workspace_bytes, stream);
}

extern "C" int spc_bn_relu_maxpool_train_backward(const float *dpool, const uint8_t *argmax, const float *ymax,
                                                  const float *y, const float *gamma, const float *beta,
                                                  const float *save_mean, const float *save_invstd, int B, int C,
                                                  int npoint, int nsample, float *dy, float *dgamma, float *dbeta,
                                                  void *stream) {
  return bn_relu_maxpool_train_backward(dpool, argmax, ymax, y, gamma, beta, save_mean, save_invstd, B, C, npoint,
                                        nsample, dy, dgamma, dbeta, stream);
}
extern "C" int spc_bn_relu_maxpool_train_backward_bf16(const void *dpool, const uint8_t *argmax, const void *ymax,
                                                       const void *y, const float *gamma, const float *beta,
                                                       const float *save_mean, const float *save_invstd, int B, int C,
                                                       int npoint, int nsample, void *dy, float *dgamma, float *dbeta,
                                                       void *stream) {
  return bn_relu_maxpool_train_backward(BF(dpool), argmax, BF(ymax), BF(y), gamma, beta, save_mean, save_invstd, B, C,
                                        npoint, nsample, BFW(dy), dgamma, dbeta, stream);
}

extern "C" int spc_bn_relu_sync_stats(const float *y, int B, int C, int S, double *stats, void *workspace,
                                      size_t workspace_bytes, void *stream) {
  return bn_relu_sync_stats(y, B, C, S, stats, workspace, workspace_bytes, stream);
}
extern "C" int spc_bn_relu_sync_stats_bf16(const void *y, int B, int C, int S, double *stats, void *workspace,
                                           size_t workspace_bytes, void *stream) {
  return bn_relu_sync_stats(BF(y), B, C, S, stats, workspace, workspace_bytes, stream);
}

extern "C" int spc_bn_relu_sync_forward(const float *y, const float *gamma, const float *beta, int B, int C, int S,
                                        int world, const double *stats_all, float eps, float momentum,
                                        float *running_mean, float *running_var, float *z, float *save_mean,
                                        float *save_invstd, void *stream) {
  return bn_relu_sync_forward(y, gamma, beta, B, C, S, world, stats_all, eps, momentum, running_mean, running_var, z,
                              save_mean, save_invstd, stream);
}
extern "C" int spc_bn_relu_sync_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C, int S,
                                             int world, const double *stats_all, float eps, float momentum,
                                             float *running_mean, float *running_var, void *z, float *save_mean,
                                             float *save_invstd, void *stream) {
  return bn_relu_sync_forward(BF(y), gamma, beta, B, C, S, world, stats_all, eps, momentum, running_mean, running_var,
                              BFW(z), save_mean, save_invstd, stream);
}

extern "C" int spc_bn_relu_sync_backward_reduce(const float *dz, const float *y, const float *gamma, const float *beta,
                                                const float *save_mean, const float *save_invstd, int B, int C, int S,
                                                float *dgamma, float *dbeta, double *stats, void *workspace,
                                                size_t workspace_bytes, void *stream) {
  return bn_relu_sync_backward_reduce(dz, y, gamma, beta, save_mean, save_invstd, B, C, S, dgamma, dbeta, stats,
                                      workspace, workspace_bytes, stream);
}
extern "C" int spc_bn_relu_sync_backward_reduce_bf16(const void *dz, const void *y, const float *gamma,
                                                     const float *beta, const float *save_mean,
                                                     const float *save_invstd, int B, int C, int S, float *dgamma,
                                                     float *dbeta, double *stats, void *workspace,
                                                     size_t workspace_bytes, void *stream) {
  return bn_relu_sync_backward_reduce(BF(dz), BF(y), gamma, beta, save_mean, save_invstd, B, C, S, dgamma, dbeta, stats,
                                      workspace, workspace_bytes, stream);
}

extern "C" int spc_bn_relu_sync_backward(const float *dz, const float *y, const float *gamma, const float *beta,
                                         const float *save_mean, const float *save_invstd, int B, int C, int S,
                                         int world, const double *stats_all, float *dy, void *workspace,
                                         size_t workspace_bytes, void *stream) {
  return bn_relu_sync_backward(dz, y, gamma, beta, save_mean, save_invstd, B, C, S, world, stats_all, dy, workspace,
                               workspace_bytes, stream);
}
extern "C" int spc_bn_relu_sync_backward_bf16(const void *dz, const void *y, const float *gamma, const float *beta,
                                              const float *save_mean, const float *save_invstd, int B, int C, int S,
                                              int world, const double *stats_all, void *dy, void *workspace,
                                              size_t workspace_bytes, void *stream) {
  return bn_relu_sync_backward(BF(dz), BF(y), gamma, beta, save_mean, save_invstd, B, C, S, world, stats_all, BFW(dy),
                               workspace, workspace_bytes, stream);
}

extern "C" int spc_bn_relu_maxpool_sync_forward(const float *y, const float *gamma, const float *beta, int B, int C,
                                                int npoint, int nsample, int world, const double *stats_all,
                                                float eps, float momentum, float *running_mean, float *running_var,
                                                float *pooled, uint8_t *argmax, float *ymax, float *save_mean,
                                                float *save_invstd, void *stream) {
  return bn_relu_maxpool_sync_forward(y, gamma, beta, B, C, npoint, nsample, world, stats_all, eps, momentum,
                                      running_mean, running_var, pooled, argmax, ymax, save_mean, save_invstd, stream);
}
extern "C" int spc_bn_relu_maxpool_sync_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C,
                                                     int npoint, int nsample, int world, const double *stats_all,
                                                     float eps, float momentum, float *running_mean,
                                                     float *running_var, void *pooled, uint8_t *argmax, void *ymax,
                                                     float *save_mean, float *save_invstd, void *stream) {
  return bn_relu_maxpool_sync_forward(BF(y), gamma, beta, B, C, npoint, nsample, world, stats_all, eps, momentum,
                                      running_mean, running_var, BFW(pooled), argmax, BFW(ymax), save_mean, save_invstd,
                                      stream);
}

extern "C" int spc_bn_relu_maxpool_sync_backward_reduce(const float *dpool, const float *ymax, const float *gamma,
                                                        const float *beta, const float *save_mean,
                                                        const float *save_invstd, int B, int C, int npoint,
                                                        int nsample, float *dgamma, float *dbeta, double *stats,
                                                        void *stream) {
  return bn_relu_maxpool_sync_backward_reduce(dpool, ymax, gamma, beta, save_mean, save_invstd, B, C, npoint, nsample,
                                              dgamma, dbeta, stats, stream);
}
extern "C" int spc_bn_relu_maxpool_sync_backward_reduce_bf16(const void *dpool, const void *ymax, const float *gamma,
                                                             const float *beta, const float *save_mean,
                                                             const float *save_invstd, int B, int C, int npoint,
                                                             int nsample, float *dgamma, float *dbeta, double *stats,
                                                             void *stream) {
  return bn_relu_maxpool_sync_backward_reduce(BF(dpool), BF(ymax), gamma, beta, save_mean, save_invstd, B, C, npoint,
                                              nsample, dgamma, dbeta, stats, stream);
}

extern "C" int spc_bn_relu_maxpool_sync_backward(const float *dpool, const uint8_t *argmax, const float *ymax,
                                                 const float *y, const float *gamma, const float *beta,
                                                 const float *save_mean, const float *save_invstd, int B, int C,
                                                 int npoint, int nsample, int world, const double *stats_all,
                                                 float *dy, void *workspace, size_t workspace_bytes, void *stream) {
  return bn_relu_maxpool_sync_backward(dpool, argmax, ymax, y, gamma, beta, save_mean, save_invstd, B, C, npoint,
                                       nsample, world, stats_all, dy, workspace, workspace_bytes, stream);
}
extern "C" int spc_bn_relu_maxpool_sync_backward_bf16(const void *dpool, const uint8_t *argmax, const void *ymax,
                                                      const void *y, const float *gamma, const float *beta,
                                                      const float *save_mean, const float *save_invstd, int B, int C,
                                                      int npoint, int nsample, int world, const double *stats_all,
                                                      void *dy, void *workspace, size_t workspace_bytes, void *stream) {
  return bn_relu_maxpool_sync_backward(BF(dpool), argmax, BF(ymax), BF(y), gamma, beta, save_mean, save_invstd, B, C,
                                       npoint, nsample, world, stats_all, BFW(dy), workspace, workspace_bytes, stream);
}
