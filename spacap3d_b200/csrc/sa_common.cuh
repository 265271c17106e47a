// sa_common.cuh -- offsets into the 128-byte-swizzle K-major shared-memory layout, weight staging, the pooled epilogue
// and the launch parameters shared by the two fused set-abstraction kernels: sa_fused.cu (projected layer 0, SA2-SA4 /
// vote aggregation) and sa_inline.cu (in-line layer 0, SA1).  The PTX wrappers they use are in ptx.cuh.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "ptx.cuh"

namespace spc {

// byte offset of the 16-byte chunk (row, kc) of a [rows x K] fp16 operand in the layout of make_smem_desc_sw128
// (ptx.cuh)
__device__ __forceinline__ uint32_t sw128_off(int row, int kc, int rows) {
  return (uint32_t)((kc >> 3) * rows * 128 + row * 128 + (((kc & 7) ^ (row & 7)) << 4));
}
// byte offset of K step kk (16 elements) relative to the operand base
__device__ __forceinline__ uint32_t sw128_kstep(int kk, int rows) {
  return (uint32_t)((kk >> 2) * rows * 128 + (kk & 3) * 32);
}

// relu + round-to-nearest fp16 conversion (saturating) + packing of two floats in ONE instruction
// (cvt.rn.satfinite.relu.f16x2.f32: first source -> upper half, second source -> lower half)
__device__ __forceinline__ uint32_t pack_relu_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// ---------------------------------------------------------------------------------------------
struct SaFusedParams {
  const float *xyz;       // (B,n,3)
  const float *new_xyz;   // (B,np,3)
  const int32_t *idx;     // (B,np,ns)
  const __half *G;        // projected form: (B,n,C1) per-point feature projection (BN scale folded)
  const float *feat;      // in-line form: (B,Cf,n) raw features or nullptr
  const float *W0;        // (C1, 3+Cf) folded, fp32; projected form: Cf = 0, i.e. the xyz columns only
  const float *b0;        // (C1)
  int Cf;
  float radius;           // divide relative xyz by this (1.0 when normalize_xyz is off)
  const __half *W1;       // (C2,C1) folded, fp16 row-major
  const float *b1;        // (C2)
  const __half *W2;       // (C3,C2)
  const float *b2;        // (C3)
  float *out;             // (B,C3,np)
  __half *out_pm;         // optional (B,np,C3): the same result point-major in fp16 (next layer's GEMM input)
  int B, n, np, ns;
  int num_tiles;          // B*np*ns/128
  int min_tiles;          // host-side launch hint (see spc_sa_fused_forward_ex), unused on the device
  unsigned tps_magic;     // ceil(2^32 / tiles_per_scene) when tile / tiles_per_scene == umulhi(tile, magic) for every
                          // tile of this launch, else 0 (the kernels then divide)
};

constexpr int SA_ROWS = 128;        // rows (centre,neighbour pairs) per tile
constexpr int SA_MAX_K0 = 3 + 13;   // the in-line form supports up to 13 raw feature channels (four K steps of 4 inputs)

// scene of a tile (tiles never straddle scenes: npoint*nsample % 128 == 0 is checked at launch)
__device__ __forceinline__ int sa_tile_scene(const SaFusedParams &p, int tile, int tiles_per_scene) {
  return p.tps_magic ? (int)__umulhi((unsigned)tile, p.tps_magic) : tile / tiles_per_scene;
}

// Row-major fp16 weights (ROWS, 8*KCH) -> the swizzled UMMA layout in shared memory; 8 x 16-byte loads in flight
// per thread.
template <int ROWS, int KCH, int NT>
__device__ __forceinline__ void sa_stage_weights(uint8_t *dst, const __half *src, int t) {
  constexpr int N = ROWS * KCH;
  for (int base = 0; base < N; base += NT * 8) {
    uint4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = base + u * NT + t;
      if (e < N) v[u] = __ldg(reinterpret_cast<const uint4 *>(src) + e);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int e = base + u * NT + t;
      if (e < N) {
        const int r = e / KCH, kc = e - r * KCH;
        *reinterpret_cast<uint4 *>(dst + sw128_off(r, kc, ROWS)) = v[u];
      }
    }
  }
}

// max of N (a multiple of 4) registers with four independent chains (a single running maximum is a serial chain of
// N dependent FMNMX in the one warp per SM sub-partition that drains a TMEM block)
template <int N>
__device__ __forceinline__ float sa_max_tree(const float *v) {
  float m0 = v[0], m1 = v[1], m2 = v[2], m3 = v[3];
#pragma unroll
  for (int t = 4; t < N; t += 4) {
    m0 = fmaxf(m0, v[t]); m1 = fmaxf(m1, v[t + 1]); m2 = fmaxf(m2, v[t + 2]); m3 = fmaxf(m3, v[t + 3]);
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}

// EPILOGUE 2, one 128-channel block: D2 (TMEM lane = output channel, 128 columns = the rows of the tile) -> max over
// the nsample columns of each centre, + b2, relu -> out (B,C3,np) fp32 and, optionally, the point-major fp16 copy.
// The 128/NS results of a lane are consecutive floats of one out row: ONE 8/16-byte store per lane instead of a
// 4-byte store per centre (lane = channel, so every store instruction touches 32 different lines: the scalar form
// cost 32 LSU wavefronts per centre -- with 4-8 centres per tile the largest single user of the L1 data pipe in the
// wide layers, ncu l1tex__data_pipe_lsu_wavefronts).
template <int C3, int NS>
__device__ __forceinline__ void sa_pool_block(const SaFusedParams &p, uint32_t taddr, int b, int j0, int ch) {
  constexpr int NC = SA_ROWS / NS;                   // centres per tile: 2, 4 or 8
  const float bias = __ldg(p.b2 + ch);
  float res[NC];
  float m64 = -INFINITY;
#pragma unroll
  for (int cb = 0; cb < SA_ROWS; cb += 32) {
    float v[32];
    tmem_ld32(taddr + cb, v);
    if (NS <= 32) {
#pragma unroll
      for (int gI = 0; gI < 32 / NS; ++gI) res[cb / NS + gI] = fmaxf(sa_max_tree<NS>(v + gI * NS) + bias, 0.f);
    } else {                                         // NS == 64: two 32-column loads per centre
      m64 = fmaxf(m64, sa_max_tree<32>(v));
      if ((cb & 32) != 0) {
        res[cb / 64] = fmaxf(m64 + bias, 0.f);
        m64 = -INFINITY;
      }
    }
  }
  // j0 and np are multiples of NC (npoint * nsample % 128 == 0) and the tensor base is 16-byte aligned (checked at
  // launch): the NC floats start on an NC*4-byte boundary
  float *o = p.out + ((size_t)b * C3 + ch) * p.np + j0;
  if (NC == 2) {
    *reinterpret_cast<float2 *>(o) = make_float2(res[0], res[1]);
  } else {
#pragma unroll
    for (int c = 0; c < NC; c += 4) *reinterpret_cast<float4 *>(o + c) = make_float4(res[c], res[c + 1], res[c + 2], res[c + 3]);
  }
  if (p.out_pm) {                                    // lanes = consecutive channels => 64-byte coalesced stores
    __half *opm = p.out_pm + ((size_t)b * p.np + j0) * C3 + ch;
#pragma unroll
    for (int c = 0; c < NC; ++c) opm[(size_t)c * C3] = to_f16_sat(res[c]);
  }
}

// grid of a persistent launch: one CTA per resident slot, fewer when the caller asks for a minimum number of tiles
// per CTA.  Every CTA pays a fixed cost (weight staging, TMEM allocation, pipeline fill); with few tiles per CTA
// that cost dominates and a smaller grid spends less SM-time for the same work (slower alone, faster when other
// streams can use the freed SMs).
inline int sa_grid(const SaFusedParams &p, int occ) {
  int grid = kNumSMs * occ;
  if (grid > p.num_tiles) grid = p.num_tiles;
  if (p.min_tiles > 0) grid = max(1, min(grid, (p.num_tiles + p.min_tiles - 1) / p.min_tiles));
  return grid;
}

// in-line form (sa_inline.cu); returns SPC_ERR_UNSUPPORTED (error text set) when no kernel matches the widths
int launch_sa_inline(const SaFusedParams &p, int C1, int C2, int C3, int nsample, cudaStream_t stream);

}  // namespace spc
