// sa_fused.cu -- fused set-abstraction forward (eval mode): grouping + relative-xyz
// normalisation + shared MLP (3 x [1x1 conv + folded BN + ReLU]) + max-pool over nsample in ONE
// warp-specialised kernel, the wide 1x1 convs on tcgen05 tensor cores with TMEM accumulators
// (sm_100a).  This file: the C-ABI entry points and the PROJECTED form (SA2-SA4, vote aggregation, multiview
// SA1); the IN-LINE form (few raw input channels: SA1) lives in sa_inline.cu, shared pieces in sa_common.cuh.
//
// Replaces, for PointnetSAModuleVotes.forward in eval mode (reference pointnet2_modules.py:244-271):
//   QueryAndGroup's two group_points launches + sub + div + cat (pointnet2_utils.py:351-362),
//   SharedMLP = 3 x (cuDNN conv, cuDNN BN, ReLU) (pytorch_utils.py:11-36) and F.max_pool2d --
// i.e. ~14 kernels that each stream a (B, C, npoint, nsample) activation through HBM
// (SURVEY 2.4: ~270 MB/scene unfused vs ~8 MB compulsory).
//
// Algorithm (per tile of 128 rows, a row = one (centre, neighbour) pair):
//   layer 0  h1 = relu(W0' . [ (p_i - c_j)/r , f_i ] + b0)
//            projected form: conv0 is linear and its feature part only depends on the POINT, not on
//            the pair, so it is hoisted out of the grouping: G[i] = W0f' . f_i is one plain GEMM per
//            layer over the n points (npoint*nsample/n = 4..16x fewer MACs) and the kernel evaluates
//            h1 = relu(G[idx] + W0x' . (p_i - c_j)/r + b0) in the gather stage -- the xyz term stays in
//            fp32 (it is a difference of nearby points; G is fp16).
//            in-line form (sa_inline.cu): one more UMMA on fp16 (hi, lo) split inputs, fp32-grade.
//   layer 1  D1[128 rows x C2]  = H1[128 x C1] . W1'^T             tcgen05.mma, M=128, N=C2
//            h2 = relu(D1 + b1) -> fp16 -> shared memory (thread per row, TMEM lane = row)
//   layer 2  D2[C3 x 128 rows]  = W2'[C3 x C2] . H2^T              tcgen05.mma, TRANSPOSED so that a
//            TMEM lane is an output CHANNEL and the 128 columns are the rows of the tile: the
//            max over the nsample neighbours of a centre is then a register-only reduction.
//   out[b, c, j] = relu(max_k D2[c, j*ns+k] + b2[c])   (ReLU and +b commute with max)
// BN (eval) is folded on the host: W' = diag(gamma/sqrt(var+eps)) W, b = beta - mean*scale.
//
// Execution: a persistent grid of warp-specialised CTAs (8 producer warps, 4 + 4 epilogue warps, 1 MMA-issuing
// warp, mbarrier hand-offs, H1 / H2 / D1 double-buffered), one CTA per SM (up to 224 KB of shared memory).
//
// Shared-memory operands: canonical UMMA K-major layout with 128-byte swizzle (a row = 128
// contiguous bytes per 64-element K atom, chunk c of row r at position c ^ (r & 7)).  With it both
// a warp writing one whole row (row-wise gather) and 8 lanes writing the same chunk of 8
// consecutive rows (epilogue, lane = row) are bank-conflict free, and no TMA descriptor is needed
// for gathered data.
#include "sa_common.cuh"

namespace spc {

// Projected layer 0: ONE WARP PER ROW PAIR so that the gather of a 2*C1-byte G row (fp16) is a coalesced request
// (2 L1 wavefronts per row instead of 16+ with lane = row).  Lane = 8 consecutive channels (one 16-byte chunk) of
// one row: one 16-byte load, 8 x (3 FMA + add + relu) with this lane's xyz weights / bias in registers, one 16-byte
// store into the swizzled H1.  A warp owns 16 rows of the tile (they share one centre: nsample >= 16) and handles
// them as two batches of 8 rows (SaProjBatch: raw G chunks + coordinates in registers), one after the other.
// Measured and rejected (round 2, B200, SA2 shape, tools/time_sa_layers.py): keeping two batches in flight across
// tiles (needs setmaxnreg 128/64 to fit; 42 us vs 37 us) and a cp.async gather that parks the raw rows in H1 and
// converts them in place (41 us): once the output stores were vectorised the kernel sits at ~80 % of the rate at
// which the epilogues can read their accumulators out of TMEM (4 B x 128 x (C2 + C3) per tile at ~64 B/clk per SM),
// and neither hiding more gather latency nor spending more L1 wavefronts on it helps.
template <int C1>
struct SaProjBatch {
  static constexpr int LPR = C1 / 8;                 // lanes per row (8 fp16 = 16 bytes each)
  static constexpr int RPI = 32 / LPR;               // rows per warp-wide load
  static constexpr int NPASS = 16 / RPI;             // passes per tile and warp
  static constexpr int HB = NPASS / 2 > 0 ? NPASS / 2 : 1;   // passes per batch
  static constexpr int ROWS = HB * RPI;              // rows per batch (8)
  uint4 g[HB];
  // the batch's 8 points are 24 words: lane w < 24 holds word w (row w / 3, component w % 3) and the matching
  // component of the centre -- one load instruction with ~8 lines instead of three per pass, one register instead
  // of three per pass; the rows get their (p - c)/r back by shuffle when the batch is computed
  float pw, cw;
};

template <int C1, int NS>
__device__ __forceinline__ void sa_proj_issue(const SaFusedParams &p, int tile, int half, int warp, int lane, int my_idx,
                                              int tiles_per_scene, SaProjBatch<C1> &q) {
  using Q = SaProjBatch<C1>;
  const int kc = lane % Q::LPR, sub = lane / Q::LPR;
  const int b = sa_tile_scene(p, tile, tiles_per_scene);
  const int j = ((tile - b * tiles_per_scene) * SA_ROWS + warp * 16) / NS;
  const __half *Gb = p.G + (size_t)b * p.n * C1 + 8 * kc;
  const int wl = lane < 3 * Q::ROWS ? lane : 0;      // lanes >= 24 repeat word 0 (never read)
  const int wr = (wl * 11) >> 5, wc = wl - 3 * wr;   // wl / 3 for wl < 32
  q.cw = __ldg(p.new_xyz + ((size_t)b * p.np + j) * 3 + wc);
  q.pw = __ldg(p.xyz + ((size_t)b * p.n + __shfl_sync(0xffffffffu, my_idx, half * Q::ROWS + wr)) * 3 + wc);
#pragma unroll
  for (int t = 0; t < Q::HB; ++t) {
    const int i = __shfl_sync(0xffffffffu, my_idx, (half * Q::HB + t) * Q::RPI + sub);   // lanes 0..15 hold the 16 indices
    q.g[t] = __ldg(reinterpret_cast<const uint4 *>(Gb + (size_t)i * C1));
  }
}

template <int C1>
__device__ __forceinline__ void sa_proj_finish(const SaProjBatch<C1> &q, int half, int warp, int lane, float inv_r,
                                               const float (&wx)[8][3], const float (&wb)[8], uint8_t *sH1) {
  using Q = SaProjBatch<C1>;
  const int kc = lane % Q::LPR, sub = lane / Q::LPR;
  // (p - c) / r as a multiplication by 1/r: this path is the fp16 one (rtol 1e-2), a 1-ulp difference to the
  // reference's true division is irrelevant here
  const float rel = (q.pw - q.cw) * inv_r;
#pragma unroll
  for (int t = 0; t < Q::HB; ++t) {
    const int rb = t * Q::RPI + sub;                 // row within the batch
    const int r = warp * 16 + half * Q::ROWS + rb;
    const float rx = __shfl_sync(0xffffffffu, rel, 3 * rb);
    const float ry = __shfl_sync(0xffffffffu, rel, 3 * rb + 1);
    const float rz = __shfl_sync(0xffffffffu, rel, 3 * rb + 2);
    const uint32_t gw[4] = {q.g[t].x, q.g[t].y, q.g[t].z, q.g[t].w};
    uint32_t ow[4];
#pragma unroll
    for (int c2 = 0; c2 < 4; ++c2) {
      const float2 g01 = __half22float2(*reinterpret_cast<const __half2 *>(&gw[c2]));                // fp16 -> f32
      const float v0 = fmaf(wx[2 * c2][2], rz, fmaf(wx[2 * c2][1], ry, fmaf(wx[2 * c2][0], rx, g01.x + wb[2 * c2])));
      const float v1 = fmaf(wx[2 * c2 + 1][2], rz, fmaf(wx[2 * c2 + 1][1], ry, fmaf(wx[2 * c2 + 1][0], rx, g01.y + wb[2 * c2 + 1])));
      ow[c2] = pack_relu_f16x2(v0, v1);
    }
    *reinterpret_cast<uint4 *>(sH1 + sw128_off(r, kc, SA_ROWS)) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
  }
}

// ================================================================================================
// Warp-specialised, double-buffered kernel.
//
// A first, serial version ran gather -> MMA1 -> epilogue1 -> MMA2 -> epilogue2 back to back in every
// CTA (tensor pipe 4-14 % active, ncu).  Here the five stages of consecutive tiles overlap:
//   warps 0-7   PRODUCERS   gather + layer 0            -> H1[s]      (s = tile parity)
//   warp  16    MMA ISSUER  one thread: MMA1(k) then MMA2(k-1)        (tcgen05, D in TMEM)
//   warps 8-11  EPILOGUE 1  D1[s] -> relu(+b1) -> fp16  -> H2[s]
//   warps 12-15 EPILOGUE 2  D2[u&1] -> max over nsample, +b2, relu -> out   (u = 128-channel unit)
// Hand-offs are mbarriers: "full" barriers are arrived on by the producing threads (after a
// generic->async proxy fence, because UMMA reads shared memory through the async proxy) or by
// tcgen05.commit; "empty" barriers by the consuming threads / by tcgen05.commit of the MMA that
// read the buffer.  TMEM: D1 double-buffered (2*C2 columns) + a 2-deep ring of 128-column D2
// blocks = at most 512 columns.  Shared memory for the widest layer (128,128,256): W1 32K + W2 64K
// + 2*H1 64K + 2*H2 64K = 224 KB.
// ================================================================================================
constexpr int SAP_PROD_WARPS = 8;
constexpr int SAP_THREADS = 17 * 32;

template <int C1, int C2, int C3>
struct SaPipeSmem {
  static constexpr int W1_BYTES = C2 * C1 * 2;
  static constexpr int W2_BYTES = C3 * C2 * 2;
  static constexpr int H1_BYTES = SA_ROWS * C1 * 2;
  static constexpr int H2_BYTES = SA_ROWS * C2 * 2;
  static constexpr int OFF_W1 = 0;
  static constexpr int OFF_W2 = OFF_W1 + W1_BYTES;
  static constexpr int OFF_H1 = OFF_W2 + W2_BYTES;            // 2 stages
  static constexpr int OFF_H2 = OFF_H1 + 2 * H1_BYTES;        // 2 stages
  static constexpr int OFF_B1 = OFF_H2 + 2 * H2_BYTES;        // C2 floats
  static constexpr int TOTAL = OFF_B1 + C2 * 4;
  static constexpr int TMEM_D2 = 2 * C2;                      // first column of the 2-deep D2 ring
  static constexpr int D2_STAGES = 2;
  static constexpr int TMEM_COLS = 512;
};

template <int C1, int C2, int C3, int NS>
__global__ void __launch_bounds__(SAP_THREADS, 1) sa_fused_pipe_kernel(const SaFusedParams p) {
  using L = SaPipeSmem<C1, C2, C3>;
  constexpr int D2S = L::D2_STAGES;
  constexpr int NB = C3 / 128;                       // 128-channel output blocks per tile
  extern __shared__ __align__(128) uint8_t smem_raw[];
  // the 128B-swizzle atoms must start on 1024-byte boundaries
  uint8_t *smem = smem_raw + ((1024u - (s2u(smem_raw) & 1023u)) & 1023u);
  // barrier groups, 2 stages each
  __shared__ __align__(8) uint64_t h1_full[2], h1_empty[2], d1_full[2], d1_empty[2], h2_full[2], h2_empty[2],
      d2_full[2], d2_empty[2];
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  uint8_t *sW1 = smem + L::OFF_W1, *sW2 = smem + L::OFF_W2, *sH1 = smem + L::OFF_H1, *sH2 = smem + L::OFF_H2;
  float *sB1 = reinterpret_cast<float *>(smem + L::OFF_B1);

  // ---- one-time setup ---------------------------------------------------------------------------
  // Only the barriers and the TMEM allocation are needed by everybody.  The 24-96 KB of folded weights are staged
  // by the NON-producer warps (all loads of a pass issued before the first store: one L2 round trip per pass
  // instead of one per element) while the producers already gather and compute their first tile; ncu had the
  // serial staging + its barrier at ~20 % of the SA2 kernel's samples and more for the smaller layers.
  if (warp == 8) tmem_alloc(&tmem_base_smem, L::TMEM_COLS);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbarrier_init(&h1_full[s], SAP_PROD_WARPS * 32);
      mbarrier_init(&h1_empty[s], 1);
      mbarrier_init(&d1_full[s], 1);
      mbarrier_init(&d1_empty[s], 128);
      mbarrier_init(&h2_full[s], 128);
      mbarrier_init(&h2_empty[s], 1);
      mbarrier_init(&d2_full[s], 1);
      mbarrier_init(&d2_empty[s], 128);
    }
    fence_mbarrier_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp >= SAP_PROD_WARPS) {
    constexpr int NT = SAP_THREADS - SAP_PROD_WARPS * 32;     // 288 staging threads
    const int t = tid - SAP_PROD_WARPS * 32;
    sa_stage_weights<C2, C1 / 8, NT>(sW1, p.W1, t);
    sa_stage_weights<C3, C2 / 8, NT>(sW2, p.W2, t);
    for (int e = t; e < C2; e += NT) sB1[e] = __ldg(p.b1 + e);
    fence_proxy_async_smem();
    named_bar_sync<1, NT>();
  }
  const uint32_t tmem_base = tmem_base_smem;
  const int tiles_per_scene = (p.np * NS) / SA_ROWS;
  const int nt = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA

  if (warp < SAP_PROD_WARPS) {
    // =============================== PRODUCERS ===================================================
    // warp per row group: lanes 0..15 carry the neighbour indices of the warp's 16 rows; every
    // lane keeps the xyz weights and bias of its 8 channels in registers
    constexpr int LPR = C1 / 8;
    float wx[8][3], wb[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int ch = (lane % LPR) * 8 + c;
      wx[c][0] = __ldg(p.W0 + ch * 3 + 0);
      wx[c][1] = __ldg(p.W0 + ch * 3 + 1);
      wx[c][2] = __ldg(p.W0 + ch * 3 + 2);
      wb[c] = __ldg(p.b0 + ch);
    }
    auto load_idx = [&](int tile) {
      return lane < 16 ? __ldg(p.idx + (long long)tile * SA_ROWS + warp * 16 + lane) : 0;
    };
    const int t0 = (int)blockIdx.x, dt = (int)gridDim.x;
    const float inv_r = 1.0f / p.radius;
    int idx_nxt = load_idx(t0);
    for (int k = 0; k < nt; ++k) {
      const int s = k & 1, n = k >> 1;
      const int tile = t0 + k * dt;
      uint8_t *h1 = sH1 + s * L::H1_BYTES;
      const int idx_cur = idx_nxt;
      if (k + 1 < nt) idx_nxt = load_idx(tile + dt);                           // a tile ahead
      SaProjBatch<C1> q;
      sa_proj_issue<C1, NS>(p, tile, 0, warp, lane, idx_cur, tiles_per_scene, q);
      mbarrier_wait_relaxed(&h1_empty[s], (unsigned)(n & 1) ^ 1u);             // MMA1(k-2) has consumed H1[s]
      sa_proj_finish<C1>(q, 0, warp, lane, inv_r, wx, wb, h1);
      sa_proj_issue<C1, NS>(p, tile, 1, warp, lane, idx_cur, tiles_per_scene, q);
      sa_proj_finish<C1>(q, 1, warp, lane, inv_r, wx, wb, h1);
      fence_proxy_async_smem();
      mbarrier_arrive(&h1_full[s]);
    }
  } else if (warp == 16) {
    // =============================== MMA ISSUER (one thread) =====================================
    if (lane == 0) {
      constexpr uint32_t IDESC1 = make_idesc_f16(128, C2);
      constexpr uint32_t IDESC2 = make_idesc_f16(128, SA_ROWS);
      const uint32_t aH1 = s2u(sH1), aH2 = s2u(sH2), aW1 = s2u(sW1), aW2 = s2u(sW2);
      for (int k = 0; k <= nt; ++k) {
        if (k < nt) {                                            // D1[s] = H1[s] . W1'^T
          const int s = k & 1, n = k >> 1;
          mbarrier_wait(&h1_full[s], (unsigned)(n & 1));
          mbarrier_wait(&d1_empty[s], (unsigned)(n & 1) ^ 1u);   // epilogue 1 has drained D1[s]
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < C1 / 16; ++kk) {
            const uint64_t da = make_smem_desc_sw128(aH1 + s * L::H1_BYTES + sw128_kstep(kk, SA_ROWS));
            const uint64_t db = make_smem_desc_sw128(aW1 + sw128_kstep(kk, C2));
            umma_f16(tmem_base + s * C2, da, db, IDESC1, kk > 0);
          }
          umma_commit(&d1_full[s]);
          umma_commit(&h1_empty[s]);
        }
        if (k >= 1) {                                            // D2[u] = W2'[h] . H2[s]^T for tile k-1
          const int kt = k - 1, s = kt & 1, n = kt >> 1;
          mbarrier_wait(&h2_full[s], (unsigned)(n & 1));
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < NB; ++h) {
            const int u = kt * NB + h, st = u % D2S, nu = u / D2S;
            mbarrier_wait(&d2_empty[st], (unsigned)(nu & 1) ^ 1u);
            tc_fence_after();
#pragma unroll
            for (int kk = 0; kk < C2 / 16; ++kk) {
              const uint64_t da = make_smem_desc_sw128(aW2 + h * 128 * 128 + sw128_kstep(kk, C3));
              const uint64_t db = make_smem_desc_sw128(aH2 + s * L::H2_BYTES + sw128_kstep(kk, SA_ROWS));
              umma_f16(tmem_base + L::TMEM_D2 + st * SA_ROWS, da, db, IDESC2, kk > 0);
            }
            umma_commit(&d2_full[st]);
          }
          umma_commit(&h2_empty[s]);
        }
      }
    }
  } else if (warp < 12) {
    // =============================== EPILOGUE 1: D1 -> H2 ========================================
    const int q = warp & 3;
    const int r = q * 32 + lane;
    for (int k = 0; k < nt; ++k) {
      const int s = k & 1, n = k >> 1;
      mbarrier_wait_relaxed(&d1_full[s], (unsigned)(n & 1));
      mbarrier_wait_relaxed(&h2_empty[s], (unsigned)(n & 1) ^ 1u);   // MMA2(k-2) has consumed H2[s]
      tc_fence_after();
      uint8_t *h2 = sH2 + s * L::H2_BYTES;
#pragma unroll
      for (int col0 = 0; col0 < C2; col0 += 32) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + s * C2 + col0, v);
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          const float4 ba = *reinterpret_cast<const float4 *>(sB1 + col0 + c8 * 8);
          const float4 bb = *reinterpret_cast<const float4 *>(sB1 + col0 + c8 * 8 + 4);
          uint4 o;
          o.x = pack_relu_f16x2(v[c8 * 8 + 0] + ba.x, v[c8 * 8 + 1] + ba.y);
          o.y = pack_relu_f16x2(v[c8 * 8 + 2] + ba.z, v[c8 * 8 + 3] + ba.w);
          o.z = pack_relu_f16x2(v[c8 * 8 + 4] + bb.x, v[c8 * 8 + 5] + bb.y);
          o.w = pack_relu_f16x2(v[c8 * 8 + 6] + bb.z, v[c8 * 8 + 7] + bb.w);
          *reinterpret_cast<uint4 *>(h2 + sw128_off(r, (col0 >> 3) + c8, SA_ROWS)) = o;
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbarrier_arrive(&h2_full[s]);
      mbarrier_arrive(&d1_empty[s]);
    }
  } else {
    // =============================== EPILOGUE 2: D2 -> max-pool -> out ==========================
    const int q = warp & 3;
    for (int k = 0; k < nt; ++k) {
      const int tile = (int)blockIdx.x + k * (int)gridDim.x;
      const int b = sa_tile_scene(p, tile, tiles_per_scene);
      const int j0 = ((tile - b * tiles_per_scene) * SA_ROWS) / NS;      // first centre of the tile
#pragma unroll
      for (int h = 0; h < NB; ++h) {
        const int u = k * NB + h, st = u % D2S, nu = u / D2S;
        mbarrier_wait_relaxed(&d2_full[st], (unsigned)(nu & 1));
        tc_fence_after();
        sa_pool_block<C3, NS>(p, tmem_base + ((uint32_t)(q * 32) << 16) + L::TMEM_D2 + st * SA_ROWS, b, j0,
                              h * 128 + q * 32 + lane);
        tc_fence_before();
        mbarrier_arrive(&d2_empty[st]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, L::TMEM_COLS);
  }
}

template <int C1, int C2, int C3, int NS>
static int launch_sa_pipe(const SaFusedParams &p, cudaStream_t stream) {
  using L = SaPipeSmem<C1, C2, C3>;
  auto kern = sa_fused_pipe_kernel<C1, C2, C3, NS>;
  const int smem = L::TOTAL + 1024;                  // + slack for the 1024-byte alignment
  SPC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  kern<<<sa_grid(p, 1), SAP_THREADS, smem, stream>>>(p);
  SPC_LAUNCH_CHECK("sa_fused_pipe_kernel");
  return SPC_OK;
}

}  // namespace spc

using namespace spc;

extern "C" int spc_sa_fused_forward(const float *xyz, const float *new_xyz, const int32_t *idx,
                                    const void *G_f16, const float *feat, const float *W0,
                                    const float *b0, int Cf, float radius, const void *W1_f16,
                                    const float *b1, const void *W2_f16, const float *b2, int B, int n,
                                    int npoint, int nsample, int C1, int C2, int C3, float *out,
                                    void *out_pm_f16, void *stream_) {
  return spc_sa_fused_forward_ex(xyz, new_xyz, idx, G_f16, feat, W0, b0, nullptr, nullptr, Cf, radius, W1_f16, b1,
                                 W2_f16, b2, B, n, npoint, nsample, C1, C2, C3, out, out_pm_f16, 0, stream_);
}

extern "C" int spc_sa_fused_forward_ex(const float *xyz, const float *new_xyz, const int32_t *idx,
                                       const void *G_f16, const float *feat, const float *W0,
                                       const float *b0, const float *W0_host, const float *b0_host, int Cf,
                                       float radius, const void *W1_f16, const float *b1, const void *W2_f16,
                                       const float *b2, int B, int n, int npoint, int nsample, int C1, int C2,
                                       int C3, float *out, void *out_pm_f16, int min_tiles_per_cta,
                                       void *stream_) {
  SPC_CHECK_ARG(B >= 0 && n >= 1 && npoint >= 0 && nsample >= 1, "sa_fused: bad sizes");
  SPC_CHECK_ARG(min_tiles_per_cta >= 0 && min_tiles_per_cta <= 4096, "sa_fused: min_tiles_per_cta %d out of range",
                min_tiles_per_cta);
  if (B == 0 || npoint == 0) return SPC_OK;
  SPC_CHECK_ARG(xyz && new_xyz && idx && W0 && b0 && W1_f16 && b1 && W2_f16 && b2 && out,
                "sa_fused: null pointer");
  SPC_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 15) == 0, "sa_fused: out must be 16-byte aligned");
  const bool proj = G_f16 != nullptr;
  SPC_CHECK_ARG(proj ? (Cf == 0) : (feat || Cf == 0), "sa_fused: missing layer-0 operands");
  const long long rows = (long long)B * npoint * nsample;
  if (rows % SA_ROWS != 0 || ((long long)npoint * nsample) % SA_ROWS != 0) {
    set_error("sa_fused: npoint*nsample=%lld is not a multiple of %d", (long long)npoint * nsample, SA_ROWS);
    return SPC_ERR_UNSUPPORTED;
  }
  if (!proj && (Cf < 0 || Cf > SA_MAX_K0 - 3)) {
    set_error("sa_fused: inline mode supports at most %d raw feature channels (got %d)", SA_MAX_K0 - 3, Cf);
    return SPC_ERR_UNSUPPORTED;
  }
  SaFusedParams p;
  p.xyz = xyz; p.new_xyz = new_xyz; p.idx = idx; p.G = (const __half *)G_f16; p.feat = feat;
  p.W0 = W0; p.b0 = b0; p.Cf = Cf; p.radius = radius;
  p.W1 = (const __half *)W1_f16; p.b1 = b1; p.W2 = (const __half *)W2_f16; p.b2 = b2;
  p.out = out; p.out_pm = (__half *)out_pm_f16; p.B = B; p.n = n; p.np = npoint; p.ns = nsample;
  p.num_tiles = (int)(rows / SA_ROWS);
  p.min_tiles = min_tiles_per_cta;
  (void)W0_host; (void)b0_host;                      // accepted and ignored: layer 0 of the in-line form is a UMMA now
  {
    // tile -> scene without a division in the kernels: magic = ceil(2^32 / tps) is exact while tile * (magic * tps
    // - 2^32) < 2^32, i.e. certainly for tile < 2^32 / tps
    const unsigned long long tps = (unsigned long long)npoint * nsample / SA_ROWS;
    p.tps_magic = 0;
    if (tps >= 2 && (unsigned long long)p.num_tiles * tps < (1ull << 32))
      p.tps_magic = (unsigned)(((1ull << 32) + tps - 1) / tps);
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!proj) return launch_sa_inline(p, C1, C2, C3, nsample, stream);
#define SA_TRY(c1, c2, c3, ns) \
  if (C1 == c1 && C2 == c2 && C3 == c3 && nsample == ns) return launch_sa_pipe<c1, c2, c3, ns>(p, stream);
  SA_TRY(64, 64, 128, 64)      // SA1 (multiview)
  SA_TRY(64, 64, 128, 32)
  SA_TRY(64, 64, 128, 16)
  SA_TRY(128, 128, 256, 64)
  SA_TRY(128, 128, 256, 32)    // SA2
  SA_TRY(128, 128, 256, 16)    // SA3, SA4
  SA_TRY(128, 128, 128, 64)
  SA_TRY(128, 128, 128, 32)
  SA_TRY(128, 128, 128, 16)    // vote aggregation
#undef SA_TRY
  set_error("sa_fused: no kernel for widths (%d,%d,%d) nsample=%d", C1, C2, C3, nsample);
  return SPC_ERR_UNSUPPORTED;
}
