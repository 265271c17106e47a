// sa_inline.cu -- fused set-abstraction forward, IN-LINE form (few raw input channels: SA1 of the backbone,
// reference pointnet2_modules.py:244-271 with mlp = [Cf, 64, 64, 128]): grouping + relative-xyz normalisation +
// three [1x1 conv + folded BN + ReLU] + max-pool over nsample in one warp-specialised kernel with ALL THREE convs on
// tcgen05 tensor cores.
//
// Rounds 1-2a evaluated layer 0 (3+Cf -> C1) with FFMAs in the gather stage: 256-512 FMAs and 8 x 16-byte stores per
// (centre, neighbour) row, a third of all warp instructions of the SA1 launch (ncu source view).  Here the gather
// stage only writes the ROW OF INPUTS and layer 0 becomes one more K = 16..64 UMMA.  To keep layer 0 at fp32 accuracy
// (it sees differences of nearby coordinates), inputs and weights are split in fp16 (hi, lo) pairs and three products
// are accumulated in fp32 by the tensor core:
//     a.w ~= a_hi.w_hi + a_lo.w_hi + a_hi.w_lo            (the dropped a_lo.w_lo term is 2^-22 relative)
// K layout: one 16-element K step per group of four inputs e = 4g .. 4g+3 (NV = 3 + Cf inputs, zero beyond NV),
//   A0 row  : [ hi0 lo0 hi1 lo1 hi2 lo2 hi3 lo3 | hi0 hi1 hi2 hi3 s s 0 0 ]      s = 1 in group 0, else 0
//   W0' row : [ wh0 wh0 wh1 wh1 wh2 wh2 wh3 wh3 | wl0 wl1 wl2 wl3 bh bl 0 0 ]    (bias in group 0 only)
// Every slot position is a compile-time constant, so a gather thread packs a K step in registers and writes it with
// two conflict-free 16-byte stores (a first version wrote 2-byte elements at run-time positions: 4-way bank conflicts,
// a third of the kernel's shared-memory store wavefronts).  The folded bias rides along on the two constant ones, so
// the layer-0 epilogue is TMEM -> relu -> fp16 -> H1 with no arithmetic.  Four groups = 16 inputs (Cf <= 13) fit the
// 64-element swizzle atom.  What the kernel is bound by now (L1 data pipe, then the TMEM read rate of the epilogues):
// profiles/r2_sa_fused_limits.md.
//
// Pipeline per 128-row tile k (a row = one (centre, neighbour) pair; all hand-offs are mbarriers):
//   warps 0-3   GATHER      idx, xyz, centre, features -> A0[k & 1]                       (thread = row)
//   warp  16    MMA ISSUER  one thread: MMA0(k)  D0 = A0 . W0'^T     (M 128, N C1, K 16..64)
//                                       MMA1(k-1) D1 = H1 . W1'^T     (M 128, N C2, K C1)
//                                       MMA2(k-2) D2 = W2' . H2^T     (M 128 channels, N 128 rows, K C2), per 128 channels
//   warps 4-7   EPILOGUE 0  D0 -> relu -> fp16 -> H1                                       (thread = row = TMEM lane)
//   warps 8-11  EPILOGUE 1  D1 + b1 -> relu -> fp16 -> H2
//   warps 12-15 EPILOGUE 2  D2 -> max over the nsample columns of a centre, + b2, relu -> out (thread = channel)
// Every stage works on a different tile at any time, so single-buffered H1 / H2 / D0 / D1 are enough (the UMMAs
// take ~0.1 us, the epilogues ~1 us); A0 is double-buffered and the gather issues a tile's loads one iteration before
// it consumes them.  TMEM: D0 (C1) + D1 (C2) + D2 (128 per block) columns; the SA1 widths
// (64, 64, 128) need 256 columns and 97 KB of shared memory, so two CTAs share an SM.
#include "sa_common.cuh"

namespace spc {

constexpr int SAI_THREADS = 17 * 32;
constexpr int SAI_GATHER_WARPS = 4;

template <int C1, int C2, int C3, int OCC>
struct SaInlineSmem {
  static constexpr int W0_BYTES = C1 * 128;                   // (C1, 64) fp16: one swizzle atom of K
  static constexpr int W1_BYTES = C2 * C1 * 2;
  static constexpr int W2_BYTES = C3 * C2 * 2;
  static constexpr int A0_BYTES = SA_ROWS * 128;              // (128, 64) fp16
  static constexpr int H1_BYTES = SA_ROWS * C1 * 2;
  static constexpr int H2_BYTES = SA_ROWS * C2 * 2;
  static constexpr int OFF_W0 = 0;
  static constexpr int OFF_W1 = OFF_W0 + W0_BYTES;
  static constexpr int OFF_W2 = OFF_W1 + W1_BYTES;
  static constexpr int OFF_A0 = OFF_W2 + W2_BYTES;            // 2 stages
  static constexpr int OFF_H1 = OFF_A0 + 2 * A0_BYTES;
  static constexpr int OFF_H2 = OFF_H1 + H1_BYTES;
  static constexpr int OFF_B1 = OFF_H2 + H2_BYTES;            // C2 floats
  static constexpr int TOTAL = OFF_B1 + C2 * 4;
  static constexpr int TMEM_D1 = C1;
  static constexpr int TMEM_D2 = C1 + C2;
  static constexpr int D2_STAGES = OCC == 2 ? 1 : 2;
  static constexpr int TMEM_COLS = OCC == 2 ? 256 : 512;
};

template <int C1, int C2, int C3, int NS, int OCC>
__global__ void __launch_bounds__(SAI_THREADS, OCC) sa_inline_kernel(const SaFusedParams p) {
  using L = SaInlineSmem<C1, C2, C3, OCC>;
  constexpr int D2S = L::D2_STAGES;
  constexpr int NB = C3 / 128;                       // 128-channel output blocks per tile
  static_assert(C1 + C2 + D2S * SA_ROWS <= L::TMEM_COLS, "TMEM budget");
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (s2u(smem_raw) & 1023u)) & 1023u);   // swizzle atoms start on 1024-byte boundaries
  __shared__ __align__(8) uint64_t a0_full[2], a0_empty[2], d0_full, d0_empty, h1_full, h1_empty, d1_full, d1_empty,
      h2_full, h2_empty, d2_full[2], d2_empty[2];
  __shared__ uint32_t tmem_base_smem;
  __shared__ float s_xyz[SAI_GATHER_WARPS][96];      // per-warp scratch of the cooperative xyz gather

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  uint8_t *sW0 = smem + L::OFF_W0, *sW1 = smem + L::OFF_W1, *sW2 = smem + L::OFF_W2, *sA0 = smem + L::OFF_A0,
          *sH1 = smem + L::OFF_H1, *sH2 = smem + L::OFF_H2;
  float *sB1 = reinterpret_cast<float *>(smem + L::OFF_B1);
  const int NV = 3 + p.Cf;                           // inputs per row
  const int nk0 = (NV + 3) >> 2;                     // K steps of MMA0 = groups of four inputs

  // ---- one-time setup ---------------------------------------------------------------------------
  if (warp == 8) tmem_alloc(&tmem_base_smem, L::TMEM_COLS);
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      mbarrier_init(&a0_full[s], SAI_GATHER_WARPS * 32);
      mbarrier_init(&a0_empty[s], 1);
      mbarrier_init(&d2_full[s], 1);
      mbarrier_init(&d2_empty[s], 128);
    }
    mbarrier_init(&d0_full, 1);
    mbarrier_init(&d0_empty, 128);
    mbarrier_init(&h1_full, 128);
    mbarrier_init(&h1_empty, 1);
    mbarrier_init(&d1_full, 1);
    mbarrier_init(&d1_empty, 128);
    mbarrier_init(&h2_full, 128);
    mbarrier_init(&h2_empty, 1);
    fence_mbarrier_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp >= SAI_GATHER_WARPS) {
    constexpr int NT = SAI_THREADS - SAI_GATHER_WARPS * 32;   // 416 staging threads
    const int t = tid - SAI_GATHER_WARPS * 32;
    // W0' image: one 16-byte chunk (half a K step of one channel) per iteration; K steps >= nk0 are never read
    for (int e = t; e < C1 * 2 * nk0; e += NT) {
      const int c = e / (2 * nk0), ch = e - c * 2 * nk0, g = ch >> 1;
      const float *wrow = p.W0 + (size_t)c * NV;
      float w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) w[u] = 4 * g + u < NV ? __ldg(wrow + 4 * g + u) : 0.f;
      uint32_t o[4];
      if ((ch & 1) == 0) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint32_t hi = __half_as_ushort(to_f16_sat(w[u]));
          o[u] = hi | (hi << 16);
        }
      } else {
        __half lo[4], hi;
#pragma unroll
        for (int u = 0; u < 4; ++u) split_f16(w[u], hi, lo[u]);
        o[0] = (uint32_t)__half_as_ushort(lo[0]) | ((uint32_t)__half_as_ushort(lo[1]) << 16);
        o[1] = (uint32_t)__half_as_ushort(lo[2]) | ((uint32_t)__half_as_ushort(lo[3]) << 16);
        __half bh = __float2half_rn(0.f), bl = bh;
        if (g == 0) split_f16(__ldg(p.b0 + c), bh, bl);
        o[2] = (uint32_t)__half_as_ushort(bh) | ((uint32_t)__half_as_ushort(bl) << 16);
        o[3] = 0u;
      }
      *reinterpret_cast<uint4 *>(sW0 + sw128_off(c, ch, C1)) = make_uint4(o[0], o[1], o[2], o[3]);
    }
    sa_stage_weights<C2, C1 / 8, NT>(sW1, p.W1, t);
    sa_stage_weights<C3, C2 / 8, NT>(sW2, p.W2, t);
    for (int e = t; e < C2; e += NT) sB1[e] = __ldg(p.b1 + e);
    fence_proxy_async_smem();
    named_bar_sync<1, NT>();
  }
  const uint32_t tmem_base = tmem_base_smem;
  const int tiles_per_scene = (p.np * NS) / SA_ROWS;
  const int t0 = (int)blockIdx.x, dt = (int)gridDim.x;
  const int nt = (p.num_tiles - t0 + dt - 1) / dt;   // tiles of this CTA

  if (warp < SAI_GATHER_WARPS) {
    // =============================== GATHER: inputs of row r -> A0[s] ============================
    // The loads of a row are ISSUED a tile ahead (raw values stay in registers) and only consumed when the tile is
    // written: with the loads issued and consumed inside one iteration every gather warp had a single tile of loads
    // in flight and the whole CTA ran at one L2/HBM round trip per tile.
    // The 12 bytes of a point are fetched COOPERATIVELY: the warp's 32 rows are 96 words, lane l loads words l, 32+l,
    // 64+l (three lanes share a point => ~11 lines per load instead of 32) and the words go back to their rows
    // through a 384-byte per-warp scratch (3 conflict-free stores + 3 stride-3 loads): 39 L1 wavefronts per warp and
    // tile instead of 96.
    const int r = tid;
    const float inv_r = 1.0f / p.radius;
    const int Cf = p.Cf;
    constexpr int NF = 8;                      // features fetched with the coordinates; more (Cf > 8) are read late
    float *scratch = s_xyz[warp];
    float rawp[3], rawc[3], rawf[NF];
    auto issue = [&](int tile, int i) {
      const int b = sa_tile_scene(p, tile, tiles_per_scene);
      const int j = ((tile - b * tiles_per_scene) * SA_ROWS + r) / NS;
      const float *pb = p.xyz + (size_t)b * p.n * 3;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int w = q * 32 + lane, wr = (w * 43) >> 7;                  // w / 3 for w < 128
        rawp[q] = __ldg(pb + 3 * __shfl_sync(0xffffffffu, i, wr) + (w - 3 * wr));
      }
      const float *cc = p.new_xyz + ((size_t)b * p.np + j) * 3;
      rawc[0] = __ldg(cc); rawc[1] = __ldg(cc + 1); rawc[2] = __ldg(cc + 2);
      const float *fp = p.feat + (size_t)b * Cf * p.n + i;
#pragma unroll
      for (int u = 0; u < NF; ++u) rawf[u] = u < Cf ? __ldg(fp + (size_t)u * p.n) : 0.f;
    };
    // one K step: inputs x0..x3 -> [hi0 lo0 .. hi3 lo3 | hi0 hi1 hi2 hi3 s s 0 0]
    auto put_group = [&](uint8_t *row, int g, float x0, float x1, float x2, float x3) {
      const float x[4] = {x0, x1, x2, x3};
      uint32_t a[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float lo = x[u] - __half2float(to_f16_sat(x[u]));
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(a[u]) : "f"(lo), "f"(x[u]));      // {upper: lo, lower: hi}
      }
      uint32_t h01, h23;
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h01) : "f"(x[1]), "f"(x[0]));
      asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(h23) : "f"(x[3]), "f"(x[2]));
      *reinterpret_cast<uint4 *>(row + sw128_off(r, 2 * g, SA_ROWS)) = make_uint4(a[0], a[1], a[2], a[3]);
      *reinterpret_cast<uint4 *>(row + sw128_off(r, 2 * g + 1, SA_ROWS)) = make_uint4(h01, h23, g == 0 ? 0x3C003C00u : 0u, 0u);
    };
    int i_cur = __ldg(p.idx + (long long)t0 * SA_ROWS + r);
    issue(t0, i_cur);
    int i_nxt = nt > 1 ? __ldg(p.idx + (long long)(t0 + dt) * SA_ROWS + r) : 0;
    for (int k = 0; k < nt; ++k) {
      const int s = k & 1, n = k >> 1;
      const int tile = t0 + k * dt;
      // finish tile k (its loads were issued an iteration ago): words back to their rows, then
      // (p - c) / r as a multiplication by 1/r -- a 1-ulp difference to the reference's true division is far below
      // the fp16 rounding of h1
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 3; ++q) scratch[q * 32 + lane] = rawp[q];
      __syncwarp();
      float v[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = (scratch[3 * lane + c] - rawc[c]) * inv_r;
      // A0 is double-buffered and MMA0 takes ~50 ns, so this wait is practically never taken: the row is written
      // first and the next tile's loads are issued afterwards (the raw registers are free by then)
      mbarrier_wait_relaxed(&a0_empty[s], (unsigned)(n & 1) ^ 1u);              // MMA0(k-2) has consumed A0[s]
      uint8_t *row = sA0 + s * L::A0_BYTES;
      put_group(row, 0, v[0], v[1], v[2], rawf[0]);
      if (nk0 > 1) put_group(row, 1, rawf[1], rawf[2], rawf[3], rawf[4]);
      if (nk0 > 2) {
        float x[5];
#pragma unroll
        for (int u = 0; u < 5; ++u) x[u] = 0.f;
        if (NV > 3 + NF) {                       // features 8..12 (inputs 11..15) are read late
          const int b = sa_tile_scene(p, tile, tiles_per_scene);
          const float *fp = p.feat + (size_t)b * Cf * p.n + i_cur;
#pragma unroll
          for (int u = 0; u < 5; ++u) x[u] = NF + u < Cf ? __ldg(fp + (size_t)(NF + u) * p.n) : 0.f;
        }
        put_group(row, 2, rawf[5], rawf[6], rawf[7], x[0]);
        if (nk0 > 3) put_group(row, 3, x[1], x[2], x[3], x[4]);
      }
      fence_proxy_async_smem();
      mbarrier_arrive(&a0_full[s]);
      if (k + 1 < nt) {
        i_cur = i_nxt;
        issue(tile + dt, i_cur);
        if (k + 2 < nt) i_nxt = __ldg(p.idx + (long long)(tile + 2 * dt) * SA_ROWS + r);
      }
    }
  } else if (warp == 16) {
    // =============================== MMA ISSUER (one thread) =====================================
    if (lane == 0) {
      constexpr uint32_t IDESC0 = make_idesc_f16(128, C1);
      constexpr uint32_t IDESC1 = make_idesc_f16(128, C2);
      constexpr uint32_t IDESC2 = make_idesc_f16(128, SA_ROWS);
      const uint32_t aA0 = s2u(sA0), aH1 = s2u(sH1), aH2 = s2u(sH2), aW0 = s2u(sW0), aW1 = s2u(sW1), aW2 = s2u(sW2);
      for (int k = 0; k < nt + 2; ++k) {
        if (k < nt) {                                            // D0 = A0[s] . W0'^T
          const int s = k & 1, n = k >> 1;
          mbarrier_wait(&a0_full[s], (unsigned)(n & 1));
          mbarrier_wait(&d0_empty, (unsigned)(k & 1) ^ 1u);      // epilogue 0 has drained D0 (tile k-1)
          tc_fence_after();
          for (int kk = 0; kk < nk0; ++kk) {
            const uint64_t da = make_smem_desc_sw128(aA0 + s * L::A0_BYTES + sw128_kstep(kk, SA_ROWS));
            const uint64_t db = make_smem_desc_sw128(aW0 + sw128_kstep(kk, C1));
            umma_f16(tmem_base, da, db, IDESC0, kk > 0);
          }
          umma_commit(&d0_full);
          umma_commit(&a0_empty[s]);
        }
        if (k >= 1 && k <= nt) {                                 // D1 = H1 . W1'^T for tile k-1
          const int kt = k - 1;
          mbarrier_wait(&h1_full, (unsigned)(kt & 1));
          mbarrier_wait(&d1_empty, (unsigned)(kt & 1) ^ 1u);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < C1 / 16; ++kk) {
            const uint64_t da = make_smem_desc_sw128(aH1 + sw128_kstep(kk, SA_ROWS));
            const uint64_t db = make_smem_desc_sw128(aW1 + sw128_kstep(kk, C2));
            umma_f16(tmem_base + L::TMEM_D1, da, db, IDESC1, kk > 0);
          }
          umma_commit(&d1_full);
          umma_commit(&h1_empty);
        }
        if (k >= 2) {                                            // D2[u] = W2'[h] . H2^T for tile k-2
          const int kt = k - 2;
          mbarrier_wait(&h2_full, (unsigned)(kt & 1));
          tc_fence_after();
#pragma unroll
          for (int h = 0; h < NB; ++h) {
            const int u = kt * NB + h, st = u % D2S, nu = u / D2S;
            mbarrier_wait(&d2_empty[st], (unsigned)(nu & 1) ^ 1u);
            tc_fence_after();
#pragma unroll
            for (int kk = 0; kk < C2 / 16; ++kk) {
              const uint64_t da = make_smem_desc_sw128(aW2 + h * 128 * 128 + sw128_kstep(kk, C3));
              const uint64_t db = make_smem_desc_sw128(aH2 + sw128_kstep(kk, SA_ROWS));
              umma_f16(tmem_base + L::TMEM_D2 + st * SA_ROWS, da, db, IDESC2, kk > 0);
            }
            umma_commit(&d2_full[st]);
          }
          umma_commit(&h2_empty);
        }
      }
    }
  } else if (warp < 8) {
    // =============================== EPILOGUE 0: D0 -> H1 ========================================
    const int q = warp & 3;
    const int r = q * 32 + lane;
    for (int k = 0; k < nt; ++k) {
      mbarrier_wait_relaxed(&d0_full, (unsigned)(k & 1));
      mbarrier_wait_relaxed(&h1_empty, (unsigned)(k & 1) ^ 1u);       // MMA1(k-1) has consumed H1
      tc_fence_after();
#pragma unroll
      for (int col0 = 0; col0 < C1; col0 += 32) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + col0, v);
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          uint4 o;
          o.x = pack_relu_f16x2(v[c8 * 8 + 0], v[c8 * 8 + 1]);
          o.y = pack_relu_f16x2(v[c8 * 8 + 2], v[c8 * 8 + 3]);
          o.z = pack_relu_f16x2(v[c8 * 8 + 4], v[c8 * 8 + 5]);
          o.w = pack_relu_f16x2(v[c8 * 8 + 6], v[c8 * 8 + 7]);
          *reinterpret_cast<uint4 *>(sH1 + sw128_off(r, (col0 >> 3) + c8, SA_ROWS)) = o;
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbarrier_arrive(&h1_full);
      mbarrier_arrive(&d0_empty);
    }
  } else if (warp < 12) {
    // =============================== EPILOGUE 1: D1 + b1 -> H2 ===================================
    const int q = warp & 3;
    const int r = q * 32 + lane;
    for (int k = 0; k < nt; ++k) {
      mbarrier_wait_relaxed(&d1_full, (unsigned)(k & 1));
      mbarrier_wait_relaxed(&h2_empty, (unsigned)(k & 1) ^ 1u);       // MMA2(k-1) has consumed H2
      tc_fence_after();
#pragma unroll
      for (int col0 = 0; col0 < C2; col0 += 32) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + L::TMEM_D1 + col0, v);
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          const float4 ba = *reinterpret_cast<const float4 *>(sB1 + col0 + c8 * 8);
          const float4 bb = *reinterpret_cast<const float4 *>(sB1 + col0 + c8 * 8 + 4);
          uint4 o;
          o.x = pack_relu_f16x2(v[c8 * 8 + 0] + ba.x, v[c8 * 8 + 1] + ba.y);
          o.y = pack_relu_f16x2(v[c8 * 8 + 2] + ba.z, v[c8 * 8 + 3] + ba.w);
          o.z = pack_relu_f16x2(v[c8 * 8 + 4] + bb.x, v[c8 * 8 + 5] + bb.y);
          o.w = pack_relu_f16x2(v[c8 * 8 + 6] + bb.z, v[c8 * 8 + 7] + bb.w);
          *reinterpret_cast<uint4 *>(sH2 + sw128_off(r, (col0 >> 3) + c8, SA_ROWS)) = o;
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbarrier_arrive(&h2_full);
      mbarrier_arrive(&d1_empty);
    }
  } else {
    // =============================== EPILOGUE 2: D2 -> max-pool -> out ==========================
    const int q = warp & 3;
    for (int k = 0; k < nt; ++k) {
      const int tile = t0 + k * dt;
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

template <int C1, int C2, int C3, int NS, int OCC>
static int launch_sa_inline_occ(const SaFusedParams &p, cudaStream_t stream) {
  using L = SaInlineSmem<C1, C2, C3, OCC>;
  auto kern = sa_inline_kernel<C1, C2, C3, NS, OCC>;
  const int smem = L::TOTAL + 1024;                  // + slack for the 1024-byte alignment
  SPC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  kern<<<sa_grid(p, OCC), SAI_THREADS, smem, stream>>>(p);
  SPC_LAUNCH_CHECK("sa_inline_kernel");
  return SPC_OK;
}

template <int C1, int C2, int C3, int NS>
static int launch_sa_inline_widths(const SaFusedParams &p, cudaStream_t stream) {
  // two CTAs per SM when 256 TMEM columns and half of the shared memory are enough (the SA1 widths)
  if constexpr (C1 + C2 + SA_ROWS <= 256 && 2 * (SaInlineSmem<C1, C2, C3, 2>::TOTAL + 2048) <= 227 * 1024)
    return launch_sa_inline_occ<C1, C2, C3, NS, 2>(p, stream);
  else
    return launch_sa_inline_occ<C1, C2, C3, NS, 1>(p, stream);
}

int launch_sa_inline(const SaFusedParams &p, int C1, int C2, int C3, int nsample, cudaStream_t stream) {
#define SAI_TRY(c1, c2, c3, ns) \
  if (C1 == c1 && C2 == c2 && C3 == c3 && nsample == ns) return launch_sa_inline_widths<c1, c2, c3, ns>(p, stream);
  SAI_TRY(64, 64, 128, 64)      // SA1
  SAI_TRY(64, 64, 128, 32)
  SAI_TRY(64, 64, 128, 16)
  SAI_TRY(128, 128, 256, 64)
  SAI_TRY(128, 128, 256, 32)
  SAI_TRY(128, 128, 256, 16)
  SAI_TRY(128, 128, 128, 64)
  SAI_TRY(128, 128, 128, 32)
  SAI_TRY(128, 128, 128, 16)
#undef SAI_TRY
  set_error("sa_fused: no kernel for widths (%d,%d,%d) nsample=%d", C1, C2, C3, nsample);
  return SPC_ERR_UNSUPPORTED;
}

}  // namespace spc
