// pm_linear.cu -- point-major 1x1-conv layer  Y = act(X . W^T + b)  on tcgen05 tensor cores, for the 1x1 convs left
// outside the fused set-abstraction kernel in eval mode: PointnetFPModule's SharedMLP (reference
// pointnet2_modules.py:412-421), VotingModule's conv1-3 (models/voting_module.py:34-61) and the proposal head
// (models/proposal_module.py:46-54, 73).  Round 1 ran them as ~30 cuBLASLt / CUTLASS launches plus layout and
// elementwise kernels; here each layer is ONE launch and the layer-specific tails are its epilogue.
//
//   X (M, K) fp16 point-major rows (M = B * points), optionally as a hi + lo pair (x = hi + lo);
//   W (N, K) BatchNorm-folded weights as a hi + lo fp16 pair, bias (N) fp32;  N <= 272, K % 8 == 0.
//
// Precision: fp16 carries 11 significant bits, so a single-fp16 GEMM is ~2e-4 per operand off the fp32 layer.  The
// weights -- and the hidden activations, which this kernel produces itself -- are therefore carried as fp16 PAIRS
// and the product is formed from three MMAs (hi.hi + lo.hi + hi.lo, fp32 accumulation in TMEM): ~2^-22 relative,
// i.e. fp32-grade, for 3x the tensor work of layers that are far too small to be tensor-bound.
//
// Execution: one CTA per (128-row tile, 128-channel slice of N; the voting tail takes whole rows), 6 warps: warp 0 = TMA producer (2-D tensor loads, 128-byte swizzle, K
// in chunks of 64), warp 1 = MMA issuer (one thread, tcgen05.mma kind::f16, M = 128, N = N), warps 2-5 = epilogue
// (TMEM lane = row, so a thread owns a point: channel-major stores are coalesced across the warp and the voting
// tail's per-point L2 norm is a register reduction).  Two- to three-stage mbarrier pipeline between producer and
// issuer; the CTA's weight slice streams through shared memory once (L2-resident: <= 0.6 MB in total).
#include <cuda.h>
#include <cuda_fp16.h>

#include <mutex>

#include "common.cuh"
#include "ptx.cuh"

namespace spc {

constexpr int PL_ROWS = 128;         // rows per tile = UMMA M
constexpr int PL_KC = 64;            // K elements per pipeline chunk = one 128-byte swizzle atom
constexpr int PL_THREADS = 192;
constexpr int PL_MAX_STAGES = 4;

struct PmLinearParams {
  int M, K, N;                 // rows, input width, output width
  int NT;                      // output channels per CTA (grid.y tiles of the N dimension; the vote tail takes all of N)
  int has_lo;                  // X comes as a hi + lo pair
  int stages;
  int tiles_per_cta;           // row tiles one CTA works through (>= 1); the accumulator is double-buffered when it fits
  int resident;                // the CTA's whole weight slice stays in shared memory (loaded with its first tile)
  int mode;
  int n;                       // points per scene (channel-major outputs)
  const float *bias;           // (N)
  __half *Y_hi, *Y_lo;         // (M, N) fp16 point-major (hidden / pm copies), Y_lo nullable
  float *out;                  // mode-dependent fp32 output
  const float *seed_cm;        // vote mode: seed features (B, D, n) fp32
  const float *seed_xyz;       // vote mode: (B, n, 3)
  float *vote_xyz;             // vote mode: (B, n, 3)
};

__global__ void __launch_bounds__(PL_THREADS, 1)
pm_linear_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                 const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                 const PmLinearParams p) {
  extern __shared__ __align__(128) uint8_t pl_smem_raw[];
  uint8_t *smem = pl_smem_raw + ((1024u - (s2u(pl_smem_raw) & 1023u)) & 1023u);   // swizzle atoms: 1024-byte aligned
  __shared__ __align__(8) uint64_t full[PL_MAX_STAGES], empty[PL_MAX_STAGES], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_smem;
  __shared__ float s_bias[288];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // this CTA's slice of the output channels: [n_off, n_off + Nt) of N, staged as Nr (multiple of 16) weight rows
  const int n_off = blockIdx.y * p.NT;
  const int Nt = min(p.NT, p.N - n_off);
  // every CTA stages round16(NT) weight rows, whatever its own Nt: the TMA box size is baked into the tensor map,
  // rows beyond N arrive as zeros and the columns they produce are never stored
  const int Nr = (p.NT + 15) / 16 * 16;
  const int N1 = Nr > 256 ? 256 : Nr, N2 = Nr - N1;    // UMMA N of the main part and of the remainder (0 or 16)
  const int A_BYTES = PL_ROWS * 128;
  const int B_BYTES = Nr * 128;
  // A pipeline stage holds one K chunk of X (hi [+ lo]) and, unless the weights are RESIDENT, the matching chunk of the
  // weight slice (hi + lo).  Resident (chosen by the host when a CTA works through several row tiles and the whole
  // slice fits next to >= 2 stages of X): the K chunks of W are loaded once, with the first tile, into their own
  // region in front of the stages, and every later tile only streams X -- half the bytes per tile for the 128-wide
  // layers, which are bound by what one SM can pull out of L2.
  const int A_STAGE = A_BYTES * (1 + p.has_lo);
  const int W_CHUNK = 2 * B_BYTES;
  const int STAGE_BYTES = p.resident ? A_STAGE : A_STAGE + W_CHUNK;
  const int KCH = (p.K + PL_KC - 1) / PL_KC;           // a partial last chunk is zero-filled by TMA (both operands)
  uint8_t *stage0 = smem + (p.resident ? (size_t)KCH * W_CHUNK : 0);
  // A CTA works through up to tiles_per_cta consecutive row tiles of its channel slice.  With more than one the
  // accumulator is double-buffered in TMEM (2 x 128 or 2 x 256 columns; the 272-wide vote tail has one buffer), so
  // the epilogue of tile i overlaps the loads and MMAs of tile i + 1, and the setup (barriers, TMEM allocation, bias)
  // is paid once: a CTA's life per tile drops from setup + load + MMA + epilogue to max(load, epilogue).
  const int num_row_tiles = (p.M + PL_ROWS - 1) / PL_ROWS;
  const int tile0 = blockIdx.x * p.tiles_per_cta;
  const int ntile = min(p.tiles_per_cta, num_row_tiles - tile0);
  const int BUFC = Nr > 128 ? 256 : 128;               // accumulator columns per buffer
  const int NBUF = (ntile > 1 && Nr <= 256) ? 2 : 1;
  const uint32_t tmem_cols = Nr > 256 ? 512u : (uint32_t)(NBUF * BUFC);

  if (tid == 0) {
    for (int s = 0; s < p.stages; ++s) { mbarrier_init(&full[s], 1); mbarrier_init(&empty[s], 1); }
    for (int u = 0; u < 2; ++u) { mbarrier_init(&acc_full[u], 1); mbarrier_init(&acc_empty[u], 128); }
    fence_mbarrier_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_smem, tmem_cols);
  for (int e = tid; e < 288; e += PL_THREADS) s_bias[e] = e < Nt ? __ldg(p.bias + n_off + e) : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (warp == 0) {
    // =============================== TMA PRODUCER (one thread) =====================================
    if (lane == 0) {
      const int BR = Nr > 256 ? Nr / 2 : Nr;                  // weight rows per TMA box (<= 256)
      for (int i = 0, g = 0; i < ntile; ++i) {
        const int row0 = (tile0 + i) * PL_ROWS;
        for (int c = 0; c < KCH; ++c, ++g) {                  // g: chunk counter over all tiles (the stage ring goes on)
          const int s = g % p.stages;
          if (g >= p.stages) mbarrier_wait(&empty[s], (unsigned)((g / p.stages - 1) & 1));
          uint8_t *st = stage0 + (size_t)s * STAGE_BYTES;
          const bool load_w = !p.resident || i == 0;
          mbarrier_arrive_expect_tx(&full[s], (unsigned)(A_STAGE + (load_w ? W_CHUNK : 0)));
          tma_load_2d(st, &tmA_hi, c * PL_KC, row0, &full[s]);
          if (p.has_lo) tma_load_2d(st + A_BYTES, &tmA_lo, c * PL_KC, row0, &full[s]);
          if (load_w) {
            uint8_t *b = p.resident ? smem + (size_t)c * W_CHUNK : st + A_STAGE;
            for (int r = 0; r < Nr; r += BR) {
              tma_load_2d(b + (size_t)r * 128, &tmB_hi, c * PL_KC, n_off + r, &full[s]);
              tma_load_2d(b + B_BYTES + (size_t)r * 128, &tmB_lo, c * PL_KC, n_off + r, &full[s]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA ISSUER (one thread) =======================================
    if (lane == 0) {
      const uint32_t idesc1 = make_idesc_f16(PL_ROWS, N1), idesc2 = make_idesc_f16(PL_ROWS, 16);
      for (int i = 0, g = 0; i < ntile; ++i) {
      const int buf = i % NBUF;
      const uint32_t tacc = tmem_base + (uint32_t)(buf * BUFC);
      if (i >= NBUF) {                                        // the epilogue has drained this buffer (tile i - NBUF)
        mbarrier_wait(&acc_empty[buf], (unsigned)((i / NBUF - 1) & 1));
        tc_fence_after();
      }
      for (int c = 0; c < KCH; ++c, ++g) {
        const int s = g % p.stages;
        mbarrier_wait(&full[s], (unsigned)((g / p.stages) & 1));
        tc_fence_after();
        const uint32_t aH = s2u(stage0 + (size_t)s * STAGE_BYTES);
        const uint32_t aL = aH + A_BYTES;
        const uint32_t bH = p.resident ? s2u(smem + (size_t)c * W_CHUNK) : aH + A_STAGE;
        const uint32_t bL = bH + B_BYTES;
#pragma unroll
        for (int kk = 0; kk < PL_KC / 16; ++kk) {
          const uint32_t ko = kk * 32;                        // 16 fp16 = 32 bytes inside the 128-byte atom
          const uint32_t acc = (c > 0 || kk > 0) ? 1u : 0u;
          umma_f16(tacc, make_smem_desc_sw128(aH + ko), make_smem_desc_sw128(bH + ko), idesc1, acc);
          umma_f16(tacc, make_smem_desc_sw128(aH + ko), make_smem_desc_sw128(bL + ko), idesc1, 1u);
          if (p.has_lo) umma_f16(tacc, make_smem_desc_sw128(aL + ko), make_smem_desc_sw128(bH + ko), idesc1, 1u);
          if (N2) {
            const uint32_t off = (uint32_t)N1 * 128u;         // weight rows N1.. : 1024-byte aligned (N1 % 8 == 0)
            umma_f16(tacc + N1, make_smem_desc_sw128(aH + ko), make_smem_desc_sw128(bH + off + ko), idesc2, acc);
            umma_f16(tacc + N1, make_smem_desc_sw128(aH + ko), make_smem_desc_sw128(bL + off + ko), idesc2, 1u);
            if (p.has_lo)
              umma_f16(tacc + N1, make_smem_desc_sw128(aL + ko), make_smem_desc_sw128(bH + off + ko), idesc2, 1u);
          }
        }
        umma_commit(&empty[s]);                               // the stage may be refilled once these MMAs have read it
      }
      umma_commit(&acc_full[buf]);
      }
    }
  } else {
    // =============================== EPILOGUE (4 warps, TMEM lane = row = point) ===================
    const int q = warp & 3;                                   // warps 2,3,4,5 -> TMEM lane quarters 2,3,0,1
    const int r = q * 32 + lane;
    for (int i = 0; i < ntile; ++i) {
    const int buf = i % NBUF;
    const long long row = (long long)(tile0 + i) * PL_ROWS + r;
    const bool ok = row < p.M;
    mbarrier_wait(&acc_full[buf], (unsigned)((i / NBUF) & 1));
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BUFC);
    const int b = ok ? (int)(row / p.n) : 0;
    const int j = ok ? (int)(row - (long long)b * p.n) : 0;
    if (p.mode != SPC_PM_VOTE) {
      // the proposal head's last conv and the set-abstraction projection have no activation
      const bool relu = p.mode == SPC_PM_HIDDEN || p.mode == SPC_PM_OUT_CM;
      for (int c0 = 0; c0 < Nr; c0 += 32) {
        float v[32];
        tmem_ld32(taddr + c0, v);
        if (!ok) continue;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          v[i] += s_bias[c0 + i];
          if (relu) v[i] = fmaxf(v[i], 0.f);
        }
        const int ch0 = n_off + c0;                           // first output channel of this block of 32
        if (p.mode == SPC_PM_OUT_PM32) {
          float *o = p.out + row * p.N + ch0;
#pragma unroll
          for (int i = 0; i < 32; ++i) if (c0 + i < Nt) o[i] = v[i];
          continue;
        }
        if (p.mode == SPC_PM_OUT_CM) {                        // (B, N, n) fp32: lanes = consecutive points, coalesced
          float *o = p.out + ((size_t)b * p.N + ch0) * p.n + j;
#pragma unroll
          for (int i = 0; i < 32; ++i) if (c0 + i < Nt) o[(size_t)i * p.n] = v[i];
        }
        // fp16 pair, point-major (the next layer's X): 64 bytes per 32 channels and array
        uint32_t hw[16], lw[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          __half h0, l0, h1, l1;
          split_f16(v[2 * i], h0, l0);
          split_f16(v[2 * i + 1], h1, l1);
          hw[i] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
          lw[i] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
        }
        // per 8-channel chunk: a slice of n_tile channels (a multiple of 16, so Nt is one too) can end halfway
        // through a block of 32
        uint4 *yh = reinterpret_cast<uint4 *>(p.Y_hi + row * p.N + ch0);
        uint4 *yl = p.Y_lo ? reinterpret_cast<uint4 *>(p.Y_lo + row * p.N + ch0) : nullptr;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (c0 + 8 * i + 8 > Nt) continue;
          yh[i] = make_uint4(hw[4 * i], hw[4 * i + 1], hw[4 * i + 2], hw[4 * i + 3]);
          if (yl) yl[i] = make_uint4(lw[4 * i], lw[4 * i + 1], lw[4 * i + 2], lw[4 * i + 3]);
        }
      }
    } else {
      // ---- voting tail (models/voting_module.py:52-61 + models/SpaCapNet.py:66-67), vote_factor 1 ----
      //   net = D + b;  v = seed_feat + net[0:D];  vote_xyz = seed_xyz + net[D:D+3];  out = v / ||v||_2
      // (the caller moves the three xyz-offset rows of conv3 behind the D feature rows, so that the feature channels
      // start at TMEM column 0 and pack into aligned 16-byte stores)
      // pass 1: the squared norm; pass 2: re-read the accumulators and write the normalised features
      const int D = p.N - 3;
      const float *sf = p.seed_cm + (size_t)b * D * p.n + j;
      float ss = 0.f;
      for (int c0 = 0; c0 < D; c0 += 32) {
        float v[32];
        tmem_ld32(taddr + c0, v);
        if (!ok) continue;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float f = __ldg(sf + (size_t)(c0 + i) * p.n) + (v[i] + s_bias[c0 + i]);
          ss = fmaf(f, f, ss);
        }
      }
      {
        float v[32];
        tmem_ld32(taddr + D, v);                              // columns D .. D+2: the xyz offsets
        if (ok) {
          const float *sx = p.seed_xyz + row * 3;
          float *vx = p.vote_xyz + row * 3;
          vx[0] = __ldg(sx + 0) + (v[0] + s_bias[D + 0]);
          vx[1] = __ldg(sx + 1) + (v[1] + s_bias[D + 1]);
          vx[2] = __ldg(sx + 2) + (v[2] + s_bias[D + 2]);
        }
      }
      const float inv = 1.0f / sqrtf(ss);
      float *o = p.out + (size_t)b * D * p.n + j;
      for (int c0 = 0; c0 < D; c0 += 32) {
        float v[32];
        tmem_ld32(taddr + c0, v);
        if (!ok) continue;
        uint32_t hw[16], lw[16];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          v[i] = (__ldg(sf + (size_t)(c0 + i) * p.n) + (v[i] + s_bias[c0 + i])) * inv;
          o[(size_t)(c0 + i) * p.n] = v[i];
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          __half h0, l0, h1, l1;
          split_f16(v[2 * i], h0, l0);
          split_f16(v[2 * i + 1], h1, l1);
          hw[i] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
          lw[i] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
        }
        uint4 *yh = reinterpret_cast<uint4 *>(p.Y_hi + row * D + c0);
#pragma unroll
        for (int i = 0; i < 4; ++i) yh[i] = make_uint4(hw[4 * i], hw[4 * i + 1], hw[4 * i + 2], hw[4 * i + 3]);
        if (p.Y_lo) {
          uint4 *yl = reinterpret_cast<uint4 *>(p.Y_lo + row * D + c0);
#pragma unroll
          for (int i = 0; i < 4; ++i) yl[i] = make_uint4(lw[4 * i], lw[4 * i + 1], lw[4 * i + 2], lw[4 * i + 3]);
        }
      }
    }
    tc_fence_before();
    mbarrier_arrive(&acc_empty[buf]);
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ---- host side --------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_tiled() {
  static std::mutex m;
  static PFN_encodeTiled fn = nullptr;
  std::lock_guard<std::mutex> lock(m);
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// (rows, K) fp16 row-major tensor, boxes of (64 x box_rows), 128-byte swizzle, rows beyond the tensor read as zero
static int make_map(CUtensorMap *tm, const void *base, long long rows, int K, int box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) { set_error("pm_linear: cuTensorMapEncodeTiled is not available"); return SPC_ERR_CUDA; }
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  const cuuint32_t box[2] = {(cuuint32_t)PL_KC, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("pm_linear: cuTensorMapEncodeTiled failed (%d)", (int)r); return SPC_ERR_CUDA; }
  return SPC_OK;
}

}  // namespace spc

using namespace spc;

extern "C" int spc_pm_linear(const void *X_hi, const void *X_lo, int M, int K, const void *W_hi, const void *W_lo,
                             const float *bias, int N, int mode, int points_per_scene, void *Y_hi, void *Y_lo,
                             float *out, const float *seed_cm, const float *seed_xyz, float *vote_xyz,
                             int n_tile, int tiles_per_cta, void *stream_) {
  // rows are K * 2 bytes apart and TMA needs 16-byte strides; K need not be a multiple of the 64-element chunk
  SPC_CHECK_ARG(M >= 0 && K >= 8 && K % 8 == 0 && K <= 4096, "pm_linear: K=%d must be a multiple of 8", K);
  SPC_CHECK_ARG(N >= 1 && N <= 272, "pm_linear: N=%d out of range (1..272)", N);
  SPC_CHECK_ARG(mode == SPC_PM_HIDDEN || mode == SPC_PM_OUT_CM || mode == SPC_PM_OUT_PM32 || mode == SPC_PM_VOTE ||
                    mode == SPC_PM_LINEAR,
                "pm_linear: unknown mode %d", mode);
  if (M == 0) return SPC_OK;
  SPC_CHECK_ARG(X_hi && W_hi && W_lo && bias, "pm_linear: null pointer");
  SPC_CHECK_ARG(points_per_scene >= 1 && M % points_per_scene == 0, "pm_linear: M=%d is not a multiple of the points "
                "per scene (%d)", M, points_per_scene);
  if (mode == SPC_PM_HIDDEN || mode == SPC_PM_OUT_CM || mode == SPC_PM_LINEAR) SPC_CHECK_ARG(Y_hi && N % 32 == 0, "pm_linear: hidden / channel-"
                "major layers need Y_hi and N %% 32 == 0 (N=%d)", N);
  if (mode == SPC_PM_OUT_CM || mode == SPC_PM_OUT_PM32) SPC_CHECK_ARG(out != nullptr, "pm_linear: missing fp32 output");
  if (mode == SPC_PM_VOTE) SPC_CHECK_ARG(out && Y_hi && seed_cm && seed_xyz && vote_xyz && N > 3 && (N - 3) % 32 == 0,
                "pm_linear: vote mode needs out, Y_hi, seed_cm, seed_xyz, vote_xyz and (N - 3) %% 32 == 0");
  PmLinearParams p;
  p.M = M; p.K = K; p.N = N;
  // the N dimension is tiled over grid.y in slices of n_tile channels (default 128: twice the CTAs for N = 256, half
  // the weight bytes each CTA streams -- the lowest latency for a layer that runs alone; one slice per row tile
  // loads X once and holds an SM for less time in total, which is what a saturated pipeline wants); the vote tail
  // needs whole rows for its L2 norm and takes all of N
  SPC_CHECK_ARG(n_tile >= 0 && n_tile % 16 == 0, "pm_linear: n_tile=%d must be 0 or a multiple of 16", n_tile);
  SPC_CHECK_ARG(tiles_per_cta >= 0 && tiles_per_cta <= 1024, "pm_linear: tiles_per_cta=%d out of range", tiles_per_cta);
  p.tiles_per_cta = tiles_per_cta > 0 ? tiles_per_cta : 1;
  const int slice = n_tile > 0 ? n_tile : 128;
  p.NT = (mode == SPC_PM_VOTE || N <= slice) ? N : slice;
  const int n_tiles = (N + p.NT - 1) / p.NT;
  const int Nr = ((p.NT < N ? p.NT : N) + 15) / 16 * 16;      // weight rows staged per CTA
  p.has_lo = X_lo != nullptr;
  p.mode = mode; p.n = points_per_scene; p.bias = bias;
  p.Y_hi = (__half *)Y_hi; p.Y_lo = (__half *)Y_lo; p.out = out;
  p.seed_cm = seed_cm; p.seed_xyz = seed_xyz; p.vote_xyz = vote_xyz;
  const int kch = (K + PL_KC - 1) / PL_KC;
  const int a_stage = PL_ROWS * 128 * (1 + p.has_lo), w_chunk = 2 * Nr * 128;
  const int budget = 220 * 1024;
  const int row_tiles = ceil_div(M, PL_ROWS);
  const int tiles_here = p.tiles_per_cta < row_tiles ? p.tiles_per_cta : row_tiles;
  p.resident = tiles_here > 1 && (long long)kch * w_chunk + 2LL * a_stage <= budget;
  const int stage_bytes = p.resident ? a_stage : a_stage + w_chunk;
  const int fixed_bytes = p.resident ? kch * w_chunk : 0;
  int stages = (budget - fixed_bytes) / stage_bytes;
  if (stages > PL_MAX_STAGES) stages = PL_MAX_STAGES;
  if (stages > kch * tiles_here) stages = kch * tiles_here;    // the stage ring runs on across a CTA's tiles
  SPC_CHECK_ARG(stages >= 1, "pm_linear: a pipeline stage of %d bytes does not fit in shared memory", stage_bytes);
  p.stages = stages;
  CUtensorMap tA_hi, tA_lo, tB_hi, tB_lo;
  int rc;
  if ((rc = make_map(&tA_hi, X_hi, M, K, PL_ROWS)) != SPC_OK) return rc;
  if ((rc = make_map(&tA_lo, X_lo ? X_lo : X_hi, M, K, PL_ROWS)) != SPC_OK) return rc;
  const int BR = Nr > 256 ? Nr / 2 : Nr;
  if ((rc = make_map(&tB_hi, W_hi, N, K, BR)) != SPC_OK) return rc;
  if ((rc = make_map(&tB_lo, W_lo, N, K, BR)) != SPC_OK) return rc;
  const size_t smem = (size_t)fixed_bytes + (size_t)stages * stage_bytes + 1024;
  SPC_CUDA(cudaFuncSetAttribute(pm_linear_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  pm_linear_kernel<<<dim3(ceil_div(ceil_div(M, PL_ROWS), p.tiles_per_cta), n_tiles), PL_THREADS, smem, (cudaStream_t)stream_>>>(tA_hi, tA_lo, tB_hi,
                                                                                                      tB_lo, p);
  SPC_LAUNCH_CHECK("pm_linear_kernel");
  return SPC_OK;
}
