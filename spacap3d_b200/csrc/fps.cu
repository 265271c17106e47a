// fps.cu -- furthest point sampling as a thread-block-cluster kernel (sm_100a).
//
// Replaces furthest_point_sampling_kernel (reference sampling_gpu.cu:69-229), which runs ONE
// 512-thread block per scene and read-modify-writes a global `temp` array every round.
//
// Design (B200-first):
//  * one CLUSTER of C CTAs per scene (C = 1..16); every point's xyz and running min-distance
//    stay in REGISTERS for the whole kernel (P points per thread) -- no global traffic at all
//    inside the npoint-1 sequential rounds;
//  * per round: P fused distance/min updates per thread, a 2-instruction warp arg-max
//    (redux.sync max on the distance bits, redux.sync min on the tie-break key), one
//    __syncthreads for the CTA-level candidate table, then every CTA pushes its candidate
//    (distance, index, x, y, z) into every peer's shared memory with st.async, whose
//    completion is counted on the peer's mbarrier (no cluster barrier, no fence) -- each CTA
//    then reduces the C candidates redundantly, so the winner's coordinates are already
//    on-chip for the next round;
//  * bit-exactness with the reference's block-tree arg-max: among equal maxima the reference
//    keeps the candidate with the smallest (bit-reversed thread id, k div T), T =
//    opt_n_threads(N) (SURVEY F4).  Points are assigned to threads in exactly that order
//    ("virtual index" v = bitrev(k mod T) * Q + k div T, Q = ceil(N/T)), so "max distance, then
//    min v" reproduces the tree, and each thread's strict '>' scan reproduces the per-thread rule;
//  * the |p|^2 <= 1e-3 skip (sampling_gpu.cu:100-101, compared in double) is evaluated once at
//    load time: skipped / out-of-range slots get min-distance -1 and can never win.
#include <cooperative_groups.h>
#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "ptx.cuh"

namespace cg = cooperative_groups;

namespace spc {

constexpr int kMaxCluster = 16;

struct FpsParams {
  const float *xyz;   // (B,N,3)
  int32_t *idx;       // (B,npoint)
  float *new_xyz;     // (B,npoint,3) or nullptr
  int N, npoint;
  int T, log2T, Q;    // reference thread count, its log2, ceil(N/T)
  const int *ordered_ok;  // per scene: 1 = "FPS(xyz)[0:npoint] is provably 0..npoint-1" (or nullptr)
  int *strict_out;        // per scene (or nullptr): 1 = every pick was the strict unique maximum (culled kernels)
};

__device__ __forceinline__ int fps_v_to_k(unsigned v, int Q, int T, int log2T) {
  const unsigned r = v / (unsigned)Q;
  const unsigned q = v - r * (unsigned)Q;
  const unsigned res = log2T ? (__brev(r) >> (32 - log2T)) : 0u;
  return (int)(q * (unsigned)T + res);
}

// ---- PTX helpers: cluster address mapping, async DSMEM store -----------------------------------
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t local_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
  return r;
}
// 16-byte + 4-byte remote stores into a peer CTA's shared memory; each store signals its bytes
// on the peer's mbarrier (complete_tx), so the receiver needs no fence and no cluster barrier
// (cg::cluster_group::sync() costs a MEMBAR.ALL.GPU + L1 invalidate per round: measured 40 % of
// the kernel in the first version).
__device__ __forceinline__ void st_async_v4(uint32_t remote_addr, uint32_t a, uint32_t b, uint32_t c,
                                            uint32_t d, uint32_t remote_bar) {
  asm volatile(
      "st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::
          "r"(remote_addr),
      "r"(a), "r"(b), "r"(c), "r"(d), "r"(remote_bar)
      : "memory");
}
__device__ __forceinline__ void st_async_b32(uint32_t remote_addr, uint32_t a, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(remote_addr),
               "r"(a), "r"(remote_bar)
               : "memory");
}

// candidate record exchanged between warps / CTAs: 32 bytes, 16-byte aligned
struct __align__(16) FpsCand {
  unsigned key;   // distance bits + 1, 0 = "no valid point"
  int k;          // point index
  float x, y;
  float z;
  unsigned pad[3];
};

// XYZ_REGS: coordinates in registers (fast path); otherwise they are read from shared memory
// every round (large-N fallback, P up to 32 with 512 threads).
//
// Tie-break without a second reduction: points are laid out so that the virtual index v grows
// with (cluster rank, warp, lane, slot).  "Largest distance, then smallest v" therefore is
// "largest key, then FIRST in (rank, warp, lane, slot) order" -- one redux.max + one ballot/ffs
// per level, and the per-thread strict '>' keeps the lowest slot.
template <int P, int THREADS, bool XYZ_REGS>
__global__ void __launch_bounds__(THREADS, (THREADS <= 256 ? 2 : 1)) fps_cluster_kernel(const FpsParams p) {
  constexpr int NW = THREADS / 32;
  extern __shared__ float s_xyz[];  // [3][P][THREADS] SoA copy of this CTA's points + [P][THREADS] index
  float *sx = s_xyz, *sy = s_xyz + P * THREADS, *sz = s_xyz + 2 * P * THREADS;
  int *sk = reinterpret_cast<int *>(s_xyz + 3 * P * THREADS);
  __shared__ FpsCand w_cand[2][NW];            // per-warp candidates (double buffered)
  __shared__ FpsCand c_cand[2][kMaxCluster];   // per-CTA candidates, written by peers via DSMEM
  __shared__ __align__(8) uint64_t c_bar[2];   // "all C candidates of this buffer have landed"

  cg::cluster_group cluster = cg::this_cluster();
  const unsigned C = cluster.num_blocks();
  const unsigned rank = cluster.block_rank();
  const int scene = blockIdx.y;
  const int tid = threadIdx.x;
  const unsigned lane = tid & 31u, warp = tid >> 5;
  const float *xyz = p.xyz + (size_t)scene * p.N * 3;
  const unsigned g = rank * THREADS + tid;      // thread id within the cluster
  const unsigned v0 = g * P;                    // first virtual index owned by this thread
  const unsigned V = (unsigned)p.T * (unsigned)p.Q;

  // Verified shortcut (see fps_prefix_check_kernel): the input is an FPS-ordered prefix, so the
  // npoint sequential rounds would return 0..npoint-1.  Every CTA of the cluster reads the same
  // flag, so they all leave together.
  if (p.ordered_ok != nullptr && p.ordered_ok[scene] != 0) {
    if (g == 0 && p.strict_out) p.strict_out[scene] = 1;   // proven: every pick was a strict unique maximum
    int32_t *oidx = p.idx + (size_t)scene * p.npoint;
    for (unsigned j = g; j < (unsigned)p.npoint; j += C * THREADS) oidx[j] = (int)j;
    if (p.new_xyz) {
      float *o = p.new_xyz + (size_t)scene * p.npoint * 3;
      for (unsigned e = g; e < 3u * (unsigned)p.npoint; e += C * THREADS) o[e] = __ldg(xyz + e);
    }
    return;
  }

  float x[P], y[P], z[P], t[P];
#pragma unroll
  for (int s = 0; s < P; ++s) {
    const unsigned v = v0 + s;
    float px = 0.f, py = 0.f, pz = 0.f, pt = -1.0f;
    int k = 0;
    if (v < V) {
      k = fps_v_to_k(v, p.Q, p.T, p.log2T);
      if (k < p.N) {
        px = __ldg(xyz + 3 * k + 0);
        py = __ldg(xyz + 3 * k + 1);
        pz = __ldg(xyz + 3 * k + 2);
        const float mag = __fmaf_rn(pz, pz, __fmaf_rn(px, px, __fmul_rn(py, py)));
        pt = ((double)mag <= 1e-3) ? -1.0f : 1e10f;   // reference compares in double (F5)
      }
    }
    sx[s * THREADS + tid] = px;
    sy[s * THREADS + tid] = py;
    sz[s * THREADS + tid] = pz;
    sk[s * THREADS + tid] = k;
    if (XYZ_REGS) { x[s] = px; y[s] = py; z[s] = pz; }
    t[s] = pt;
  }
  // point 0 is always the first pick (sampling_gpu.cu:85-86) and the fallback when no valid
  // point exists (every thread reports best=-1, besti=0 => dists_i[0] == 0).
  const float p0x = __ldg(xyz + 0), p0y = __ldg(xyz + 1), p0z = __ldg(xyz + 2);
  float ox = p0x, oy = p0y, oz = p0z;
  int32_t *idx = p.idx + (size_t)scene * p.npoint;
  float *nxyz = p.new_xyz ? p.new_xyz + (size_t)scene * p.npoint * 3 : nullptr;
  // the output writer sits in the LAST warp so that the first warp (which drives the cluster
  // exchange) never lags behind
  const bool writer = (rank == 0 && tid == THREADS - 1);
  if (writer) {
    idx[0] = 0;
    if (nxyz) { nxyz[0] = ox; nxyz[1] = oy; nxyz[2] = oz; }
  }
  const unsigned tx_bytes = 20u * C;
  uint32_t r_slot0 = 0, r_slot1 = 0, r_bar0 = 0, r_bar1 = 0;   // my slot / barrier in peer `lane`
  if (C > 1) {
    if (tid == 0) {
      mbarrier_init(&c_bar[0], 1);
      mbarrier_init(&c_bar[1], 1);
      fence_mbarrier_init();
      mbarrier_arrive_expect_tx(&c_bar[0], tx_bytes);
      mbarrier_arrive_expect_tx(&c_bar[1], tx_bytes);
    }
    cluster.sync();   // peers' barriers are initialised before anyone stores into them
    if (warp == 0 && lane < C) {
      r_slot0 = mapa_cluster(s2u(&c_cand[0][rank]), lane);
      r_slot1 = mapa_cluster(s2u(&c_cand[1][rank]), lane);
      r_bar0 = mapa_cluster(s2u(&c_bar[0]), lane);
      r_bar1 = mapa_cluster(s2u(&c_bar[1]), lane);
    }
  } else {
    __syncthreads();
  }

  for (int j = 1; j < p.npoint; ++j) {
    const int buf = j & 1;
    float best = -1.0f;
    int bs = 0;
#pragma unroll
    for (int s = 0; s < P; ++s) {
      float d;
      if (XYZ_REGS) d = sqdist_ref(x[s], y[s], z[s], ox, oy, oz);
      else d = sqdist_ref(sx[s * THREADS + tid], sy[s * THREADS + tid], sz[s * THREADS + tid], ox, oy, oz);
      const float d2 = fminf(d, t[s]);
      t[s] = d2;
      if (d2 > best) { best = d2; bs = s; }   // strict '>': lowest slot (= lowest v) wins ties
    }
    // every lane fetches its own candidate (overlaps the reduction latency; no divergent chain)
    const float mx = sx[bs * THREADS + tid], my = sy[bs * THREADS + tid], mz = sz[bs * THREADS + tid];
    const int mk = sk[bs * THREADS + tid];
    // ---- warp arg-max: redux.max on the distance bits; first lane among equals wins ----------
    const unsigned key = best < 0.f ? 0u : __float_as_uint(best) + 1u;
    const unsigned wmax = __reduce_max_sync(0xffffffffu, key);
    // first lane among equals: redux.min on the lane id (26 cycles vs 66 for ballot + ffs)
    if (lane == __reduce_min_sync(0xffffffffu, key == wmax ? lane : 32u)) {
      FpsCand *e = &w_cand[buf][warp];
      *reinterpret_cast<uint4 *>(e) = make_uint4(wmax, (unsigned)mk, __float_as_uint(mx), __float_as_uint(my));
      e->z = mz;
    }
    __syncthreads();
    // ---- CTA arg-max, computed redundantly by every warp (first warp among equals wins) ------
    uint4 e4 = make_uint4(0u, 0u, 0u, 0u);
    float ez = 0.f;
    if (lane < NW) {
      e4 = *reinterpret_cast<const uint4 *>(&w_cand[buf][lane]);
      ez = w_cand[buf][lane].z;
    }
    unsigned bmax = __reduce_max_sync(0xffffffffu, e4.x);
    unsigned src = __reduce_min_sync(0xffffffffu, (lane < NW && e4.x == bmax) ? lane : 32u);
    unsigned wk = __shfl_sync(0xffffffffu, e4.y, src);
    unsigned wxb = __shfl_sync(0xffffffffu, e4.z, src);
    unsigned wyb = __shfl_sync(0xffffffffu, e4.w, src);
    float wz = __shfl_sync(0xffffffffu, ez, src);
    if (C > 1) {
      // ---- push this CTA's candidate to every CTA of the cluster; data + completion in one op --
      if (warp == 0 && lane < C) {
        const uint32_t rs = buf ? r_slot1 : r_slot0, rb = buf ? r_bar1 : r_bar0;
        st_async_v4(rs, bmax, wk, wxb, wyb, rb);
        st_async_b32(rs + 16, __float_as_uint(wz), rb);
      }
      mbarrier_wait(&c_bar[buf], (unsigned)((j - 1) >> 1) & 1u);           // u-th use of this buffer
      if (tid == 0) mbarrier_arrive_expect_tx(&c_bar[buf], tx_bytes);   // re-arm for round j+2
      e4 = make_uint4(0u, 0u, 0u, 0u);
      ez = 0.f;
      if (lane < C) {
        e4 = *reinterpret_cast<const uint4 *>(&c_cand[buf][lane]);
        ez = c_cand[buf][lane].z;
      }
      bmax = __reduce_max_sync(0xffffffffu, e4.x);
      src = __reduce_min_sync(0xffffffffu, (lane < C && e4.x == bmax) ? lane : 32u);
      wk = __shfl_sync(0xffffffffu, e4.y, src);
      wxb = __shfl_sync(0xffffffffu, e4.z, src);
      wyb = __shfl_sync(0xffffffffu, e4.w, src);
      wz = __shfl_sync(0xffffffffu, ez, src);
    }
    int old = 0;
    if (bmax == 0u) { ox = p0x; oy = p0y; oz = p0z; }
    else { ox = __uint_as_float(wxb); oy = __uint_as_float(wyb); oz = wz; old = (int)wk; }
    if (writer) {
      idx[j] = old;
      if (nxyz) { nxyz[3 * j + 0] = ox; nxyz[3 * j + 1] = oy; nxyz[3 * j + 2] = oz; }
    }
  }
  if (writer && p.strict_out) p.strict_out[scene] = 0;   // this kernel does not track ties: "unknown"
  if (C > 1) cluster.sync();  // no CTA may exit while a peer can still store into its smem
}

// ================================================================================================
// Morton sort (prepass of the bucketed sampler below): spatially compact runs of consecutive points.
// ================================================================================================
constexpr int FMS_THREADS = 1024;
constexpr int FMS_BINS = 32768;       // 32^3 cells

__device__ __forceinline__ unsigned morton_spread5(unsigned x) {   // 5 bits -> every third bit
  x = (x | (x << 8)) & 0x0000100Fu;
  x = (x | (x << 4)) & 0x000010C3u;
  x = (x | (x << 2)) & 0x00001249u;   // bits 0,3,6,9,12
  return x;
}

// Position of cell (x, y, z) of a 32^3 grid along the 3-D Hilbert curve (Skilling's transpose algorithm, 5 bits per
// axis).  Unlike the Z-order curve it has no long jumps, so a run of consecutive sorted points is always a spatially
// connected blob: bounding boxes of 64-point runs are ~1/3 tighter (10.4 instead of 15.5 buckets touched per FPS
// round on a 40 k-point room).  Any order gives the same picks; this one gives the fewest bucket visits.
__device__ __forceinline__ unsigned hilbert15(unsigned x0, unsigned x1, unsigned x2) {
  unsigned X[3] = {x0, x1, x2};
#pragma unroll
  for (unsigned Q = 16; Q > 1; Q >>= 1) {
    const unsigned P = Q - 1;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (X[i] & Q) X[0] ^= P;
      else { const unsigned t = (X[0] ^ X[i]) & P; X[0] ^= t; X[i] ^= t; }
    }
  }
  X[1] ^= X[0];
  X[2] ^= X[1];
  unsigned t = 0;
#pragma unroll
  for (unsigned Q = 16; Q > 1; Q >>= 1) if (X[2] & Q) t ^= Q - 1;
  X[0] ^= t; X[1] ^= t; X[2] ^= t;
  return (morton_spread5(X[0]) << 2) | (morton_spread5(X[1]) << 1) | morton_spread5(X[2]);
}

// one CTA per scene: bounding box -> 15-bit Hilbert cell per point -> counting sort -> perm[b][N].
// N <= FMS_THREADS * FMS_ITEMS (the culled kernel's own capacity); every thread keeps the cell codes of
// its <= 40 points in registers (two per register) between the counting and the scatter pass, and
// loads are issued eight points at a time so that the three passes are not latency-bound.
constexpr int FMS_ITEMS = 40;
constexpr int FMS_BATCH = 8;

__global__ void __launch_bounds__(FMS_THREADS) fps_morton_sort_kernel(const float *__restrict__ xyz, int N,
                                                                      int32_t *__restrict__ perm) {
  extern __shared__ int s_cnt[];                 // [FMS_BINS]
  __shared__ float s_red[6][32];
  __shared__ float s_box[6];
  __shared__ int s_part[32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float *P = xyz + (size_t)b * N * 3;
  for (int c = tid; c < FMS_BINS; c += FMS_THREADS) s_cnt[c] = 0;
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int i0 = 0; i0 < FMS_ITEMS; i0 += FMS_BATCH) {
    float v[FMS_BATCH][3];
#pragma unroll
    for (int i = 0; i < FMS_BATCH; ++i) {
      const int k = tid + (i0 + i) * FMS_THREADS;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[i][c] = k < N ? __ldg(P + 3 * k + c) : NAN;   // NaN: ignored by fmin/fmax
    }
#pragma unroll
    for (int i = 0; i < FMS_BATCH; ++i)
#pragma unroll
      for (int c = 0; c < 3; ++c) { mn[c] = fminf(mn[c], v[i][c]); mx[c] = fmaxf(mx[c], v[i][c]); }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      mn[c] = fminf(mn[c], __shfl_xor_sync(0xffffffffu, mn[c], o));
      mx[c] = fmaxf(mx[c], __shfl_xor_sync(0xffffffffu, mx[c], o));
    }
    if (lane == 0) { s_red[c][warp] = mn[c]; s_red[3 + c][warp] = mx[c]; }
  }
  __syncthreads();
  if (tid < 3) {
    float lo = s_red[tid][0], hi = s_red[3 + tid][0];
    for (int w = 1; w < FMS_THREADS / 32; ++w) { lo = fminf(lo, s_red[tid][w]); hi = fmaxf(hi, s_red[3 + tid][w]); }
    const float ext = hi - lo;
    s_box[tid] = lo;
    s_box[3 + tid] = (ext > 0.f && ext < INFINITY) ? 32.0f / ext : 0.f;
  }
  __syncthreads();
  const float bx = s_box[0], by = s_box[1], bz = s_box[2], gx = s_box[3], gy = s_box[4], gz = s_box[5];
  unsigned codes[FMS_ITEMS / 2];
#pragma unroll
  for (int i0 = 0; i0 < FMS_ITEMS; i0 += FMS_BATCH) {
    float v[FMS_BATCH][3];
#pragma unroll
    for (int i = 0; i < FMS_BATCH; ++i) {
      const int k = tid + (i0 + i) * FMS_THREADS;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[i][c] = k < N ? __ldg(P + 3 * k + c) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < FMS_BATCH; ++i) {
      const int k = tid + (i0 + i) * FMS_THREADS;
      const unsigned qx = (unsigned)min(31, max(0, (int)((v[i][0] - bx) * gx)));
      const unsigned qy = (unsigned)min(31, max(0, (int)((v[i][1] - by) * gy)));
      const unsigned qz = (unsigned)min(31, max(0, (int)((v[i][2] - bz) * gz)));
      const unsigned code = hilbert15(qx, qy, qz);
      if (k < N) atomicAdd(&s_cnt[code], 1);
      if ((i & 1) == 0) codes[(i0 + i) >> 1] = code;
      else codes[(i0 + i) >> 1] |= code << 16;
    }
  }
  __syncthreads();
  constexpr int PER = FMS_BINS / FMS_THREADS;
  const int c0 = tid * PER;
  int sum = 0;
#pragma unroll 8
  for (int c = c0; c < c0 + PER; ++c) sum += s_cnt[c];
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_part[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = s_part[lane], inc2 = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += u; }
    s_part[lane] = inc2 - v;
  }
  __syncthreads();
  int run = s_part[warp] + incl - sum;
#pragma unroll 8
  for (int c = c0; c < c0 + PER; ++c) { const int n = s_cnt[c]; s_cnt[c] = run; run += n; }
  __syncthreads();
  int32_t *out = perm + (size_t)b * N;
#pragma unroll
  for (int i = 0; i < FMS_ITEMS; ++i) {
    const int k = tid + i * FMS_THREADS;
    const unsigned code = (codes[i >> 1] >> ((i & 1) * 16)) & 0xffffu;
    if (k < N) out[atomicAdd(&s_cnt[code], 1)] = k;
  }
}

// ================================================================================================
// Bucketed sampler: ONE small CTA per scene, points parked in L2.
//
// What limits detector throughput is not how long one sampling call takes but how much of the GPU it
// holds while it runs: the kernels above keep every point of a scene on-chip, which pins 2.7-4 SMs
// per 40 k-point scene for the whole 1.3-1.5 ms (60 % of all SM time of a forward in round 1).  Yet after
// the first few dozen picks a new centre changes the min-distance of a few dozen points only.
//
// Here the Morton-sorted points live in GLOBAL memory as float4 (x, y, z, running min-distance) -- 640 KB per
// 40 k-point scene, L2-resident -- cut into buckets of BS consecutive points.  The CTA keeps per bucket, in
// shared memory (48 B): the bounding box of its selectable points and its current best candidate
// (key = min-distance bits + 1, tie-break index v, point index, coordinates).  A round is
//   1. cull   : every thread tests 2-3 buckets: can the new centre lower any min-distance in it?
//               (box distance^2 * (1 - 1e-5) >= the bucket's largest min-distance => provably not); the
//               touched buckets (a handful once ~100 centres exist) are appended to a list;
//   2. update : one warp per touched bucket loads its BS points from L2 (the only global access on the
//               round's dependency chain: ~250 cycles, the same as the DSMEM exchange of the cluster kernel),
//               updates the min-distances, stores the changed ones, and re-derives the bucket's candidate;
//   3. select : arg-max over the bucket candidates (threads scan 2-3 records each, two redux levels).
// No cluster, no DSMEM, three bar.sync per round; 256 threads and ~32 KB of shared memory, so FOUR scenes
// share an SM.  Same arithmetic as everywhere else (sqdist_ref, fminf, strict tie-break on the reference's
// virtual index), so the picks are bit-identical.
//
// Two picks per round.  The round's pick a1 (bucket A1) and the best candidate a2 of every other bucket are
// both known after step 3.  a2 is provably the next sequential pick when
//   (1) key2(A1) < key(a2), key2 = the bucket's second-largest key: a1 itself drops to distance 0 and nothing
//       else in A1 reaches a2 (keys only fall);
//   (2) a2 is the strict unique maximum outside A1 (no other bucket reaches its key, no tie inside its bucket);
//   (3) sqdist_ref(a2, a1) >= value(a2): the update with centre a1 leaves a2 unchanged;
//   (4) a2's key is above 1 (a1's key after its own update) and the call still needs two picks.
// Then the round emits both and the next one applies both centres (fminf twice: exact, so the order is free).
// On a 40 k-point room ~93 % of the rounds take two picks; a round costs a few more bucket visits but the
// fixed part (cull, three arg-max levels, barrier) is paid ~1,060 times instead of 2,047.
// ================================================================================================
constexpr unsigned FB_KEY_INIT = 0x501502F9u + 1u;      // __float_as_uint(1e10f) + 1

__device__ __forceinline__ unsigned fb_v_of_k(unsigned k, int T, int log2T, int Q) {
  const unsigned res = log2T ? (__brev(k & (unsigned)(T - 1)) >> (32 - log2T)) : 0u;
  return res * (unsigned)Q + (k >> log2T);      // T is a power of two
}

// warp per bucket: gather the Morton-sorted points into (x, y, z, t0), t0 = 1e10 or -1 for points the reference
// never selects (|p|^2 <= 1e-3, F5) and for the padding; bounding box of the selectable points.
template <int BS>
__global__ void __launch_bounds__(256) fps_bucket_build_kernel(const float *__restrict__ xyz_all,
                                                               const int32_t *__restrict__ perm_all, int N, int NB,
                                                               float4 *__restrict__ pts_all,
                                                               int32_t *__restrict__ kk_all,
                                                               float *__restrict__ boxes_all) {
  const int scene = blockIdx.y;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= NB) return;
  const float *xyz = xyz_all + (size_t)scene * N * 3;
  const int32_t *perm = perm_all + (size_t)scene * N;
  float4 *pts = pts_all + (size_t)scene * NB * BS;
  int32_t *kk = kk_all + (size_t)scene * NB * BS;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int u = 0; u < BS / 32; ++u) {
    const int q = b * BS + u * 32 + lane;
    float4 v = make_float4(0.f, 0.f, 0.f, -1.0f);
    int k = 0;
    if (q < N) {
      k = __ldg(perm + q);
      v.x = __ldg(xyz + 3 * k + 0);
      v.y = __ldg(xyz + 3 * k + 1);
      v.z = __ldg(xyz + 3 * k + 2);
      const float mag = __fmaf_rn(v.z, v.z, __fmaf_rn(v.x, v.x, __fmul_rn(v.y, v.y)));
      v.w = ((double)mag <= 1e-3) ? -1.0f : 1e10f;   // reference compares in double (F5)
      if (v.w > 0.f) {
        lo[0] = fminf(lo[0], v.x); lo[1] = fminf(lo[1], v.y); lo[2] = fminf(lo[2], v.z);
        hi[0] = fmaxf(hi[0], v.x); hi[1] = fmaxf(hi[1], v.y); hi[2] = fmaxf(hi[2], v.z);
      }
    }
    pts[q] = v;
    kk[q] = k;
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      lo[c] = fminf(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
      hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
    }
  }
  if (lane < 6) boxes_all[((size_t)scene * NB + b) * 6 + lane] = lane < 3 ? lo[lane] : hi[lane - 3];
}

// Equal keys: does point ka come before point kb in the reference's tie-break order?  Out of line: ties are rare
// and their arithmetic must not sit in every round's instruction stream.
__device__ __noinline__ bool fb_tie_before(int ka, int kb, int T, int log2T, int Q) {
  return fb_v_of_k((unsigned)ka, T, log2T, Q) < fb_v_of_k((unsigned)kb, T, log2T, Q);
}
// Several lanes hold the maximal key: lane of the smallest virtual index.
__device__ __noinline__ unsigned fb_resolve_tie(bool hit, int k, unsigned lane, int T, int log2T, int Q) {
  const unsigned v = hit ? fb_v_of_k((unsigned)k, T, log2T, Q) : 0xffffffffu;
  const unsigned vmin = __reduce_min_sync(0xffffffffu, v);
  return __reduce_min_sync(0xffffffffu, (hit && v == vmin) ? lane : 32u);
}

__host__ __device__ constexpr size_t fb_smem_per_scene(int W, int S) {
  // kxyz 16 B + box 24 B per table entry (W * 32 * S entries), per-warp candidates (best and runner-up, double
  // buffered), per-warp queues
  return (size_t)W * 32 * S * 40 + (size_t)W * 128 + (((size_t)W * 32 * S * 2 + 15) & ~(size_t)15);
}

// W warps work on one scene, G scenes share a CTA (W * G * 32 threads; the scenes of a CTA only share the SM, they
// synchronise on separate named barriers).  Bucket b belongs to warp b % W, lane (b / W) % 32, slot (b / W) / 32:
// every lane keeps the candidate key of its <= S buckets in registers, so the cull test and the arg-max read no
// shared memory but the boxes, and spatial neighbours (consecutive buckets) land in different warps.
template <int BS, int W, int G, int S>
__global__ void __launch_bounds__(W * G * 32, G == 1 ? (W <= 8 ? 4 : (W <= 16 ? 2 : 1)) : 1)
fps_bucket_kernel(const FpsParams p, float4 *pts_all, const int32_t *__restrict__ kk_all,
                  const float *__restrict__ boxes_all, int NB, int B) {
  constexpr int PPL = BS / 32;                        // points per lane and bucket
  constexpr int QCAP = 32 * S;                        // a warp owns at most this many buckets
  extern __shared__ __align__(16) unsigned char fb_smem[];
  const int grp = threadIdx.x / (W * 32);             // scene slot of this CTA
  const int scene = blockIdx.x * G + grp;
  if (scene >= B) return;                             // whole scene groups leave; they own their barrier
  const int t = threadIdx.x - grp * (W * 32);
  const unsigned lane = t & 31u, w = t >> 5;
  // per scene: candidate coordinates [NB] float4 (k bits, x, y, z), boxes [NB] float4 + float2, per-warp queues,
  // per-warp candidates (double buffered)
  // The per-bucket tables are indexed by (warp, slot * 32 + lane), NOT by bucket: consecutive lanes then read
  // consecutive 16-byte entries (indexed by bucket the lanes were W * 16 bytes apart -- a 32-way bank conflict on
  // every box read, 13.5 M conflict wavefronts per call in ncu).
  constexpr int NL = W * QCAP;                        // table entries per scene
  unsigned char *base = fb_smem + (size_t)grp * fb_smem_per_scene(W, S);
  float4 *s_kxyz = reinterpret_cast<float4 *>(base) + w * QCAP;    // my warp's slice of each table
  float4 *s_box4 = reinterpret_cast<float4 *>(base) + NL + w * QCAP;
  float2 *s_box2 = reinterpret_cast<float2 *>(reinterpret_cast<float4 *>(base) + 2 * NL) + w * QCAP;
  uint4 *s_wc = reinterpret_cast<uint4 *>(reinterpret_cast<float2 *>(reinterpret_cast<float4 *>(base) + 2 * NL) + NL);
  uint16_t *s_q = reinterpret_cast<uint16_t *>(s_wc + 8 * W) + w * QCAP;      // s_wc: [2][W] x 4 uint4

  const float *xyz = p.xyz + (size_t)scene * p.N * 3;
  if (p.ordered_ok != nullptr && p.ordered_ok[scene] != 0) {       // verified shortcut, as in fps_cluster_kernel
    if (t == 0 && p.strict_out) p.strict_out[scene] = 1;
    int32_t *oidx = p.idx + (size_t)scene * p.npoint;
    for (int j = t; j < p.npoint; j += W * 32) oidx[j] = j;
    if (p.new_xyz) {
      float *o = p.new_xyz + (size_t)scene * p.npoint * 3;
      for (int e = t; e < 3 * p.npoint; e += W * 32) o[e] = __ldg(xyz + e);
    }
    return;
  }
  float4 *pts = pts_all + (size_t)scene * NB * BS;
  const int32_t *kk = kk_all + (size_t)scene * NB * BS;
  const float *boxes = boxes_all + (size_t)scene * NB * 6;
  unsigned key[S];                                    // candidate key of my buckets; 0 = nothing selectable
  // second-largest key of my buckets (== key[s]: another point of the bucket holds the candidate's key, a tie)
  unsigned key2[S];
  // "Every pick so far was the strict unique maximum" (p.strict_out): then FPS over any prefix of the OUTPUT is the
  // identity and the next set-abstraction layers skip their sampling without the proof kernels.  Every candidate
  // carries one bit "another point holds the same key" up the three arg-max levels; only the winner's bit counts.
  bool strict = true;                                 // uniform over the scene's threads
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int b = (s * 32 + (int)lane) * W + (int)w;
    key[s] = 0u;
    if (b < NB) {
      const float lx = __ldg(boxes + 6 * b + 0), ly = __ldg(boxes + 6 * b + 1), lz = __ldg(boxes + 6 * b + 2);
      const float hx = __ldg(boxes + 6 * b + 3), hy = __ldg(boxes + 6 * b + 4), hz = __ldg(boxes + 6 * b + 5);
      s_box4[s * 32 + lane] = make_float4(lx, ly, lz, hx);
      s_box2[s * 32 + lane] = make_float2(hy, hz);
      s_kxyz[s * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
      key[s] = hx >= lx ? FB_KEY_INIT : 0u;           // every min-distance starts at 1e10
    }
    key2[s] = key[s];                                 // until the first visit: conservative
  }
  const float p0x = __ldg(xyz + 0), p0y = __ldg(xyz + 1), p0z = __ldg(xyz + 2);
  // the centres the next update applies: the last round's picks, (q) == (o) after a round with one pick
  float ox = p0x, oy = p0y, oz = p0z, qx = p0x, qy = p0y, qz = p0z;
  int32_t *idx = p.idx + (size_t)scene * p.npoint;
  float *nxyz = p.new_xyz ? p.new_xyz + (size_t)scene * p.npoint * 3 : nullptr;
  const bool writer = t == W * 32 - 1;
  if (writer) {
    idx[0] = 0;
    if (nxyz) { nxyz[0] = ox; nxyz[1] = oy; nxyz[2] = oz; }
  }
  __syncwarp();                                       // every table entry is written and read by its own warp only

  unsigned buf = 0u;                                  // s_wc buffer of this round (alternates per round, not per pick)
  for (int j = 1; j < p.npoint; buf ^= 1u) {
    // ---- 1. cull my buckets: which of them can these centres change? ------------------------------
    int nq = 0;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      // no branch around the test: the S slots are independent chains the scheduler can interleave (entries past
      // the last bucket hold whatever shared memory held; their key is 0, so the result is discarded)
      const float4 b4 = s_box4[s * 32 + lane];
      const float2 b2 = s_box2[s * 32 + lane];
      const float ex = fmaxf(0.f, fmaxf(b4.x - ox, ox - b4.w)), ey = fmaxf(0.f, fmaxf(b4.y - oy, oy - b2.x)),
                  ez = fmaxf(0.f, fmaxf(b4.z - oz, oz - b2.y));
      const float fx = fmaxf(0.f, fmaxf(b4.x - qx, qx - b4.w)), fy = fmaxf(0.f, fmaxf(b4.y - qy, qy - b2.x)),
                  fz = fmaxf(0.f, fmaxf(b4.z - qz, qz - b2.y));
      // conservative w.r.t. fp32 rounding
      const float lb2 = fminf(ex * ex + ey * ey + ez * ez, fx * fx + fy * fy + fz * fz) * 0.99999f;
      const bool touch = key[s] != 0u && lb2 < __uint_as_float(key[s] - 1u);
      const unsigned m = __ballot_sync(0xffffffffu, touch);
      if (touch) s_q[nq + __popc(m & ((1u << lane) - 1u))] = (uint16_t)(s * 32 + (int)lane);
      nq += __popc(m);
    }
    __syncwarp();
    // ---- 2. update the touched buckets (whole warp per bucket, the next bucket's loads in flight) ----
    float4 pt[PPL], ptn[PPL];
    int kq[PPL], kqn[PPL];
    int sl = 0, sln = 0;
    auto issue = [&](int e, float4 (&P)[PPL], int (&K)[PPL], int &slot) {
      slot = (int)s_q[e];
      const int b = slot * W + (int)w;
#pragma unroll
      for (int q = 0; q < PPL; ++q) {
        const int pos = b * BS + q * 32 + (int)lane;
        P[q] = pts[pos];
        K[q] = __ldg(kk + pos);
      }
    };
    if (nq > 0) issue(0, ptn, kqn, sln);
    for (int e = 0; e < nq; ++e) {
#pragma unroll
      for (int q = 0; q < PPL; ++q) { pt[q] = ptn[q]; kq[q] = kqn[q]; }
      sl = sln;
      if (e + 1 < nq) issue(e + 1, ptn, kqn, sln);
      const int b = sl * W + (int)w;
      unsigned bkey = 0u, skey = 0u;                  // my best and second-best key
      int bq = 0;
#pragma unroll
      for (int q = 0; q < PPL; ++q) {
        const float t1 = fminf(sqdist_ref(pt[q].x, pt[q].y, pt[q].z, ox, oy, oz), pt[q].w);
        const float t2 = fminf(sqdist_ref(pt[q].x, pt[q].y, pt[q].z, qx, qy, qz), t1);
        if (t2 < pt[q].w) pts[b * BS + q * 32 + (int)lane].w = t2;
        const unsigned kq_ = t2 < 0.f ? 0u : __float_as_uint(t2) + 1u;
        if (kq_ > bkey) { skey = bkey; bkey = kq_; bq = q; }
        else {
          skey = max(skey, kq_);
          if (q > 0 && kq_ == bkey && kq_ != 0u && fb_tie_before(kq[q], kq[bq], p.T, p.log2T, p.Q)) bq = q;
        }
      }
      float4 c = pt[0];
      int ck = kq[0];
#pragma unroll
      for (int q = 1; q < PPL; ++q) if (bq == q) { c = pt[q]; ck = kq[q]; }
      const unsigned kmax = __reduce_max_sync(0xffffffffu, bkey);
      const bool hit = bkey == kmax;
      const unsigned ties = __ballot_sync(0xffffffffu, hit);
      unsigned src = __ffs(ties) - 1u;
      if (kmax != 0u && (ties & (ties - 1u)) != 0u) src = fb_resolve_tie(hit, ck, lane, p.T, p.log2T, p.Q);
      if (lane == src) s_kxyz[sl] = make_float4(__int_as_float(ck), c.x, c.y, c.z);
      const unsigned kmax2 = __reduce_max_sync(0xffffffffu, lane == src ? skey : bkey);
      const int owner = sl & 31, oslot = sl >> 5;
#pragma unroll
      for (int s = 0; s < S; ++s)
        if (s == oslot && (int)lane == owner) { key[s] = kmax; key2[s] = kmax2; }
    }
    __syncwarp();
    // ---- 3. select: my best bucket -> the warp's -> the scene's, and the runner-up at every level ----
    unsigned mkey = key[0];
    int ms = 0;
    bool mtie = false;                                // two of my buckets hold the same best key
#pragma unroll
    for (int s = 1; s < S; ++s) {
      if (key[s] > mkey) { mkey = key[s]; ms = s; mtie = false; }
      else if (key[s] == mkey && mkey != 0u) {
        mtie = true;
        if (fb_tie_before(__float_as_int(s_kxyz[s * 32 + lane].x), __float_as_int(s_kxyz[ms * 32 + lane].x), p.T,
                          p.log2T, p.Q))
          ms = s;
      }
    }
    unsigned mkey2 = key2[0];                         // second key of my best bucket
    unsigned rkey = 0u;                               // my runner-up: the best of my other buckets
    int rs = ms;
    bool rtie = false;
#pragma unroll
    for (int s = 0; s < S; ++s) {
      if (s == ms) mkey2 = key2[s];
      else if (key[s] > rkey) { rkey = key[s]; rs = s; rtie = key2[s] == key[s]; }
      else if (key[s] == rkey) rtie = true;
    }
    mtie = mtie || mkey2 == mkey;
    const unsigned wmax = __reduce_max_sync(0xffffffffu, mkey);
    {
      uint4 *dst = s_wc + (buf * W + w) * 4;
      const bool hit = mkey == wmax;
      const unsigned ties = __ballot_sync(0xffffffffu, hit);
      unsigned src = __ffs(ties) - 1u;
      if (wmax != 0u && (ties & (ties - 1u)) != 0u)
        src = fb_resolve_tie(hit, hit ? __float_as_int(s_kxyz[ms * 32 + lane].x) : 0, lane, p.T, p.log2T, p.Q);
      const bool wtie = (ties & (ties - 1u)) != 0u || __any_sync(0xffffffffu, hit && mtie);
      if (lane == src) {
        const float4 c = wmax != 0u ? s_kxyz[ms * 32 + lane] : make_float4(0.f, 0.f, 0.f, 0.f);
        dst[0] = make_uint4(wmax, __float_as_uint(c.x), wtie ? 1u : 0u, mkey2);
        dst[1] = make_uint4(__float_as_uint(c.x), __float_as_uint(c.y), __float_as_uint(c.z), __float_as_uint(c.w));
      }
      // the warp's runner-up: my runner-up if I hold the warp's best, else my best.  Among equal keys any holder
      // will do: a tied runner-up is never taken
      const bool top = lane == src;
      const unsigned ckey = top ? rkey : mkey;
      const unsigned rmax = __reduce_max_sync(0xffffffffu, ckey);
      const bool rhit = ckey == rmax;
      const unsigned rties = __ballot_sync(0xffffffffu, rhit);
      const bool rwtie = (rties & (rties - 1u)) != 0u || __any_sync(0xffffffffu, rhit && (top ? rtie : mtie));
      if (lane == __ffs(rties) - 1u) {
        const float4 c = s_kxyz[(top ? rs : ms) * 32 + lane];
        dst[2] = make_uint4(rmax, rwtie ? 1u : 0u, 0u, 0u);
        dst[3] = make_uint4(__float_as_uint(c.x), __float_as_uint(c.y), __float_as_uint(c.z), __float_as_uint(c.w));
      }
    }
    if (W > 1) asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(W * 32) : "memory");
    else __syncwarp();
    const uint4 *wc = s_wc + buf * W * 4;
    uint4 c2 = make_uint4(0u, 0u, 0u, 0u), r2 = make_uint4(0u, 0u, 0u, 0u);
    if (lane < W) { c2 = wc[lane * 4]; r2 = wc[lane * 4 + 2]; }
    const unsigned bmax = __reduce_max_sync(0xffffffffu, c2.x);
    unsigned csrc;
    {
      const bool hit = c2.x == bmax && lane < W;
      const unsigned ties = __ballot_sync(0xffffffffu, hit);
      csrc = __ffs(ties) - 1u;
      if (bmax != 0u && (ties & (ties - 1u)) != 0u) csrc = fb_resolve_tie(hit, (int)c2.y, lane, p.T, p.log2T, p.Q);
      strict = strict && bmax != 0u && (ties & (ties - 1u)) == 0u && !__any_sync(0xffffffffu, hit && c2.z != 0u);
    }
    csrc &= 31u;
    // the scene's runner-up a2: the best candidate of every bucket but the pick's
    const bool ctop = lane == csrc;
    const unsigned ckey = ctop ? r2.x : c2.x;
    const unsigned smax = __reduce_max_sync(0xffffffffu, ckey);
    const bool shit = ckey == smax && lane < W;
    const unsigned sties = __ballot_sync(0xffffffffu, shit);
    const bool suniq = (sties & (sties - 1u)) == 0u && !__any_sync(0xffffffffu, shit && (ctop ? r2.y : c2.z) != 0u);
    const unsigned ssrc = (__ffs(sties) - 1u) & 31u;
    const unsigned akey2 = __shfl_sync(0xffffffffu, c2.w, csrc);   // key2(A1)
    int old = 0;
    if (bmax == 0u) { ox = p0x; oy = p0y; oz = p0z; }
    else {
      const uint4 c = wc[csrc * 4 + 1];
      old = (int)c.x; ox = __uint_as_float(c.y); oy = __uint_as_float(c.z); oz = __uint_as_float(c.w);
    }
    // a2 may hold the same key as a1 (the other bucket of a1's lane, or any other bucket): a1 won that tie on the
    // virtual index, drops to 0 with its own update, and a2 is then the unique maximum -- taking it is what the
    // sequential algorithm does.  What is never taken is a tie among the candidates OUTSIDE A1 (suniq).
    int old2 = 0;
    bool two = false;
    if (suniq && smax > 1u && smax > akey2 && j + 1 < p.npoint) {
      const uint4 c = wc[ssrc * 4 + (ssrc == csrc ? 3 : 1)];
      old2 = (int)c.x; qx = __uint_as_float(c.y); qy = __uint_as_float(c.z); qz = __uint_as_float(c.w);
      two = sqdist_ref(qx, qy, qz, ox, oy, oz) >= __uint_as_float(smax - 1u);
    }
    if (!two) { qx = ox; qy = oy; qz = oz; }
    if (writer) {
      idx[j] = old;
      if (nxyz) { nxyz[3 * j + 0] = ox; nxyz[3 * j + 1] = oy; nxyz[3 * j + 2] = oz; }
      if (two) {
        idx[j + 1] = old2;
        if (nxyz) { nxyz[3 * j + 3] = qx; nxyz[3 * j + 4] = qy; nxyz[3 * j + 5] = qz; }
      }
    }
    j += two ? 2 : 1;
  }
  if (writer && p.strict_out) p.strict_out[scene] = strict ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
// "Verify in parallel what would be constructed sequentially".
// SA2..SA4 of the detector run FPS on the OUTPUT of the previous FPS (an FPS-ordered point list),
// where the answer is 0..npoint-1 unless exact distance ties interfere (SURVEY F10: the reference
// model silently relies on this).  Whether FPS(xyz)[0:npoint] == identity can be CHECKED with no
// sequential dependency: with the first j points selected, point j must be the unique maximum of
// the running min-distance among all not-yet-selected points.  Kernel A computes
// D[j] = min_{i<j} d(p_j, p_i) (what round j's winner scored); kernel B recomputes every point's
// running min-distance and flags any k > j that reaches D[j] (a tie or a larger value -- then
// the tie-break / order decides and the full kernel must run).  Same fp32 arithmetic as the
// sequential kernel (sqdist_ref, fminf, temp = 1e10), so the proof is exact, not approximate.
// Cost: N*npoint distance evaluations, fully parallel (~10 us for 2048 -> 1024 at B=8) instead
// of npoint-1 sequential rounds (~290 us).
// ------------------------------------------------------------------------------------------------
__global__ void fps_fill_kernel(int *p, int n, int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

constexpr int CHK_THREADS = 128;
constexpr int CHK_TILE = 256;

__device__ __forceinline__ bool fps_skipped(float x, float y, float z) {
  const float mag = __fmaf_rn(z, z, __fmaf_rn(x, x, __fmul_rn(y, y)));
  return (double)mag <= 1e-3;
}

// D[b][j] = min(1e10, min_{i<j} d(p_j, p_i)) for j < npoint;   ok[b] = 0 if a prefix point other than
// p_0 is one the reference never selects (|p|^2 <= 1e-3)
__global__ void __launch_bounds__(CHK_THREADS) fps_prefix_dist_kernel(const float *__restrict__ xyz, int N,
                                                                       int npoint, float *__restrict__ D,
                                                                       int *__restrict__ ok,
                                                                       const int *__restrict__ known) {
  __shared__ float sx[CHK_TILE], sy[CHK_TILE], sz[CHK_TILE];
  const int b = blockIdx.y;
  if (known != nullptr && known[b] != 0) return;   // already established by the call that produced xyz
  const float *P = xyz + (size_t)b * N * 3;
  const int j = blockIdx.x * CHK_THREADS + threadIdx.x;
  const bool act = j < npoint;
  const float px = act ? __ldg(P + 3 * j) : 0.f, py = act ? __ldg(P + 3 * j + 1) : 0.f,
              pz = act ? __ldg(P + 3 * j + 2) : 0.f;
  if (act && j > 0 && fps_skipped(px, py, pz)) ok[b] = 0;
  float m = 1e10f;
  const int jmax = min(npoint, (int)(blockIdx.x + 1) * CHK_THREADS);   // largest j of this block + 1
  for (int base = 0; base < jmax - 1; base += CHK_TILE) {
    const int tile = min(CHK_TILE, jmax - 1 - base);
    __syncthreads();
    for (int e = threadIdx.x; e < tile * 3; e += CHK_THREADS) {
      const float v = __ldg(P + (size_t)base * 3 + e);
      const int pt = e / 3, c = e - pt * 3;
      (c == 0 ? sx : c == 1 ? sy : sz)[pt] = v;
    }
    __syncthreads();
    const int lim = min(tile, j - base);          // only i < j
    for (int i = 0; i < lim; ++i) {
      // the reference never updates temp from a skipped centre?  No: the CENTRE may be any point
      // (only index 0 can be a skipped one, and it is used as a centre like any other)
      m = fminf(sqdist_ref(px, py, pz, sx[i], sy[i], sz[i]), m);
    }
  }
  if (act) {
    D[(size_t)b * npoint + j] = m;
    // a winner at distance 0 (duplicate of an earlier point) ties with every selected point
    if (j > 0 && !(m > 0.f)) ok[b] = 0;
  }
}

// ok[b] &= for all rounds j in [1, npoint) and all points k > j (not skipped):
//            min(1e10, min_{i<j} d(p_k, p_i)) < D[j]
__global__ void __launch_bounds__(CHK_THREADS) fps_prefix_check_kernel(const float *__restrict__ xyz, int N,
                                                                        int npoint,
                                                                        const float *__restrict__ D,
                                                                        int *__restrict__ ok,
                                                                        const int *__restrict__ known) {
  __shared__ float sx[CHK_TILE], sy[CHK_TILE], sz[CHK_TILE], sd[CHK_TILE];
  const int b = blockIdx.y;
  if (known != nullptr && known[b] != 0) return;
  const float *P = xyz + (size_t)b * N * 3;
  const float *Db = D + (size_t)b * npoint;
  const int k = blockIdx.x * CHK_THREADS + threadIdx.x;
  const bool act = k < N;
  const float px = act ? __ldg(P + 3 * k) : 0.f, py = act ? __ldg(P + 3 * k + 1) : 0.f,
              pz = act ? __ldg(P + 3 * k + 2) : 0.f;
  const bool cand = act && !fps_skipped(px, py, pz);   // skipped points are never candidates
  float m = 1e10f;
  bool bad = false;
  for (int base = 0; base < npoint - 1; base += CHK_TILE) {
    const int tile = min(CHK_TILE, npoint - 1 - base);
    __syncthreads();
    for (int e = threadIdx.x; e < tile * 3; e += CHK_THREADS) {
      const float v = __ldg(P + (size_t)base * 3 + e);
      const int pt = e / 3, c = e - pt * 3;
      (c == 0 ? sx : c == 1 ? sy : sz)[pt] = v;
    }
    for (int e = threadIdx.x; e < tile; e += CHK_THREADS) sd[e] = __ldg(Db + base + e + 1);   // D[j], j = i+1
    __syncthreads();
    for (int i = 0; i < tile; ++i) {
      m = fminf(sqdist_ref(px, py, pz, sx[i], sy[i], sz[i]), m);
      // round j = base+i+1 picks among points with index > j - 1 that are not yet selected
      bad |= (k > base + i + 1) && (m >= sd[i]);
    }
  }
  if (cand && bad) ok[b] = 0;   // benign race: every writer stores 0
}

template <int P, int THREADS, bool XYZ_REGS>
static int launch_fps(const FpsParams &p, int B, int C, cudaStream_t stream) {
  auto kern = fps_cluster_kernel<P, THREADS, XYZ_REGS>;
  const size_t smem = (size_t)4 * P * THREADS * sizeof(float);
  SPC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (C > 8) SPC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(C, B, 1);
  cfg.blockDim = dim3(THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  SPC_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  return SPC_OK;
}

// how many clusters of size C (512 threads, given smem) can be co-resident; cached per C
template <int P, int THREADS, bool XYZ_REGS>
static int max_active_clusters(int C) {
  auto kern = fps_cluster_kernel<P, THREADS, XYZ_REGS>;
  const size_t smem = (size_t)4 * P * THREADS * sizeof(float);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (C > 8) cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(C, 1, 1);
  cfg.blockDim = dim3(THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
  return n;
}

}  // namespace spc

using namespace spc;

#define FPS_CASE(PV, TH, REGS)                                         \
  case PV: return launch_fps<PV, TH, REGS>(p, B, C, stream);

static int fps_impl(const float *xyz, int B, int N, int npoint, int32_t *idx, float *new_xyz,
                    int hint_ordered, const int32_t *known_ordered, int32_t *strict_out, void *workspace,
                    size_t workspace_bytes, int algo, void *stream_);

// bucket size of the bucketed sampler for a cloud of N points (0 = not applicable): ~500-1300 buckets keep the
// per-round scan of the bucket table at 2-5 entries per thread
static int fb_bucket_size(int N) {
  if (N < 4096 || N > FMS_THREADS * FMS_ITEMS) return 0;   // the Morton sort's capacity bounds this path
  return N <= 20480 ? 32 : 64;
}
static size_t fb_align16(size_t x) { return (x + 15) & ~(size_t)15; }

// workspace layout: D (B,npoint) f32 | ok (B) i32 | perm (B,N) i32 | [16-byte aligned] pts (B,NB*BS) float4 |
// kk (B,NB*BS) i32 | boxes (B,NB,6) f32
extern "C" size_t spc_fps_workspace_bytes(int B, int N, int npoint) {
  size_t bytes = ((size_t)B * (size_t)(npoint > 0 ? npoint : 0) + (size_t)B + (size_t)B * (size_t)(N > 0 ? N : 0)) * 4;
  const int BS = fb_bucket_size(N);
  if (BS) {
    const size_t NB = ((size_t)N + BS - 1) / BS;
    bytes = fb_align16(bytes) + (size_t)B * NB * BS * 20 + (size_t)B * NB * 24;
  }
  return bytes;
}

extern "C" int spc_furthest_point_sampling(const float *xyz, int B, int N, int npoint,
                                           int32_t *idx, float *new_xyz, void *stream_) {
  return fps_impl(xyz, B, N, npoint, idx, new_xyz, 0, nullptr, nullptr, nullptr, 0, SPC_FPS_AUTO, stream_);
}

extern "C" int spc_furthest_point_sampling_ex(const float *xyz, int B, int N, int npoint,
                                              int32_t *idx, float *new_xyz, int hint_ordered,
                                              void *workspace, size_t workspace_bytes,
                                              void *stream_) {
  return fps_impl(xyz, B, N, npoint, idx, new_xyz, hint_ordered, nullptr, nullptr, workspace, workspace_bytes,
                  SPC_FPS_AUTO, stream_);
}

extern "C" int spc_furthest_point_sampling_ex2(const float *xyz, int B, int N, int npoint, int32_t *idx,
                                               float *new_xyz, int hint_ordered, const int32_t *known_ordered,
                                               int32_t *strict_out, void *workspace, size_t workspace_bytes,
                                               int algo, void *stream_) {
  SPC_CHECK_ARG(algo == SPC_FPS_AUTO || algo == SPC_FPS_CLUSTER || algo == SPC_FPS_BUCKET,
                "fps: algo %d is not one of SPC_FPS_AUTO / _CLUSTER / _BUCKET", algo);
  return fps_impl(xyz, B, N, npoint, idx, new_xyz, hint_ordered, known_ordered, strict_out, workspace,
                  workspace_bytes, algo, stream_);
}

template <int BS, int W, int G, int S>
static int launch_fps_bucket_cfg(const FpsParams &p, int B, int NB, float4 *pts, const int32_t *kk, const float *boxes,
                                 cudaStream_t stream) {
  auto kern = fps_bucket_kernel<BS, W, G, S>;
  const size_t smem = fb_smem_per_scene(W, S) * G;
  if (smem > 227 * 1024) {
    set_error("fps: bucket table of %d entries x %d scenes does not fit in shared memory", NB, G);
    return SPC_ERR_UNSUPPORTED;
  }
  SPC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<ceil_div(B, G), W * G * 32, smem, stream>>>(p, pts, kk, boxes, NB, B);
  SPC_LAUNCH_CHECK("fps_bucket_kernel");
  return SPC_OK;
}

template <int BS>
static int launch_fps_bucket(const FpsParams &p, int B, int N, int32_t *perm, void *ws_tail, cudaStream_t stream) {
  const int NB = (N + BS - 1) / BS;
  float4 *pts = reinterpret_cast<float4 *>(ws_tail);
  int32_t *kk = reinterpret_cast<int32_t *>(pts + (size_t)B * NB * BS);
  float *boxes = reinterpret_cast<float *>(kk + (size_t)B * NB * BS);
  const size_t sort_smem = (size_t)FMS_BINS * sizeof(int);
  SPC_CUDA(cudaFuncSetAttribute(fps_morton_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
  fps_morton_sort_kernel<<<B, FMS_THREADS, sort_smem, stream>>>(p.xyz, N, perm);
  SPC_LAUNCH_CHECK("fps_morton_sort_kernel");
  fps_bucket_build_kernel<BS><<<dim3(ceil_div(NB, 8), B), 256, 0, stream>>>(p.xyz, perm, N, NB, pts, kk, boxes);
  SPC_LAUNCH_CHECK("fps_bucket_build_kernel");
  // 16 warps per scene, one scene per CTA.  Measured on B200 (8 x 40 k -> 2048; ms per call alone / k scenes per second
  // with 32 sampler calls in flight / k scenes per second of the whole detector pipeline), after the bank-conflict fix:
  //   W8 G1 3.65 / 48.3 / 17.6;   W16 G1 3.04 / 56.6 / 18.8;   W32 G1 2.86 / 43.9 / 17.1
  // and before it, scenes packed onto one SM:  W8 G2 4.9 / 42.8 / 16.4;  W8 G4 7.0 / 33.7 / 14.2;  W4 G8 8.3 / 26.8 / 12.5.
  // A round is a chain of dependent instructions (cull -> L2 load -> update -> three arg-max levels): more warps
  // shorten the per-warp chain and balance the bucket visits, scenes sharing an SM slow each other down.
  constexpr int W = 16;
  const int S = ceil_div(ceil_div(NB, W), 32);
  switch (S) {
    case 1: return launch_fps_bucket_cfg<BS, W, 1, 1>(p, B, NB, pts, kk, boxes, stream);
    case 2: return launch_fps_bucket_cfg<BS, W, 1, 2>(p, B, NB, pts, kk, boxes, stream);
  }
  set_error("fps: no bucket kernel for %d buckets", NB);
  return SPC_ERR_UNSUPPORTED;
}

static int fps_impl(const float *xyz, int B, int N, int npoint, int32_t *idx, float *new_xyz,
                    int hint_ordered, const int32_t *known_ordered, int32_t *strict_out, void *workspace,
                    size_t workspace_bytes, int algo, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && N >= 1 && npoint >= 0, "fps: bad sizes B=%d N=%d npoint=%d", B, N, npoint);
  SPC_CHECK_ARG(xyz && (idx || npoint == 0 || B == 0), "fps: null pointer");
  if (B == 0 || npoint == 0) return SPC_OK;
  cudaStream_t stream = (cudaStream_t)stream_;
  FpsParams p;
  p.xyz = xyz; p.idx = idx; p.new_xyz = new_xyz; p.N = N; p.npoint = npoint;
  p.T = ref_opt_n_threads(N);
  p.log2T = 0;
  while ((1 << p.log2T) < p.T) ++p.log2T;
  p.Q = (N + p.T - 1) / p.T;
  p.ordered_ok = nullptr;
  p.strict_out = strict_out;
  // ---- optional verified shortcut for FPS-ordered inputs ---------------------------------------
  if (hint_ordered && workspace && npoint >= 2 && npoint <= N &&
      workspace_bytes >= spc_fps_workspace_bytes(B, N, npoint) && B <= 65535 &&
      (long long)N * npoint <= (1LL << 26)) {
    float *D = reinterpret_cast<float *>(workspace);
    int *ok = reinterpret_cast<int *>(D + (size_t)B * npoint);
    fps_fill_kernel<<<ceil_div(B, 128), 128, 0, stream>>>(ok, B, 1);
    fps_prefix_dist_kernel<<<dim3(ceil_div(npoint, CHK_THREADS), B), CHK_THREADS, 0, stream>>>(xyz, N, npoint, D, ok, known_ordered);
    fps_prefix_check_kernel<<<dim3(ceil_div(N, CHK_THREADS), B), CHK_THREADS, 0, stream>>>(xyz, N, npoint, D, ok, known_ordered);
    SPC_LAUNCH_CHECK("fps_prefix_check");
    p.ordered_ok = ok;
  }
  if (p.ordered_ok == nullptr && known_ordered != nullptr && npoint <= N) p.ordered_ok = known_ordered;
  const long long V = (long long)p.T * p.Q;

  // ---- small clouds: one CTA of 256 threads -------------------------------------------------
  if (V <= 256 * 16) {
    const int C = 1;
    const int need = (int)((V + 255) / 256);
    const int P = need <= 1 ? 1 : need <= 2 ? 2 : need <= 4 ? 4 : need <= 8 ? 8 : 16;
    switch (P) {
      FPS_CASE(1, 256, true) FPS_CASE(2, 256, true) FPS_CASE(4, 256, true)
      FPS_CASE(8, 256, true) FPS_CASE(16, 256, true)
    }
  }
  // ---- bucketed sampler (points parked in L2, one small CTA per scene): needs the caller's workspace -------
  const int BS = fb_bucket_size(N);
  // SPC_FPS_AUTO serves the single call: the cluster sampler finishes a 40 k-point scene in 1.25 ms, the bucketed one
  // in 4 ms -- but it holds a quarter of an SM instead of four, which is what a pipeline with many batches in flight
  // wants (spacap3d_b200/pipeline.py asks for it explicitly).
  if (algo == SPC_FPS_BUCKET && BS && workspace && workspace_bytes >= spc_fps_workspace_bytes(B, N, npoint) &&
      npoint >= 2) {
    const size_t head = ((size_t)B * npoint + (size_t)B + (size_t)B * N) * 4;
    int32_t *perm = reinterpret_cast<int32_t *>(workspace) + (size_t)B * npoint + (size_t)B;
    void *tail = reinterpret_cast<char *>(workspace) + fb_align16(head);
    SPC_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "fps: workspace must be 16-byte aligned");
    return BS == 32 ? launch_fps_bucket<32>(p, B, N, perm, tail, stream)
                    : launch_fps_bucket<64>(p, B, N, perm, tail, stream);
  }
  if (algo == SPC_FPS_BUCKET) {
    set_error("fps: SPC_FPS_BUCKET needs a workspace of spc_fps_workspace_bytes() and 4096 <= N <= %d (got N=%d)",
              FMS_THREADS * FMS_ITEMS, N);
    return SPC_ERR_UNSUPPORTED;
  }
  // ---- clusters of 512-thread CTAs ------------------------------------------------------------
  // The rounds are latency-bound, so all B scenes should be co-resident.  Measured on B200
  // (B=8, N=40k): C=8 0.81 us/round, C=16 1.03 (slower exchange across a non-portable cluster),
  // C=4 1.19 (xyz no longer fits in registers) -> prefer 8.
  // The occupancy answers depend on the DEVICE (nn.DataParallel drives several from one process): cached per device.
  static std::mutex occ_mutex;
  static int cached_max16[64], cached_max8[64];
  static bool cached_init = false;
  int dev = 0;
  SPC_CUDA(cudaGetDevice(&dev));
  dev = dev < 0 || dev >= 64 ? 0 : dev;
  int max8, max16 = -1;
  {
    std::lock_guard<std::mutex> lock(occ_mutex);
    if (!cached_init) { for (int d = 0; d < 64; ++d) cached_max16[d] = cached_max8[d] = -1; cached_init = true; }
    if (cached_max8[dev] < 0) cached_max8[dev] = max_active_clusters<10, 512, true>(8);
    max8 = cached_max8[dev];
  }
  int C = 8;
  if (max8 > 0 && max8 < B) C = (B * 4 <= kNumSMs) ? 4 : 2;
  int need = (int)((V + (long long)C * 512 - 1) / ((long long)C * 512));
  while (need > 27 && C < 16) { C *= 2; need = (int)((V + (long long)C * 512 - 1) / ((long long)C * 512)); }
  if (C == 16) {
    std::lock_guard<std::mutex> lock(occ_mutex);
    if (cached_max16[dev] < 0) cached_max16[dev] = max_active_clusters<6, 512, true>(16);
    max16 = cached_max16[dev];
  }
  if (C == 16 && max16 <= 0) {
    set_error("fps: N=%d needs a 16-CTA cluster which this device cannot schedule", N);
    return SPC_ERR_UNSUPPORTED;
  }
  if (need > 27) {
    set_error("fps: N=%d exceeds the on-chip capacity of a 16-CTA cluster (max %d points)", N, 16 * 512 * 27);
    return SPC_ERR_UNSUPPORTED;
  }
  while (C > 1 && need <= 1) { C /= 2; need = (int)((V + (long long)C * 512 - 1) / ((long long)C * 512)); }
  // 256-thread CTAs with 20 points per thread and TWO CTAs per SM whenever the cloud fits: fewer
  // warps per reduction level make a round faster (1.32 vs 1.51 ms for 40k -> 2048 at batch 8) and
  // two latency-bound CTAs (of different scenes / batches) share one SM's issue slots.
  {
    const int need256 = (int)((V + (long long)C * 256 - 1) / ((long long)C * 256));
    if (need256 <= 20 && need256 > 4) {
      const int P256 = need256 <= 8 ? 8 : need256 <= 10 ? 10 : need256 <= 16 ? 16 : 20;
      switch (P256) {
        FPS_CASE(8, 256, true) FPS_CASE(10, 256, true) FPS_CASE(16, 256, true) FPS_CASE(20, 256, true)
      }
    }
  }
  // P = 27 is the most that fits: 4 arrays x 27 x 512 x 4 B = 216 KB of the 227 KB a CTA may use
  static const int opts[] = {2, 3, 4, 5, 6, 8, 10, 12, 16, 20, 24, 27};
  int P = 27;
  for (int o : opts) if (o >= need) { P = o; break; }
  switch (P) {
    FPS_CASE(2, 512, true) FPS_CASE(3, 512, true) FPS_CASE(4, 512, true) FPS_CASE(5, 512, true)
    FPS_CASE(6, 512, true) FPS_CASE(8, 512, true) FPS_CASE(10, 512, true) FPS_CASE(12, 512, true)
    FPS_CASE(16, 512, true) FPS_CASE(20, 512, true) FPS_CASE(24, 512, false) FPS_CASE(27, 512, false)
  }
  set_error("fps: internal dispatch error");
  return SPC_ERR_UNSUPPORTED;
}
