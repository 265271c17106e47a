// group.cu -- gather_points / group_points and their backward passes (sm_100a).
//
// Replaces gather_points_kernel, gather_points_grad_kernel (reference sampling_gpu.cu:8-57) and
// group_points_kernel, group_points_grad_kernel (reference group_points_gpu.cu:8-75).  The
// reference launches one block per scene, stores with a stride of nsample floats between
// adjacent threads and gathers 4 bytes at a time straight from L2 (SURVEY F6).
//
// group_points is the HBM-bound op of the path (out = C*npoint*nsample floats).  Design:
//  * a CTA stages CT whole channel rows (CT*N floats) of one scene in shared memory with ONE
//    bulk-TMA copy (cp.async.bulk, completion on an mbarrier) -- the rows of a scene are
//    contiguous in the (B,C,N) layout, so no tensor map is needed;
//  * the random 4-byte gathers then hit shared memory instead of 32-byte L2 sectors, the index
//    tile is read once per CTA with 16-byte loads and reused for all CT channels, and the
//    output is written with coalesced 16-byte streaming stores (4 consecutive positions / thread);
//  * rows that do not fit in shared memory (N > ~50k) fall back to read-only-cache gathers.
// The backward pass mirrors it: CT accumulator rows live in shared memory, duplicates inside a
// warp are pre-combined (warp-aggregated atomics, __match_any_sync) before a shared-memory
// atomic, and rows are flushed with plain coalesced stores (or global atomics when the
// position range had to be split across CTAs to fill the machine).
// group_points and its backward are instantiated for float and bf16 storage (common.cuh): bf16 rows are grouped as
// bf16, and the backward reads a bf16 grad_out and accumulates and writes an fp32 gradient (B,C,N), nsample times
// smaller than grad_out, so the accumulation logic and the partitions are the same for both.
#include "common.cuh"
#include "ptx.cuh"

namespace spc {

// ----------------------------------------------------------------------------------------------
// gather_points:  out[b,c,j] = points[b,c,idx[b,j]]      (tiny: C is 3 in SpaCap3D)
// ----------------------------------------------------------------------------------------------
__global__ void gather_points_kernel(const float *__restrict__ points,
                                     const int32_t *__restrict__ idx, int C, int N, int M,
                                     float *__restrict__ out) {
  const int b = blockIdx.z;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= M) return;
  const int a = __ldg(idx + (size_t)b * M + j);
  for (int c = blockIdx.y; c < C; c += gridDim.y)
    out[((size_t)b * C + c) * M + j] = __ldg(points + ((size_t)b * C + c) * N + a);
}

__global__ void gather_points_grad_kernel(const float *__restrict__ grad_out,
                                          const int32_t *__restrict__ idx, int C, int N, int M,
                                          float *__restrict__ grad_points) {
  const int b = blockIdx.z;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= M) return;
  const int a = __ldg(idx + (size_t)b * M + j);
  for (int c = blockIdx.y; c < C; c += gridDim.y)
    atomicAdd(grad_points + ((size_t)b * C + c) * N + a, __ldg(grad_out + ((size_t)b * C + c) * M + j));
}

// ----------------------------------------------------------------------------------------------
// group_points forward
// ----------------------------------------------------------------------------------------------
constexpr int GP_THREADS = 512;

// grid = (position chunks, channel tiles, B).  STAGED: rows in smem, else gathers via LDG.
template <class T, bool STAGED, bool VEC4>
__global__ void __launch_bounds__(GP_THREADS) group_points_kernel(
    const T *__restrict__ points, const int32_t *__restrict__ idx, int C, int N, int S, int CT,
    int chunk, T *__restrict__ out) {
  extern __shared__ __align__(128) float s_smem[];
  T *s_rows = reinterpret_cast<T *>(s_smem);        // [CT][N]
  __shared__ __align__(8) uint64_t bar;
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * CT;
  const int ct = min(CT, C - c0);
  const int p0 = blockIdx.x * chunk;
  const int p1 = min(S, p0 + chunk);
  const T *src = points + ((size_t)b * C + c0) * N;
  const int32_t *ix = idx + (size_t)b * S;
  T *dst = out + ((size_t)b * C + c0) * S;
  const int tid = threadIdx.x;

  if (STAGED) {
    const size_t bytes = (size_t)ct * N * sizeof(T);
    const bool bulk_ok = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && (bytes % 16 == 0);
    if (bulk_ok) {
      if (tid == 0) { mbarrier_init(&bar, 1); fence_mbarrier_init(); }
      __syncthreads();
      if (tid == 0) {
        // expect_tx is limited to 2^20-1 bytes per call; our rows are <= 227 KB
        mbarrier_arrive_expect_tx(&bar, (unsigned)bytes);
        bulk_g2s(s_rows, src, (unsigned)bytes, &bar);
      }
      mbarrier_wait(&bar, 0);
    } else {
      for (size_t e = tid; e < (size_t)ct * N; e += GP_THREADS) s_rows[e] = __ldg(src + e);
      __syncthreads();
    }
  }

  if (VEC4) {
    // S % 4 == 0 and chunk % 4 == 0: 4 consecutive positions per thread, 16-byte idx load, 4 * sizeof(T)-byte store.
    // The index loads of UNR iterations are issued together: with one CTA per SM (a 160 KB row)
    // the loop is otherwise bound by the L2 latency of one idx load per thread.
    constexpr int UNR = 4;
    int t = p0 + tid * 4;
    for (; t + (UNR - 1) * GP_THREADS * 4 < p1; t += UNR * GP_THREADS * 4) {
      int4 i4[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) i4[u] = __ldg(reinterpret_cast<const int4 *>(ix + t + u * GP_THREADS * 4));
#pragma unroll 2
      for (int c = 0; c < ct; ++c) {
        const T *r = STAGED ? s_rows + (size_t)c * N : src + (size_t)c * N;
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
          T a0, a1, a2, a3;
          if (STAGED) { a0 = r[i4[u].x]; a1 = r[i4[u].y]; a2 = r[i4[u].z]; a3 = r[i4[u].w]; }
          else { a0 = __ldg(r + i4[u].x); a1 = __ldg(r + i4[u].y); a2 = __ldg(r + i4[u].z); a3 = __ldg(r + i4[u].w); }
          st_cs4(dst + (size_t)c * S + t + u * GP_THREADS * 4, a0, a1, a2, a3);
        }
      }
    }
    for (; t < p1; t += GP_THREADS * 4) {
      const int4 i4 = __ldg(reinterpret_cast<const int4 *>(ix + t));
#pragma unroll 4
      for (int c = 0; c < ct; ++c) {
        T a0, a1, a2, a3;
        if (STAGED) {
          const T *r = s_rows + (size_t)c * N;
          a0 = r[i4.x]; a1 = r[i4.y]; a2 = r[i4.z]; a3 = r[i4.w];
        } else {
          const T *r = src + (size_t)c * N;
          a0 = __ldg(r + i4.x); a1 = __ldg(r + i4.y); a2 = __ldg(r + i4.z); a3 = __ldg(r + i4.w);
        }
        st_cs4(dst + (size_t)c * S + t, a0, a1, a2, a3);
      }
    }
  } else {
    for (int t = p0 + tid; t < p1; t += GP_THREADS) {
      const int i = __ldg(ix + t);
      for (int c = 0; c < ct; ++c)
        dst[(size_t)c * S + t] = STAGED ? s_rows[(size_t)c * N + i] : __ldg(src + (size_t)c * N + i);
    }
  }
}

// ----------------------------------------------------------------------------------------------
// group_points backward:  grad_points[b,c,idx[b,t]] += grad_out[b,c,t]
// ----------------------------------------------------------------------------------------------
// Warp-aggregated add into a shared (or global) accumulator row: lanes holding the same index
// are combined first, so the ball-query padding (one index repeated up to nsample times) costs
// one atomic instead of a same-address serialisation.  `peers` = lanes with my index
// (__match_any_sync, computed once per position and reused for every channel).
__device__ __forceinline__ void warp_agg_add(float *row, int i, float v, unsigned peers) {
  const unsigned lane = lane_id();
  if (peers == (1u << lane)) {  // common case: my index is unique in the warp
    atomicAdd(row + i, v);
    return;
  }
  float sum = 0.f;
  for (unsigned m = peers; m; m &= m - 1) sum += __shfl_sync(peers, v, __ffs(m) - 1);
  if ((int)lane == __ffs(peers) - 1) atomicAdd(row + i, sum);
}

template <class T, bool STAGED>
__global__ void __launch_bounds__(GP_THREADS) group_points_grad_kernel(
    const T *__restrict__ grad_out, const int32_t *__restrict__ idx, int C, int N, int S,
    int CT, int chunk, int use_global_atomics, float *__restrict__ grad_points) {
  extern __shared__ __align__(128) float s_rows[];  // [CT][N] accumulators
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * CT;
  const int ct = min(CT, C - c0);
  const int p0 = blockIdx.x * chunk;
  const int p1 = min(S, p0 + chunk);
  const T *g = grad_out + ((size_t)b * C + c0) * S;
  const int32_t *ix = idx + (size_t)b * S;
  float *dst = grad_points + ((size_t)b * C + c0) * N;
  const int tid = threadIdx.x;

  if (STAGED) {
    for (int e = tid; e < ct * N; e += GP_THREADS) s_rows[e] = 0.f;
    __syncthreads();
  }
  const int span = p1 - p0;
  const int iters = (span + GP_THREADS - 1) / GP_THREADS;
  for (int it = 0; it < iters; ++it) {
    const int t = p0 + it * GP_THREADS + tid;
    const bool active = t < p1;
    const int i = active ? __ldg(ix + t) : 0;
    const unsigned act = __ballot_sync(0xffffffffu, active);
    if (!active) continue;
    const unsigned peers = __match_any_sync(act, i);
    for (int c = 0; c < ct; ++c) {
      const float v = to_f32(__ldg(g + (size_t)c * S + t));
      warp_agg_add(STAGED ? s_rows + (size_t)c * N : dst + (size_t)c * N, i, v, peers);
    }
  }
  if (STAGED) {
    __syncthreads();
    if (use_global_atomics) {
      for (int e = tid; e < ct * N; e += GP_THREADS) {
        const float v = s_rows[e];
        if (v != 0.f) atomicAdd(dst + e, v);
      }
    } else {
      for (int e = tid; e < ct * N; e += GP_THREADS) dst[e] = s_rows[e];
    }
  }
}

// channel-tile / chunk heuristics shared by forward and backward
struct GroupPlan {
  bool staged;
  int CT, chunk, nchunks;
  size_t smem;
};

// esz: bytes per staged element (the forward stages rows of its storage type, the backward fp32 accumulators)
static GroupPlan plan_group(int B, int C, int N, int S, bool backward, size_t esz) {
  GroupPlan g;
  const size_t row = (size_t)N * esz;
  const size_t budget = 200 * 1024;
  g.staged = row <= budget && N > 0;
  if (!g.staged) {
    g.CT = 4;
    g.smem = 0;
  } else {
    // rows per CTA: as many as fit in ~64 KB (several CTAs/SM) but at least one
    int ct = (int)((64 * 1024) / row);
    if (ct < 1) ct = 1;
    if (ct > C) ct = C;
    if (ct > 16) ct = 16;
    g.CT = ct;
    g.smem = (size_t)ct * row;
  }
  const int ctiles = ceil_div(C, g.CT);
  // split the position range until the grid has ~2 waves, but keep chunks >= 4096 positions so
  // that the per-CTA row staging is amortised
  int nchunks = 1;
  const long long want = 2LL * kNumSMs;
  while ((long long)B * ctiles * nchunks < want && S / (nchunks * 2) >= 4096) nchunks *= 2;
  if (backward && !g.staged) nchunks = max(nchunks, 1);
  int chunk = ceil_div(S, nchunks);
  chunk = (chunk + 3) & ~3;
  g.chunk = chunk;
  g.nchunks = ceil_div(S, chunk);
  return g;
}

// ----------------------------------------------------------------------------------------------
// group_points backward, atomic-free formulation (used when the caller provides a workspace)
// ----------------------------------------------------------------------------------------------
// Shared-memory fp32 atomicAdd is a compare-and-swap loop (ATOMS.CAST.SPIN), and the ball-query
// padding makes a few low-index points the target of a large share of all positions, so the
// accumulator kernel above runs at 2-6 % of HBM bandwidth.  Here the index tensor is inverted once
// per call into a CSR list (point -> positions that reference it, ascending) that all C channels
// share, and the scatter becomes a gather:
//    grad_points[b,c,i] = sum over t in list(b,i) of grad_out[b,c,t]
// A CTA stages CT rows of grad_out (one position partition of <= 24576 floats each) in shared memory
// with one bulk-TMA copy, then every thread sums the short lists of its points from shared memory and
// whole warps share the long ones (lane-strided + butterfly).  No floating-point atomics, coalesced
// 16-bit list reads, and the summation order is fixed by the list => bit-reproducible results when
// the position range fits one or two partitions (two partial sums commute); with more partitions the
// <= H partial sums per element are combined with global RED in arbitrary order.
constexpr int GG_THREADS = 512;
constexpr int GG_PART_MAX = 24576;   // positions per partition: 96 KB of fp32 => two CTAs per SM
constexpr int GG_CT_MAX = 4;
constexpr int GG_SHORT = 32;         // lists up to this length are summed by one thread
constexpr int GG_LONG_CAP = 2048;    // long lists per CTA handled warp-wide (overflow: one thread each)

struct GradPlan {
  int H, Sp, CT, Np;
  bool lists_smem;
  size_t smem;
};

// esz: bytes per staged grad_out element (rows of the storage type)
static GradPlan plan_group_grad(int C, int N, int S, size_t esz) {
  GradPlan g;
  g.H = ceil_div(S, GG_PART_MAX);
  g.Sp = ((ceil_div(S, g.H) + 7) / 8) * 8;     // multiples of 8 keep the uint16 lists 16-byte aligned
  g.H = ceil_div(S, g.Sp);
  g.Np = ((N + 1 + 3) / 4) * 4;                // offsets row stride (16-byte aligned rows)
  int ct = (int)((64 * 1024) / ((size_t)g.Sp * esz));
  g.CT = max(1, min(min(ct, GG_CT_MAX), C));
  const size_t rows = (size_t)g.CT * g.Sp * esz;
  const size_t lists = (size_t)g.Sp * sizeof(uint16_t) + (size_t)g.Np * sizeof(int);
  g.lists_smem = rows + lists <= 112 * 1024;   // still two CTAs per SM
  g.smem = rows + (g.lists_smem ? lists : 0);
  return g;
}

// in-place inclusive scan of offsets[r][1..N]  (one CTA per offsets row r)
__global__ void __launch_bounds__(1024) gg_scan_kernel(int N, int Np, int *__restrict__ offsets) {
  __shared__ int s_part[32];
  int *row = offsets + (size_t)blockIdx.x * Np + 1;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (N + 1023) / 1024;
  const int e0 = min(N, tid * per), e1 = min(N, e0 + per);
  int sum = 0;
  for (int e = e0; e < e1; ++e) sum += row[e];
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_part[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int v = s_part[lane];
    int inc2 = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += u; }
    s_part[lane] = inc2 - v;
  }
  __syncthreads();
  int run = s_part[warp] + incl - sum;
  for (int e = e0; e < e1; ++e) { run += row[e]; row[e] = run; }
}

// ----------------------------------------------------------------------------------------------
// List build (N <= 8192): histogram + scan + a TWO-LEVEL stable counting sort in ONE kernel per (scene, partition).
//   A. the positions are first bucketed by key >> 5 (<= 256 buckets): warp w walks its contiguous chunk of
//      positions, counts per bucket (match.any, no atomics: a row of counters per warp), the counters are
//      turned into start offsets (bucket b starts where the list of key 32b starts, then warp by warp), and
//      a second walk in the same order scatters the positions => stable;
//   B. one warp per bucket orders its (short) region by the low 5 key bits with per-key cursors, again in
//      position order => every list ascending, so group_points_grad_csr_kernel sums each list in a fixed order.
// Work: 2 x Sp/32 + Sp/32 + N/32 warp iterations per partition.  A warp per 32 points scanning all Sp positions
// (N/32 x Sp/32 warp iterations) took 43 us at the SA2 shape, a third of the whole backward.
// ----------------------------------------------------------------------------------------------
constexpr int GB_THREADS = 1024;
constexpr int GB_MAX_N = 8192;

static constexpr size_t gg_build_smem(int N, int Sp, int Np) {
  const int nbk = (N + 31) >> 5;
  return (size_t)Sp * sizeof(int) + (size_t)Np * sizeof(int) + (size_t)32 * nbk * sizeof(int) +
         (size_t)Sp * sizeof(uint16_t) + 16;
}
// plan_group_grad keeps Sp <= GG_PART_MAX, so every N <= GB_MAX_N fits one CTA
static_assert(gg_build_smem(GB_MAX_N, GG_PART_MAX, (GB_MAX_N + 1 + 3) / 4 * 4) <= 220 * 1024,
              "gg_build_kernel's shared memory must fit at every N <= GB_MAX_N");

__global__ void __launch_bounds__(GB_THREADS) gg_build_kernel(const int32_t *__restrict__ idx, int N, int S, int Sp,
                                                              int H, int Np, int *__restrict__ offsets,
                                                              uint16_t *__restrict__ order) {
  extern __shared__ __align__(128) int gb_smem[];
  __shared__ int s_part[32];
  __shared__ int s_cur[32][32];
  __shared__ __align__(8) uint64_t bar;
  const int h = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int p0 = h * Sp, len = min(S, p0 + Sp) - p0;
  const int NBK = (N + 31) >> 5;
  int *s_idx = gb_smem;                 // [Sp]
  int *s_off = s_idx + Sp;              // [Np]  histogram, then exclusive offsets (slot i = start of list i)
  int *s_cnt = s_off + Np;              // [32 warps][NBK]
  uint16_t *s_bk = reinterpret_cast<uint16_t *>(s_cnt + 32 * NBK);   // [Sp] positions grouped by bucket
  const int32_t *ix = idx + (size_t)b * S + p0;
  const bool bulk_ok = ((reinterpret_cast<uintptr_t>(ix) & 15) == 0) && (len % 4 == 0);
  if (bulk_ok) {
    if (tid == 0) { mbarrier_init(&bar, 1); fence_mbarrier_init(); }
    __syncthreads();
    if (tid == 0) {
      mbarrier_arrive_expect_tx(&bar, (unsigned)(len * sizeof(int)));
      bulk_g2s(s_idx, ix, (unsigned)(len * sizeof(int)), &bar);
    }
  } else {
    for (int e = tid; e < len; e += GB_THREADS) s_idx[e] = __ldg(ix + e);
  }
  for (int e = tid; e < Np; e += GB_THREADS) s_off[e] = 0;
  for (int e = tid; e < 32 * NBK; e += GB_THREADS) s_cnt[e] = 0;
  if (bulk_ok) mbarrier_wait(&bar, 0);
  __syncthreads();
  // ---- histogram and scan: s_off[i] = number of positions with key < i ---------------------------------
  for (int t = tid; t < len; t += GB_THREADS) {
    const int k = s_idx[t];
    if ((unsigned)k < (unsigned)N) atomicAdd(&s_off[1 + k], 1);
  }
  __syncthreads();
  {
    int *row = s_off + 1;
    const int per = (N + GB_THREADS - 1) / GB_THREADS;
    const int e0 = min(N, tid * per), e1 = min(N, e0 + per);
    int sum = 0;
    for (int e = e0; e < e1; ++e) sum += row[e];
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_part[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      const int v = s_part[lane];
      int inc2 = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += u; }
      s_part[lane] = inc2 - v;
    }
    __syncthreads();
    int run = s_part[warp] + incl - sum;
    for (int e = e0; e < e1; ++e) { run += row[e]; row[e] = run; }
  }
  __syncthreads();
  int *off_g = offsets + ((size_t)b * H + h) * Np;
  for (int e = tid; e < Np; e += GB_THREADS) off_g[e] = e <= N ? s_off[e] : 0;
  // ---- A: stable bucketing by key >> 5 ---------------------------------------------------------------
  const int CH = (((len + 31) / 32 + 31) / 32) * 32;     // positions per warp, a multiple of 32
  const int c0 = min(len, warp * CH), c1 = min(len, c0 + CH);
  int *cw = s_cnt + warp * NBK;
  const unsigned lt = (1u << lane) - 1u;
  for (int t0 = c0; t0 < c1; t0 += 32) {
    const int t = t0 + lane;
    const int k = t < c1 ? s_idx[t] : -1;
    const bool valid = (unsigned)k < (unsigned)N;
    const int bkt = k >> 5;
    const unsigned peers = __match_any_sync(0xffffffffu, valid ? bkt : NBK + lane);
    if (valid && (peers & lt) == 0u) cw[bkt] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  for (int bk = tid; bk < NBK; bk += GB_THREADS) {
    int run = s_off[32 * bk];
    for (int w = 0; w < 32; ++w) { const int c = s_cnt[w * NBK + bk]; s_cnt[w * NBK + bk] = run; run += c; }
  }
  __syncthreads();
  for (int t0 = c0; t0 < c1; t0 += 32) {
    const int t = t0 + lane;
    const int k = t < c1 ? s_idx[t] : -1;
    const bool valid = (unsigned)k < (unsigned)N;
    const int bkt = k >> 5;
    const unsigned peers = __match_any_sync(0xffffffffu, valid ? bkt : NBK + lane);
    const int base = valid ? cw[bkt] : 0;
    __syncwarp();
    if (valid) {
      const unsigned before = peers & lt;
      s_bk[base + __popc(before)] = (uint16_t)t;
      if (before == 0u) cw[bkt] = base + __popc(peers);
    }
    __syncwarp();
  }
  __syncthreads();
  // ---- B: one warp per bucket, stable by the low five key bits ----------------------------------------
  uint16_t *ord = order + (size_t)b * S + p0;
  for (int bk = warp; bk < NBK; bk += 32) {
    const int k0 = 32 * bk;
    const int r0 = s_off[k0], r1 = s_off[min(N, k0 + 32)];
    s_cur[warp][lane] = (k0 + lane < N) ? s_off[k0 + lane] : 0;
    __syncwarp();
    for (int e0 = r0; e0 < r1; e0 += 32) {
      const int e = e0 + lane;
      const bool valid = e < r1;
      const int pos = valid ? (int)s_bk[e] : 0;
      const int kl = valid ? (s_idx[pos] & 31) : 0;
      const unsigned peers = __match_any_sync(0xffffffffu, valid ? kl : 32 + lane);
      const int base = valid ? s_cur[warp][kl] : 0;
      __syncwarp();
      if (valid) {
        const unsigned before = peers & lt;
        ord[base + __popc(before)] = (uint16_t)pos;
        if (before == 0u) s_cur[warp][kl] = base + __popc(peers);
      }
      __syncwarp();
    }
    __syncwarp();
  }
}

template <class T, int CT, bool LISTS_SMEM>
__global__ void __launch_bounds__(GG_THREADS) group_points_grad_csr_kernel(
    const T *__restrict__ grad_out, const int *__restrict__ offsets, const uint16_t *__restrict__ order,
    int C, int N, int S, int Sp, int H, int Np, float *__restrict__ grad_points) {
  extern __shared__ __align__(128) float s_smem[];
  T *s_rows = reinterpret_cast<T *>(s_smem);        // [CT][Sp] (+ uint16 [Sp] lists + int [Np] offsets)
  __shared__ __align__(8) uint64_t bar;
  __shared__ int s_long[GG_LONG_CAP];
  __shared__ int s_nlong;
  const int b = blockIdx.z, h = blockIdx.x;
  const int c0 = blockIdx.y * CT;
  const int ct = min(CT, C - c0);
  const int p0 = h * Sp;
  const int len = min(S, p0 + Sp) - p0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const T *g = grad_out + ((size_t)b * C + c0) * S + p0;
  const int *off_g = offsets + ((size_t)b * H + h) * Np;
  const uint16_t *ord_g = order + (size_t)b * S + p0;
  uint16_t *s_ord = reinterpret_cast<uint16_t *>(s_rows + (size_t)CT * Sp);
  int *s_off = reinterpret_cast<int *>(s_ord + Sp);
  if (tid == 0) s_nlong = 0;
  // ---- stage ct partial rows (row r at s_rows + r*Sp) and, if they fit, the lists --------------------
  const bool bulk_ok = ((reinterpret_cast<uintptr_t>(g) & 15) == 0) && (S % 8 == 0) && (len % 8 == 0) &&
                       ((reinterpret_cast<uintptr_t>(ord_g) & 15) == 0) && ((reinterpret_cast<uintptr_t>(off_g) & 15) == 0);
  if (bulk_ok) {
    if (tid == 0) { mbarrier_init(&bar, 1); fence_mbarrier_init(); }
    __syncthreads();
    if (tid == 0) {
      unsigned bytes = (unsigned)(ct * len * sizeof(T));
      if (LISTS_SMEM) bytes += (unsigned)(len * sizeof(uint16_t) + Np * sizeof(int));
      mbarrier_arrive_expect_tx(&bar, bytes);
      if (LISTS_SMEM) {       // lists first: they are needed first and come from L2
        bulk_g2s(s_off, off_g, (unsigned)(Np * sizeof(int)), &bar);
        bulk_g2s(s_ord, ord_g, (unsigned)(len * sizeof(uint16_t)), &bar);
      }
      for (int r = 0; r < ct; ++r) bulk_g2s(s_rows + (size_t)r * Sp, g + (size_t)r * S, (unsigned)(len * sizeof(T)), &bar);
    }
    mbarrier_wait(&bar, 0);
  } else {
    for (int r = 0; r < ct; ++r)
      for (int e = tid; e < len; e += GG_THREADS) s_rows[(size_t)r * Sp + e] = __ldg(g + (size_t)r * S + e);
    if (LISTS_SMEM) {
      for (int e = tid; e < len; e += GG_THREADS) s_ord[e] = ord_g[e];
      for (int e = tid; e <= N; e += GG_THREADS) s_off[e] = off_g[e];
    }
    __syncthreads();
  }
  const int *off = LISTS_SMEM ? s_off : off_g;
  const uint16_t *ord = LISTS_SMEM ? s_ord : ord_g;
  float *dst = grad_points + ((size_t)b * C + c0) * N;
  // ---- short lists: one thread per point ----------------------------------------------------------
  for (int i = tid; i < N; i += GG_THREADS) {
    const int o0 = off[i], o1 = off[i + 1];
    if (o1 - o0 > GG_SHORT) {
      const int q = atomicAdd(&s_nlong, 1);
      if (q < GG_LONG_CAP) { s_long[q] = i; continue; }
    }
    float acc[CT];
#pragma unroll
    for (int r = 0; r < CT; ++r) acc[r] = 0.f;
    int k = o0;
    for (; k + 4 <= o1; k += 4) {
      const int q0 = ord[k], q1 = ord[k + 1], q2 = ord[k + 2], q3 = ord[k + 3];
#pragma unroll
      for (int r = 0; r < CT; ++r) {
        const T *row = s_rows + (size_t)r * Sp;
        acc[r] = ((acc[r] + to_f32(row[q0])) + to_f32(row[q1])) + to_f32(row[q2]);
        acc[r] += to_f32(row[q3]);
      }
    }
    for (; k < o1; ++k) {
      const int q0 = ord[k];
#pragma unroll
      for (int r = 0; r < CT; ++r) acc[r] += to_f32(s_rows[(size_t)r * Sp + q0]);
    }
#pragma unroll
    for (int r = 0; r < CT; ++r) {
      if (r < ct) {
        if (H == 1) dst[(size_t)r * N + i] = acc[r];
        else if (acc[r] != 0.f) atomicAdd(dst + (size_t)r * N + i, acc[r]);
      }
    }
  }
  __syncthreads();
  // ---- long lists: one warp per point ---------------------------------------------------------------
  const int nlong = min(s_nlong, GG_LONG_CAP);
  for (int q = warp; q < nlong; q += GG_THREADS / 32) {
    const int i = s_long[q];
    const int o0 = off[i], o1 = off[i + 1];
    float acc[CT];
#pragma unroll
    for (int r = 0; r < CT; ++r) acc[r] = 0.f;
    for (int k = o0 + lane; k < o1; k += 32) {
      const int qq = ord[k];
#pragma unroll
      for (int r = 0; r < CT; ++r) acc[r] += to_f32(s_rows[(size_t)r * Sp + qq]);
    }
#pragma unroll
    for (int r = 0; r < CT; ++r)
#pragma unroll
      for (int o = 16; o; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < CT; ++r) {
        if (r < ct) {
          if (H == 1) dst[(size_t)r * N + i] = acc[r];
          else if (acc[r] != 0.f) atomicAdd(dst + (size_t)r * N + i, acc[r]);
        }
      }
    }
  }
}

template <int CT, bool LISTS_SMEM, class T>
static int launch_group_grad_csr(const T *grad_out, const int *offsets, const uint16_t *order, int B, int C,
                                 int N, int S, const GradPlan &g, float *grad_points, cudaStream_t stream) {
  auto kern = group_points_grad_csr_kernel<T, CT, LISTS_SMEM>;
  if (g.smem > 40 * 1024)
    SPC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
  dim3 grid(g.H, ceil_div(C, CT), B);
  kern<<<grid, GG_THREADS, g.smem, stream>>>(grad_out, offsets, order, C, N, S, g.Sp, g.H, g.Np, grad_points);
  SPC_LAUNCH_CHECK("group_points_grad_csr_kernel");
  return SPC_OK;
}

// ----------------------------------------------------------------------------------------------
// group_points backward (reference group_points_gpu.cu:43-75: one atomicAdd per element), large clouds
// (N > 8192: the input level of the detector, e.g. C = 132 multiview features over 40 k points).
// Staging position partitions does not pay here: a partition of <= 24 576 positions touches a small, different
// subset of the N points, so every (channel, partition) CTA walked all N offsets for a few thousand hits and
// combined its partial sums with global atomics (2.45 ms for 727 MB at C = 132, 4.5 % of HBM, round 1).
// Point-owned gather instead: ONE list per point over all positions (32-bit positions, built with warp-aggregated
// atomic cursors: three launches of a few microseconds; the order inside a list is not deterministic, the sum is
// within fp32 rounding), a thread owns a point and CT = 8 channels, reads its positions once and gathers the 8
// rows of grad_out straight from global memory (each row is read exactly once overall; it stays in L2 while the
// CTAs of its (scene, channel tile) run), and writes its 8 results with coalesced stores.  No floating-point
// atomics, no memset.
// ----------------------------------------------------------------------------------------------
constexpr int GL_THREADS = 256;
constexpr int GL_CT = 8;
constexpr int GL_LONG = 48;          // lists longer than this are summed by a whole warp
constexpr int GL_LONG_CAP = 256;

// counts[b][1 + idx[b,t]] += 1, one atomic per distinct index of a warp (the ball-query padding repeats one index)
__global__ void gl_hist_kernel(const int32_t *__restrict__ idx, int N, int S, int Np, int *__restrict__ offsets) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = t < S;
  const int i = ok ? __ldg(idx + (size_t)b * S + t) : -1;
  const bool valid = ok && (unsigned)i < (unsigned)N;
  const unsigned peers = __match_any_sync(0xffffffffu, valid ? i : -1 - (int)lane_id());
  if (valid && (peers & ((1u << lane_id()) - 1u)) == 0u) atomicAdd(offsets + (size_t)b * Np + 1 + i, __popc(peers));
}

// order[b][offsets[b][i] + k] = k-th position (in arrival order) that references point i
__global__ void gl_fill_kernel(const int32_t *__restrict__ idx, int N, int S, int Np, const int *__restrict__ offsets,
                               int *__restrict__ cursor, int32_t *__restrict__ order) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const bool ok = t < S;
  const int i = ok ? __ldg(idx + (size_t)b * S + t) : -1;
  const bool valid = ok && (unsigned)i < (unsigned)N;
  const unsigned lane = lane_id();
  const unsigned peers = __match_any_sync(0xffffffffu, valid ? i : -1 - (int)lane);
  const unsigned before = peers & ((1u << lane) - 1u);
  int base = 0;
  if (valid && before == 0u) base = atomicAdd(cursor + (size_t)b * Np + i, __popc(peers));
  base = __shfl_sync(0xffffffffu, base, __ffs(peers) - 1);
  if (valid) order[(size_t)b * S + __ldg(offsets + (size_t)b * Np + i) + base + __popc(before)] = t;
}

template <class T>
__global__ void __launch_bounds__(GL_THREADS) group_points_grad_gather_kernel(
    const T *__restrict__ grad_out, const int *__restrict__ offsets, const int32_t *__restrict__ order, int C,
    int N, int S, int Np, float *__restrict__ grad_points) {
  __shared__ int s_long[GL_LONG_CAP];
  __shared__ int s_nlong;
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * GL_CT;
  const int ct = min(GL_CT, C - c0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int i = blockIdx.x * GL_THREADS + tid;
  const T *g = grad_out + ((size_t)b * C + c0) * S;
  const int *off = offsets + (size_t)b * Np;
  const int32_t *ord = order + (size_t)b * S;
  float *dst = grad_points + ((size_t)b * C + c0) * N;
  if (tid == 0) s_nlong = 0;
  __syncthreads();
  if (i < N) {
    const int o0 = __ldg(off + i), o1 = __ldg(off + i + 1);
    bool mine = true;
    if (o1 - o0 > GL_LONG) {
      const int q = atomicAdd(&s_nlong, 1);
      if (q < GL_LONG_CAP) { s_long[q] = i; mine = false; }
    }
    if (mine) {
      float acc[GL_CT];
#pragma unroll
      for (int r = 0; r < GL_CT; ++r) acc[r] = 0.f;
      int k = o0;
      for (; k + 2 <= o1; k += 2) {                      // two positions x 8 rows = 16 independent loads in flight
        const int q0 = __ldg(ord + k), q1 = __ldg(ord + k + 1);
        float v0[GL_CT], v1[GL_CT];
#pragma unroll
        for (int r = 0; r < GL_CT; ++r) {
          v0[r] = r < ct ? to_f32(__ldg(g + (size_t)r * S + q0)) : 0.f;
          v1[r] = r < ct ? to_f32(__ldg(g + (size_t)r * S + q1)) : 0.f;
        }
#pragma unroll
        for (int r = 0; r < GL_CT; ++r) acc[r] = (acc[r] + v0[r]) + v1[r];
      }
      if (k < o1) {
        const int q0 = __ldg(ord + k);
#pragma unroll
        for (int r = 0; r < GL_CT; ++r) acc[r] += r < ct ? to_f32(__ldg(g + (size_t)r * S + q0)) : 0.f;
      }
#pragma unroll
      for (int r = 0; r < GL_CT; ++r)
        if (r < ct) dst[(size_t)r * N + i] = acc[r];
    }
  }
  __syncthreads();
  // ---- long lists (hubs of the ball-query padding): one warp per point ---------------------------------------
  const int nlong = min(s_nlong, GL_LONG_CAP);
  for (int q = warp; q < nlong; q += GL_THREADS / 32) {
    const int pi = s_long[q];
    const int o0 = __ldg(off + pi), o1 = __ldg(off + pi + 1);
    float acc[GL_CT];
#pragma unroll
    for (int r = 0; r < GL_CT; ++r) acc[r] = 0.f;
    for (int k = o0 + lane; k < o1; k += 32) {
      const int qq = __ldg(ord + k);
#pragma unroll
      for (int r = 0; r < GL_CT; ++r) acc[r] += r < ct ? to_f32(__ldg(g + (size_t)r * S + qq)) : 0.f;
    }
#pragma unroll
    for (int r = 0; r < GL_CT; ++r)
#pragma unroll
      for (int o = 16; o; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < GL_CT; ++r)
        if (r < ct) dst[(size_t)r * N + pi] = acc[r];
    }
  }
}

// workspace of the large-cloud path: offsets (B, Np) + cursors (B, Np) + order (B, S), all int32
static size_t gl_workspace_bytes(int B, int N, long long S) {
  const size_t Np = ((size_t)N + 1 + 3) / 4 * 4;
  return 2 * (size_t)B * Np * sizeof(int) + (size_t)B * (size_t)S * sizeof(int32_t);
}

}  // namespace spc

using namespace spc;

extern "C" int spc_gather_points(const float *points, const int32_t *idx, int B, int C, int N,
                                 int M, float *out, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && M >= 0, "gather_points: bad sizes");
  if (B == 0 || C == 0 || M == 0) return SPC_OK;
  SPC_CHECK_ARG(points && idx && out, "gather_points: null pointer");
  SPC_CHECK_ARG(B <= 65535, "gather_points: B too large");
  dim3 grid(ceil_div(M, 256), min(C, 64), B);
  gather_points_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>(points, idx, C, N, M, out);
  SPC_LAUNCH_CHECK("gather_points_kernel");
  return SPC_OK;
}

extern "C" int spc_gather_points_grad(const float *grad_out, const int32_t *idx, int B, int C,
                                      int N, int M, float *grad_points, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && M >= 0, "gather_points_grad: bad sizes");
  if (B == 0 || C == 0 || N == 0) return SPC_OK;
  SPC_CHECK_ARG(grad_points && (M == 0 || (grad_out && idx)), "gather_points_grad: null pointer");
  SPC_CHECK_ARG(B <= 65535, "gather_points_grad: B too large");
  cudaStream_t stream = (cudaStream_t)stream_;
  SPC_CUDA(cudaMemsetAsync(grad_points, 0, (size_t)B * C * N * sizeof(float), stream));
  if (M == 0) return SPC_OK;
  dim3 grid(ceil_div(M, 256), min(C, 64), B);
  gather_points_grad_kernel<<<grid, 256, 0, stream>>>(grad_out, idx, C, N, M, grad_points);
  SPC_LAUNCH_CHECK("gather_points_grad_kernel");
  return SPC_OK;
}

template <class T>
static int group_points(const T *points, const int32_t *idx, int B, int C, int N, int npoint, int nsample, T *out,
                        void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && npoint >= 0 && nsample >= 0, "group_points: bad sizes");
  const long long S64 = (long long)npoint * nsample;
  SPC_CHECK_ARG(S64 < (1LL << 31), "group_points: npoint*nsample overflows int32");
  const int S = (int)S64;
  if (B == 0 || C == 0 || S == 0) return SPC_OK;
  SPC_CHECK_ARG(points && idx && out, "group_points: null pointer");
  SPC_CHECK_ARG(B <= 65535, "group_points: B too large");
  cudaStream_t stream = (cudaStream_t)stream_;
  const GroupPlan g = plan_group(B, C, N, S, false, sizeof(T));
  const bool vec4 = (S % 4 == 0) && ((reinterpret_cast<uintptr_t>(idx) & 15) == 0) &&
                    ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
  dim3 grid(g.nchunks, ceil_div(C, g.CT), B);
  SPC_CHECK_ARG(grid.y <= 65535, "group_points: too many channel tiles");
#define GP_LAUNCH(ST, V4)                                                                       \
  do {                                                                                          \
    if (g.smem > 40 * 1024)                                                                     \
      SPC_CUDA(cudaFuncSetAttribute(group_points_kernel<T, ST, V4>,                             \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem)); \
    group_points_kernel<T, ST, V4><<<grid, GP_THREADS, g.smem, stream>>>(points, idx, C, N, S,  \
                                                                         g.CT, g.chunk, out);   \
  } while (0)
  if (g.staged) { if (vec4) GP_LAUNCH(true, true); else GP_LAUNCH(true, false); }
  else { if (vec4) GP_LAUNCH(false, true); else GP_LAUNCH(false, false); }
#undef GP_LAUNCH
  SPC_LAUNCH_CHECK("group_points_kernel");
  return SPC_OK;
}

template <class T>
static int group_points_grad(const T *grad_out, const int32_t *idx, int B, int C, int N, int npoint, int nsample,
                             float *grad_points, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && npoint >= 0 && nsample >= 0, "group_points_grad: bad sizes");
  const long long S64 = (long long)npoint * nsample;
  SPC_CHECK_ARG(S64 < (1LL << 31), "group_points_grad: npoint*nsample overflows int32");
  const int S = (int)S64;
  if (B == 0 || C == 0 || N == 0) return SPC_OK;
  SPC_CHECK_ARG(grad_points && (S == 0 || (grad_out && idx)), "group_points_grad: null pointer");
  SPC_CHECK_ARG(B <= 65535, "group_points_grad: B too large");
  cudaStream_t stream = (cudaStream_t)stream_;
  if (S == 0) {
    SPC_CUDA(cudaMemsetAsync(grad_points, 0, (size_t)B * C * N * sizeof(float), stream));
    return SPC_OK;
  }
  const GroupPlan g = plan_group(B, C, N, S, true, sizeof(float));
  const int global_atomics = (!g.staged || g.nchunks > 1) ? 1 : 0;
  if (global_atomics)
    SPC_CUDA(cudaMemsetAsync(grad_points, 0, (size_t)B * C * N * sizeof(float), stream));
  dim3 grid(g.nchunks, ceil_div(C, g.CT), B);
  SPC_CHECK_ARG(grid.y <= 65535, "group_points_grad: too many channel tiles");
  if (g.staged) {
    if (g.smem > 40 * 1024)
      SPC_CUDA(cudaFuncSetAttribute(group_points_grad_kernel<T, true>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
    group_points_grad_kernel<T, true><<<grid, GP_THREADS, g.smem, stream>>>(
        grad_out, idx, C, N, S, g.CT, g.chunk, global_atomics, grad_points);
  } else {
    group_points_grad_kernel<T, false><<<grid, GP_THREADS, 0, stream>>>(
        grad_out, idx, C, N, S, g.CT, g.chunk, 1, grad_points);
  }
  SPC_LAUNCH_CHECK("group_points_grad_kernel");
  return SPC_OK;
}

extern "C" size_t spc_group_points_grad_workspace_bytes(int B, int N, int npoint, int nsample) {
  if (B <= 0 || N <= 0 || npoint <= 0 || nsample <= 0) return 0;
  const long long S = (long long)npoint * nsample;
  if (S >= (1LL << 31)) return 0;
  if (N > GB_MAX_N) return gl_workspace_bytes(B, N, S);
  const GradPlan g = plan_group_grad(1, N, (int)S, sizeof(float));   // H and Np do not depend on the element size
  // offsets (B,H,Np) int32  +  order (B,S) uint16, both starting 16-byte aligned
  return (size_t)B * g.H * (size_t)g.Np * sizeof(int) + (((size_t)B * (size_t)S * sizeof(uint16_t) + 15) & ~(size_t)15);
}

template <class T>
static int group_points_grad_ex(const T *grad_out, const int32_t *idx, int B, int C, int N, int npoint, int nsample,
                                float *grad_points, void *workspace, size_t workspace_bytes, void *stream_) {
  SPC_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && npoint >= 0 && nsample >= 0, "group_points_grad: bad sizes");
  const long long S64 = (long long)npoint * nsample;
  SPC_CHECK_ARG(S64 < (1LL << 31), "group_points_grad: npoint*nsample overflows int32");
  const int S = (int)S64;
  const size_t need = spc_group_points_grad_workspace_bytes(B, N, npoint, nsample);
  // The list build is shared by all C channels: worth it once C is a few channels (SA2-SA4, vote aggregation,
  // every input level with features); with fewer the atomic kernel is faster.
  if (!workspace || need == 0 || workspace_bytes < need || (reinterpret_cast<uintptr_t>(workspace) & 15) || C < 4 ||
      (N <= GB_MAX_N && (long long)N > 512LL * C) || B == 0 || B > 65535)
    return group_points_grad(grad_out, idx, B, C, N, npoint, nsample, grad_points, stream_);
  SPC_CHECK_ARG(grad_points && grad_out && idx, "group_points_grad: null pointer");
  cudaStream_t stream = (cudaStream_t)stream_;
  if (N > GB_MAX_N) {
    // large cloud: one list per point over all positions, point-owned gather (see group_points_grad_gather_kernel)
    const size_t Np = ((size_t)N + 1 + 3) / 4 * 4;
    int *offsets = reinterpret_cast<int *>(workspace);
    int *cursor = offsets + (size_t)B * Np;
    int32_t *order = cursor + (size_t)B * Np;
    SPC_CUDA(cudaMemsetAsync(offsets, 0, 2 * (size_t)B * Np * sizeof(int), stream));
    gl_hist_kernel<<<dim3(ceil_div(S, 256), B), 256, 0, stream>>>(idx, N, S, (int)Np, offsets);
    gg_scan_kernel<<<B, 1024, 0, stream>>>(N, (int)Np, offsets);
    gl_fill_kernel<<<dim3(ceil_div(S, 256), B), 256, 0, stream>>>(idx, N, S, (int)Np, offsets, cursor, order);
    SPC_LAUNCH_CHECK("group_points_grad list build (large cloud)");
    SPC_CHECK_ARG(ceil_div(C, GL_CT) <= 65535, "group_points_grad: too many channel tiles");
    group_points_grad_gather_kernel<<<dim3(ceil_div(N, GL_THREADS), ceil_div(C, GL_CT), B), GL_THREADS, 0, stream>>>(
        grad_out, offsets, order, C, N, S, (int)Np, grad_points);
    SPC_LAUNCH_CHECK("group_points_grad_gather_kernel");
    return SPC_OK;
  }
  const GradPlan g = plan_group_grad(C, N, S, sizeof(T));
  SPC_CHECK_ARG(ceil_div(C, g.CT) <= 65535 && g.H <= 65535, "group_points_grad: grid too large");
  int *offsets = reinterpret_cast<int *>(workspace);
  const size_t off_bytes = (size_t)B * g.H * (size_t)g.Np * sizeof(int);
  uint16_t *order = reinterpret_cast<uint16_t *>(reinterpret_cast<char *>(workspace) + off_bytes);
  // histogram + scan + two-level stable sort in one kernel per (scene, partition)
  const size_t build_smem = gg_build_smem(N, g.Sp, g.Np);
  SPC_CUDA(cudaFuncSetAttribute(gg_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)build_smem));
  gg_build_kernel<<<dim3(g.H, B), GB_THREADS, build_smem, stream>>>(idx, N, S, g.Sp, g.H, g.Np, offsets, order);
  SPC_LAUNCH_CHECK("group_points_grad list build");
  if (g.H > 1) SPC_CUDA(cudaMemsetAsync(grad_points, 0, (size_t)B * C * N * sizeof(float), stream));
#define GG_CASE(ct)                                                                                              \
  case ct:                                                                                                       \
    return g.lists_smem ? launch_group_grad_csr<ct, true>(grad_out, offsets, order, B, C, N, S, g, grad_points, stream) \
                        : launch_group_grad_csr<ct, false>(grad_out, offsets, order, B, C, N, S, g, grad_points, stream);
  switch (g.CT) {
    GG_CASE(1) GG_CASE(2) GG_CASE(3)
    default:
      return g.lists_smem ? launch_group_grad_csr<4, true>(grad_out, offsets, order, B, C, N, S, g, grad_points, stream)
                          : launch_group_grad_csr<4, false>(grad_out, offsets, order, B, C, N, S, g, grad_points, stream);
  }
#undef GG_CASE
}

// ---- C entry points: fp32 storage, and bf16 storage (points / out / grad_out are __nv_bfloat16 tensors) ------------
extern "C" int spc_group_points(const float *points, const int32_t *idx, int B, int C, int N,
                                int npoint, int nsample, float *out, void *stream) {
  return group_points(points, idx, B, C, N, npoint, nsample, out, stream);
}
extern "C" int spc_group_points_bf16(const void *points, const int32_t *idx, int B, int C, int N,
                                     int npoint, int nsample, void *out, void *stream) {
  return group_points(static_cast<const bf16 *>(points), idx, B, C, N, npoint, nsample, static_cast<bf16 *>(out),
                      stream);
}

extern "C" int spc_group_points_grad(const float *grad_out, const int32_t *idx, int B, int C,
                                     int N, int npoint, int nsample, float *grad_points,
                                     void *stream) {
  return group_points_grad(grad_out, idx, B, C, N, npoint, nsample, grad_points, stream);
}
extern "C" int spc_group_points_grad_bf16(const void *grad_out, const int32_t *idx, int B, int C,
                                          int N, int npoint, int nsample, float *grad_points,
                                          void *stream) {
  return group_points_grad(static_cast<const bf16 *>(grad_out), idx, B, C, N, npoint, nsample, grad_points, stream);
}

extern "C" int spc_group_points_grad_ex(const float *grad_out, const int32_t *idx, int B, int C, int N, int npoint,
                                        int nsample, float *grad_points, void *workspace, size_t workspace_bytes,
                                        void *stream) {
  return group_points_grad_ex(grad_out, idx, B, C, N, npoint, nsample, grad_points, workspace, workspace_bytes, stream);
}
extern "C" int spc_group_points_grad_ex_bf16(const void *grad_out, const int32_t *idx, int B, int C, int N, int npoint,
                                             int nsample, float *grad_points, void *workspace, size_t workspace_bytes,
                                             void *stream) {
  return group_points_grad_ex(static_cast<const bf16 *>(grad_out), idx, B, C, N, npoint, nsample, grad_points,
                              workspace, workspace_bytes, stream);
}
