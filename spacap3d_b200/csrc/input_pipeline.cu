// input_pipeline.cu -- device side of the training / evaluation input pipeline (SURVEY row N4; reference
// lib/dataset.py:291-531 `ScannetReferenceDataset.__getitem__`, which runs in numpy on DataLoader workers).
//
// The B200-first design keeps the WHOLE pre-processed ScanNet set resident in HBM (1 201 train scenes x 50 k vertices
// x 9 floats = 2.2 GB; with the 128-d multiview features 30 GB of the 180 GB) as one packed vertex table, so that a
// batch is assembled by three kernels instead of per-item numpy work + h5py reads (the reference's README blames the
// multiview fetch for +6 h of training, README.md:187-191):
//   * spc_scene_floor_height   : np.percentile(z, 0.99) of one scene (lib/dataset.py:331) -- once per scene, cached;
//   * spc_prepare_point_clouds : row gather by the sampled indices + colour normalisation + height channel +
//                                flips / three rotations / translation (lib/dataset.py:309-335, 366-404);
//   * spc_vote_labels          : per-instance bounding-box centres of the SAMPLED, AUGMENTED cloud and the vote
//                                targets (lib/dataset.py:421-431);
//   * spc_augment_boxes        : the same flips / rotations / translation applied to the axis-aligned GT boxes
//                                (lib/dataset.py:369-404, data/scannet/model_util_scannet.py:47-82).
// Random draws stay on the host (spacap3d_b200/input_pipeline.py restates the reference's np.random call order), so a
// seed gives the batch the reference's __getitem__ would give.  Arithmetic follows numpy's dtypes: the cloud is float32
// between steps, every product with a (float64) rotation matrix / mean colour / translation is evaluated in float64
// and rounded to float32 on assignment.
#include "common.cuh"
#include "ptx.cuh"

namespace spc {

// ------------------------------------------------------------------------------------------------------------------
// floor height = np.percentile(col, q) with numpy >= 2.0 float32 semantics (the quantile arrives as float32 q/100,
// the virtual index, gamma and the lerp are float32; numpy/lib/_function_base_impl.py `_quantile`, `_lerp`).
// One CTA: 4-pass 8-bit radix select of the order statistic i = floor((M-1)*q), then the next one.
// ------------------------------------------------------------------------------------------------------------------
constexpr int FH_THREADS = 1024;

__device__ __forceinline__ uint32_t float_key(float f) {            // monotone float -> uint32
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

__global__ void __launch_bounds__(FH_THREADS) floor_height_kernel(const float *__restrict__ verts, int M, int stride,
                                                                  int col, float quantile, float *__restrict__ out) {
  __shared__ unsigned s_hist[256];
  __shared__ unsigned s_prefix, s_rank, s_count_eq, s_next;
  const float v = __fmul_rn((float)(M - 1), quantile);               // (n - 1) * quantiles, float32
  const float fl = floorf(v);
  int i0 = (int)fl;
  float t = __fsub_rn(v, fl);                                        // gamma
  if (v >= (float)(M - 1)) { i0 = M - 1; }                           // _get_indexes: above bounds -> last element
  if (v < 0.f) { i0 = 0; }
  if (threadIdx.x == 0) { s_prefix = 0; s_rank = (unsigned)i0; }
  __syncthreads();
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    if (threadIdx.x < 256) s_hist[threadIdx.x] = 0;
    __syncthreads();
    const unsigned prefix = s_prefix;
    const unsigned himask = pass == 0 ? 0u : (0xFFFFFFFFu << (shift + 8));
    for (int i = threadIdx.x; i < M; i += FH_THREADS) {
      const uint32_t k = float_key(__ldg(verts + (size_t)i * stride + col));
      if ((k & himask) == prefix) atomicAdd(&s_hist[(k >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned r = s_rank, acc = 0;
      int b = 0;
      for (; b < 256; ++b) {
        if (acc + s_hist[b] > r) break;
        acc += s_hist[b];
      }
      s_rank = r - acc;
      s_prefix = prefix | ((unsigned)b << shift);
      if (pass == 3) s_count_eq = s_hist[b];
    }
    __syncthreads();
  }
  const uint32_t ka = s_prefix;                                      // key of the i0-th smallest value
  // next order statistic: the same value if enough duplicates remain, else the smallest key above it
  if (threadIdx.x == 0) s_next = 0xFFFFFFFFu;
  __syncthreads();
  uint32_t local = 0xFFFFFFFFu;
  for (int i = threadIdx.x; i < M; i += FH_THREADS) {
    const uint32_t k = float_key(__ldg(verts + (size_t)i * stride + col));
    if (k > ka && k < local) local = k;
  }
  local = __reduce_min_sync(0xFFFFFFFFu, local);
  if (lane_id() == 0) atomicMin(&s_next, local);
  __syncthreads();
  if (threadIdx.x == 0) {
    const float a = key_float(ka);
    float b;
    if (i0 >= M - 1 || v < 0.f) b = a;                               // next index clamped like _get_indexes
    else if (s_rank + 1 < s_count_eq) b = a;
    else b = key_float(s_next);
    const float d = __fsub_rn(b, a);                                 // _lerp: a + (b-a)*t, or b - (b-a)*(1-t) for t >= 0.5
    float r = __fadd_rn(a, __fmul_rn(d, t));
    if (t >= 0.5f) r = __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.f, t)));
    out[0] = r;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// point-cloud assembly.  aug (B,32) f64 per item: [flip_x, flip_y, Rx(9), Ry(9), Rz(9), t(3)], row-major matrices as
// returned by rotx/roty/rotz (utils/pc_utils.py:282-320).
// ------------------------------------------------------------------------------------------------------------------
// rows per CTA (template): the CTA's output span (PP_ROWS x C_out floats) is staged in shared memory; 64 with multiview
// features (35 KB tiles, 6 CTAs / SM), 256 without (one thread per row in phase 1)
constexpr int PP_THREADS = 256;

struct PrepArgs {
  const float *verts; int vstride;
  const float *multiview; int n_mv;
  const int64_t *row0; const int32_t *choices;
  const float *floor_height; const double *aug;
  double mean_rgb[3];
  int P, use_color, use_normal, use_height, C_out;
  float *out;
};

__device__ __forceinline__ float rot_row(const double *R, float x, float y, float z) {
  // np.dot(pc[:, 0:3], rot_mat.T)[i, j] = sum_k pc[i,k] * R[j,k]: float32 promoted to float64, dgemm accumulation
  // order k = 0,1,2; rounded to float32 by the assignment into the float32 cloud (lib/dataset.py:390)
  return (float)fma((double)z, R[2], fma((double)y, R[1], (double)x * R[0]));
}

// Phase 1: one thread per row computes the <= 10 "small" channels (fp64 where numpy uses fp64) into the tile.
// Phase 2: one warp per row gathers the 4*n_mv-byte multiview row with 16-byte loads (eight rows in flight per warp).
// Phase 3: the tile -- a contiguous span of the output -- leaves with ONE bulk TMA store (cp.async.bulk.global.shared),
//          or a coalesced scalar loop when the span is not 16-byte aligned.
template <int PP_ROWS>
__global__ void __launch_bounds__(PP_THREADS) prepare_points_kernel(PrepArgs a) {
  extern __shared__ __align__(128) float s_tile[];                    // [PP_ROWS][C_out]
  __shared__ int64_t s_src[PP_ROWS];
  const int b = blockIdx.y;
  const int r0 = blockIdx.x * PP_ROWS;
  const int nrows = min(PP_ROWS, a.P - r0);
  const int t = threadIdx.x;
  const int C = a.C_out, n_mv = a.n_mv;
  const int n_pre = 3 + (a.use_color ? 3 : 0) + (a.use_normal ? 3 : 0);
  if (t < nrows) {
    const int64_t src = a.row0[b] + (int64_t)__ldg(a.choices + (size_t)b * a.P + r0 + t);
    s_src[t] = src;
    float *o = s_tile + t * C;
    const float *v = a.verts + (size_t)src * a.vstride;
    float x = __ldg(v), y = __ldg(v + 1), z = __ldg(v + 2);
    int c = 3;
    if (a.use_color) {                      // (rgb - MEAN_COLOR_RGB) / 256.0 in float64 -> float32 (dataset.py:314)
      for (int k = 0; k < 3; ++k) o[c++] = (float)(((double)__ldg(v + 3 + k) - a.mean_rgb[k]) / 256.0);
    }
    if (a.use_normal) {                     // copied as stored; the reference does not rotate normals (dataset.py:317-319)
      for (int k = 0; k < 3; ++k) o[c++] = __ldg(v + 6 + k);
    }
    if (a.use_height) o[n_pre + n_mv] = __fsub_rn(z, __ldg(a.floor_height + b));   // before augmentation (dataset.py:330-333)
    if (a.aug != nullptr) {
      const double *p = a.aug + (size_t)b * 32;
      if (p[0] != 0.0) x = -x;              // flip along the YZ plane (dataset.py:369)
      if (p[1] != 0.0) y = -y;              // flip along the XZ plane (dataset.py:379)
#pragma unroll
      for (int r = 0; r < 3; ++r) {         // rotations about x, y, z (dataset.py:388-401)
        const double *R = p + 2 + 9 * r;
        const float nx = rot_row(R, x, y, z), ny = rot_row(R + 3, x, y, z), nz = rot_row(R + 6, x, y, z);
        x = nx; y = ny; z = nz;
      }
      x = (float)((double)x + p[29]);       // coords += factor (dataset.py:240): float64 add, float32 store
      y = (float)((double)y + p[30]);
      z = (float)((double)z + p[31]);
    }
    o[0] = x; o[1] = y; o[2] = z;
  }
  __syncthreads();
  if (n_mv > 0) {
    const int warp = t >> 5, lane = t & 31;
    constexpr int NW = PP_THREADS / 32;
    const bool vec = (n_mv & 3) == 0 && ((uintptr_t)a.multiview & 15) == 0;
    if (vec) {
      const int nv = n_mv >> 2;                                       // float4 per row
      for (int q0 = lane; q0 < nv; q0 += 32) {
        float4 val[PP_ROWS / NW];
#pragma unroll
        for (int k = 0; k < PP_ROWS / NW; ++k) {
          const int row = warp + k * NW;
          if (row < nrows) val[k] = __ldcs(reinterpret_cast<const float4 *>(a.multiview + (size_t)s_src[row] * n_mv) + q0);
        }
#pragma unroll
        for (int k = 0; k < PP_ROWS / NW; ++k) {
          const int row = warp + k * NW;
          if (row < nrows) {
            float *o = s_tile + row * C + n_pre + 4 * q0;
            o[0] = val[k].x; o[1] = val[k].y; o[2] = val[k].z; o[3] = val[k].w;
          }
        }
      }
    } else {
      for (int row = warp; row < nrows; row += NW)
        for (int c = lane; c < n_mv; c += 32)
          s_tile[row * C + n_pre + c] = __ldg(a.multiview + (size_t)s_src[row] * n_mv + c);
    }
    __syncthreads();
  }
  float *o = a.out + ((size_t)b * a.P + r0) * C;
  const unsigned bytes = (unsigned)nrows * C * 4u;
  if ((((uintptr_t)o | bytes) & 15) == 0) {
    if (t == 0) {
      fence_proxy_async_smem();
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(o), "r"(s2u(s_tile)), "r"(bytes)
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the tile must outlive the copy's reads
    }
  } else {
    for (int i = t; i < nrows * C; i += PP_THREADS) __stcs(o + i, s_tile[i]);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// vote labels (dataset.py:421-431).  Per item: for every instance id present among the sampled points, the axis-aligned
// bounding box of its (augmented) points; centre = 0.5*(min+max) in float32; vote = centre - x for the points of
// instances whose FIRST sampled point carries a semantic label in `sem_mask` (DC.nyu40ids).
// ws (B, I, 8) int32: [min xyz keys, max xyz keys, first position, unused].
// ------------------------------------------------------------------------------------------------------------------
constexpr int VL_THREADS = 1024;

__device__ __forceinline__ int fkey(float f) {                       // monotone float -> signed int
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7FFFFFFF;
}
__device__ __forceinline__ float fkey_inv(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7FFFFFFF); }

__global__ void vote_init_kernel(int *__restrict__ ws, size_t n_entries) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_entries * 8) return;
  const int f = (int)(i & 7);
  ws[i] = f < 3 ? INT_MAX : (f < 6 ? INT_MIN : INT_MAX);
}

__global__ void __launch_bounds__(VL_THREADS) vote_reduce_kernel(const float *__restrict__ pc, int C, int P,
                                                                 const int32_t *__restrict__ inst_labels,
                                                                 const int64_t *__restrict__ row0,
                                                                 const int32_t *__restrict__ choices, int I,
                                                                 int *__restrict__ ws, int *__restrict__ overflow) {
  extern __shared__ int s_tab[];                                      // (I, 7)
  const int b = blockIdx.y;
  for (int i = threadIdx.x; i < I * 7; i += VL_THREADS) {
    const int f = i % 7;
    s_tab[i] = f < 3 ? INT_MAX : (f < 6 ? INT_MIN : INT_MAX);
  }
  __syncthreads();
  const int j = blockIdx.x * VL_THREADS + threadIdx.x;
  int id = -1;
  int kx = 0, ky = 0, kz = 0;
  if (j < P) {
    id = __ldg(inst_labels + row0[b] + (int64_t)__ldg(choices + (size_t)b * P + j));
    const float *p = pc + ((size_t)b * P + j) * C;
    kx = fkey(__ldg(p)); ky = fkey(__ldg(p + 1)); kz = fkey(__ldg(p + 2));
    if (id < 0 || id >= I) { if (overflow) atomicExch(overflow, 1); id = -1; }
  }
  // warp-aggregated: one shared-memory atomic per (warp, instance, field) instead of one per point -- the
  // unannotated instance 0 alone owns a third of a ScanNet scene
  unsigned todo = __ballot_sync(0xFFFFFFFFu, id >= 0);
  while (todo) {
    const int leader = __ffs(todo) - 1;
    const int gid = __shfl_sync(0xFFFFFFFFu, id, leader);
    const bool mine = (id == gid);
    const unsigned grp = __ballot_sync(0xFFFFFFFFu, mine);
    const int mnx = __reduce_min_sync(0xFFFFFFFFu, mine ? kx : INT_MAX), mxx = __reduce_max_sync(0xFFFFFFFFu, mine ? kx : INT_MIN);
    const int mny = __reduce_min_sync(0xFFFFFFFFu, mine ? ky : INT_MAX), mxy = __reduce_max_sync(0xFFFFFFFFu, mine ? ky : INT_MIN);
    const int mnz = __reduce_min_sync(0xFFFFFFFFu, mine ? kz : INT_MAX), mxz = __reduce_max_sync(0xFFFFFFFFu, mine ? kz : INT_MIN);
    const int first = __reduce_min_sync(0xFFFFFFFFu, mine ? j : INT_MAX);
    if ((int)lane_id() == leader) {
      int *e = s_tab + gid * 7;
      atomicMin(e + 0, mnx); atomicMin(e + 1, mny); atomicMin(e + 2, mnz);
      atomicMax(e + 3, mxx); atomicMax(e + 4, mxy); atomicMax(e + 5, mxz);
      atomicMin(e + 6, first);
    }
    todo &= ~grp;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < I; i += VL_THREADS) {
    const int *e = s_tab + i * 7;
    if (e[6] == INT_MAX) continue;                                    // instance absent from this CTA's points
    int *g = ws + ((size_t)b * I + i) * 8;
    atomicMin(g + 0, e[0]); atomicMin(g + 1, e[1]); atomicMin(g + 2, e[2]);
    atomicMax(g + 3, e[3]); atomicMax(g + 4, e[4]); atomicMax(g + 5, e[5]);
    atomicMin(g + 6, e[6]);
  }
}

__global__ void __launch_bounds__(256) vote_write_kernel(const float *__restrict__ pc, int C, int P,
                                                         const int32_t *__restrict__ inst_labels,
                                                         const int32_t *__restrict__ sem_labels,
                                                         const int64_t *__restrict__ row0,
                                                         const int32_t *__restrict__ choices, int I,
                                                         unsigned long long sem_mask, const int *__restrict__ ws,
                                                         float *__restrict__ vote_label,
                                                         int64_t *__restrict__ vote_mask) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= P) return;
  const int id = __ldg(inst_labels + row0[b] + (int64_t)__ldg(choices + (size_t)b * P + j));
  float vx = 0.f, vy = 0.f, vz = 0.f;
  int64_t m = 0;
  if (id >= 0 && id < I) {
    const int *g = ws + ((size_t)b * I + id) * 8;
    const int first = __ldg(g + 6);
    const int sem = __ldg(sem_labels + row0[b] + (int64_t)__ldg(choices + (size_t)b * P + first));
    if (sem >= 0 && sem < 64 && ((sem_mask >> sem) & 1ull)) {
      const float *p = pc + ((size_t)b * P + j) * C;
      // center = 0.5 * (x.min(0) + x.max(0)); point_votes = center - x      (float32 cloud => float32 arithmetic)
      const float cx = __fmul_rn(0.5f, __fadd_rn(fkey_inv(__ldg(g + 0)), fkey_inv(__ldg(g + 3))));
      const float cy = __fmul_rn(0.5f, __fadd_rn(fkey_inv(__ldg(g + 1)), fkey_inv(__ldg(g + 4))));
      const float cz = __fmul_rn(0.5f, __fadd_rn(fkey_inv(__ldg(g + 2)), fkey_inv(__ldg(g + 5))));
      vx = __fsub_rn(cx, __ldg(p)); vy = __fsub_rn(cy, __ldg(p + 1)); vz = __fsub_rn(cz, __ldg(p + 2));
      m = 1;
    }
  }
  float *o = vote_label + ((size_t)b * P + j) * 9;                    // np.tile(point_votes, (1, 3))
#pragma unroll
  for (int r = 0; r < 3; ++r) { o[3 * r] = vx; o[3 * r + 1] = vy; o[3 * r + 2] = vz; }
  vote_mask[(size_t)b * P + j] = m;
}

// ------------------------------------------------------------------------------------------------------------------
// GT box augmentation, float64 throughout (dataset.py:369-404; rotate_aligned_boxes_along_axis,
// data/scannet/model_util_scannet.py:47-82 -- including its use of the first two columns of the corner array for
// every axis).  boxes (B,K,6) = centre xyz + lengths.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double drow(const double *R, double x, double y, double z) {
  return fma(z, R[2], fma(y, R[1], x * R[0]));
}

__global__ void augment_boxes_kernel(const double *__restrict__ boxes, const double *__restrict__ aug, int B, int K,
                                     double *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * K) return;
  const int b = i / K;
  const double *p = aug + (size_t)b * 32;
  const double *s = boxes + (size_t)i * 6;
  double c[3] = {s[0], s[1], s[2]}, l[3] = {s[3], s[4], s[5]};
  if (p[0] != 0.0) c[0] = -1 * c[0];
  if (p[1] != 0.0) c[1] = -1 * c[1];
  for (int r = 0; r < 3; ++r) {
    const double *R = p + 2 + 9 * r;
    const double nc0 = drow(R, c[0], c[1], c[2]), nc1 = drow(R + 3, c[0], c[1], c[2]), nc2 = drow(R + 6, c[0], c[1], c[2]);
    c[0] = nc0; c[1] = nc1; c[2] = nc2;
    const int i1 = r == 0 ? 1 : 0, i2 = r == 2 ? 1 : 2;               // axis x: (ly, lz); y: (lx, lz); z: (lx, ly)
    const double d1 = l[i1] / 2.0, d2 = l[i2] / 2.0;
    const double sg[4][2] = {{-1, -1}, {1, -1}, {1, 1}, {-1, 1}};
    double m1 = -INFINITY, m2 = -INFINITY;
    for (int q = 0; q < 4; ++q) {
      const double a0 = sg[q][0] * d1, a1 = sg[q][1] * d2;
      m1 = fmax(m1, drow(R, a0, a1, 0.0));
      m2 = fmax(m2, drow(R + 3, a0, a1, 0.0));
    }
    l[i1] = 2.0 * m1; l[i2] = 2.0 * m2;
  }
  c[0] += p[29]; c[1] += p[30]; c[2] += p[31];
  double *o = out + (size_t)i * 6;
  o[0] = c[0]; o[1] = c[1]; o[2] = c[2]; o[3] = l[0]; o[4] = l[1]; o[5] = l[2];
}

}  // namespace spc

using namespace spc;

extern "C" int spc_scene_floor_height(const float *verts, int M, int stride, int col, float quantile, float *out,
                                      void *stream) {
  SPC_CHECK_ARG(verts && out, "spc_scene_floor_height: null pointer");
  SPC_CHECK_ARG(M >= 1 && stride >= 1 && col >= 0 && col < stride, "spc_scene_floor_height: bad M=%d stride=%d col=%d",
                M, stride, col);
  SPC_CHECK_ARG(M <= (1 << 24), "spc_scene_floor_height: M=%d exceeds 2^24 (float32 index arithmetic of numpy)", M);
  SPC_CHECK_ARG(quantile >= 0.f && quantile <= 1.f, "spc_scene_floor_height: quantile %g outside [0,1]", quantile);
  floor_height_kernel<<<1, FH_THREADS, 0, (cudaStream_t)stream>>>(verts, M, stride, col, quantile, out);
  SPC_LAUNCH_CHECK("floor_height_kernel");
  return SPC_OK;
}

extern "C" int spc_prepare_point_clouds(const float *verts, int vstride, const float *multiview, int n_mv,
                                        const int64_t *row0, const int32_t *choices, const float *floor_height,
                                        const double *aug, double mean_r, double mean_g, double mean_b, int B, int P,
                                        int use_color, int use_normal, float *out, void *stream) {
  SPC_CHECK_ARG(verts && row0 && choices && out, "spc_prepare_point_clouds: null pointer");
  SPC_CHECK_ARG(B >= 0 && P >= 0, "spc_prepare_point_clouds: bad B=%d P=%d", B, P);
  SPC_CHECK_ARG(vstride >= 3 + (use_color ? 3 : 0) && (!use_normal || vstride >= 9),
                "spc_prepare_point_clouds: vertex stride %d too small for the requested channels", vstride);
  SPC_CHECK_ARG((multiview != nullptr) == (n_mv > 0), "spc_prepare_point_clouds: multiview pointer / width mismatch");
  if (B == 0 || P == 0) return SPC_OK;
  PrepArgs a;
  a.verts = verts; a.vstride = vstride; a.multiview = multiview; a.n_mv = n_mv; a.row0 = row0; a.choices = choices;
  a.floor_height = floor_height; a.aug = aug;
  a.mean_rgb[0] = mean_r; a.mean_rgb[1] = mean_g; a.mean_rgb[2] = mean_b;
  a.P = P; a.use_color = use_color != 0; a.use_normal = use_normal != 0; a.use_height = floor_height != nullptr;
  a.C_out = 3 + (a.use_color ? 3 : 0) + (a.use_normal ? 3 : 0) + n_mv + (a.use_height ? 1 : 0);
  a.out = out;
  const int rows = n_mv > 0 ? 64 : 256;
  const size_t smem = (size_t)rows * a.C_out * sizeof(float);
  SPC_CHECK_ARG(smem <= 200 * 1024, "spc_prepare_point_clouds: %d output channels exceed the shared-memory tile", a.C_out);
  dim3 grid(ceil_div(P, rows), B);
  if (n_mv > 0) {
    if (smem > 48 * 1024)
      SPC_CUDA(cudaFuncSetAttribute(prepare_points_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    prepare_points_kernel<64><<<grid, PP_THREADS, smem, (cudaStream_t)stream>>>(a);
  } else {
    prepare_points_kernel<256><<<grid, PP_THREADS, smem, (cudaStream_t)stream>>>(a);
  }
  SPC_LAUNCH_CHECK("prepare_points_kernel");
  return SPC_OK;
}

extern "C" size_t spc_vote_labels_workspace_bytes(int B, int max_instances) {
  return (size_t)B * (size_t)max_instances * 8 * sizeof(int);
}

extern "C" int spc_vote_labels(const float *point_clouds, int C, const int32_t *instance_labels,
                               const int32_t *semantic_labels, const int64_t *row0, const int32_t *choices, int B,
                               int P, int max_instances, uint64_t sem_mask, float *vote_label,
                               int64_t *vote_label_mask, int32_t *overflow, void *workspace, size_t workspace_bytes,
                               void *stream) {
  SPC_CHECK_ARG(point_clouds && instance_labels && semantic_labels && row0 && choices && vote_label &&
                vote_label_mask && workspace, "spc_vote_labels: null pointer");
  SPC_CHECK_ARG(C >= 3 && B >= 0 && P >= 0, "spc_vote_labels: bad C=%d B=%d P=%d", C, B, P);
  SPC_CHECK_ARG(max_instances >= 1 && max_instances <= 8192, "spc_vote_labels: max_instances=%d outside 1..8192",
                max_instances);
  SPC_CHECK_ARG(workspace_bytes >= spc_vote_labels_workspace_bytes(B, max_instances),
                "spc_vote_labels: workspace too small");
  if (B == 0 || P == 0) return SPC_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int I = max_instances;
  const size_t smem = (size_t)I * 7 * sizeof(int);
  if (smem > 48 * 1024) {
    SPC_CUDA(cudaFuncSetAttribute(vote_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  if (overflow) SPC_CUDA(cudaMemsetAsync(overflow, 0, sizeof(int32_t), st));
  const size_t n_entries = (size_t)B * I;
  vote_init_kernel<<<ceil_div((long long)n_entries * 8, 256), 256, 0, st>>>((int *)workspace, n_entries);
  SPC_LAUNCH_CHECK("vote_init_kernel");
  vote_reduce_kernel<<<dim3(ceil_div(P, VL_THREADS), B), VL_THREADS, smem, st>>>(
      point_clouds, C, P, instance_labels, row0, choices, I, (int *)workspace, overflow);
  SPC_LAUNCH_CHECK("vote_reduce_kernel");
  vote_write_kernel<<<dim3(ceil_div(P, 256), B), 256, 0, st>>>(point_clouds, C, P, instance_labels, semantic_labels,
                                                              row0, choices, I, (unsigned long long)sem_mask,
                                                              (const int *)workspace, vote_label, vote_label_mask);
  SPC_LAUNCH_CHECK("vote_write_kernel");
  return SPC_OK;
}

extern "C" int spc_augment_boxes(const double *boxes, const double *aug, int B, int K, double *out, void *stream) {
  SPC_CHECK_ARG(boxes && aug && out, "spc_augment_boxes: null pointer");
  SPC_CHECK_ARG(B >= 0 && K >= 0, "spc_augment_boxes: bad B=%d K=%d", B, K);
  if (B * K == 0) return SPC_OK;
  augment_boxes_kernel<<<ceil_div((long long)B * K, 128), 128, 0, (cudaStream_t)stream>>>(boxes, aug, B, K, out);
  SPC_LAUNCH_CHECK("augment_boxes_kernel");
  return SPC_OK;
}
