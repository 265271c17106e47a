/*
 * spacap3d_ops.h -- C ABI of libspacap3d_ops.so: B200 (sm_100a) kernels for the PointNet++ /
 * VoteNet point-set operators that SpaCap3D's detector runs on.
 *
 * This is the drop-in boundary.  Each entry point replaces one function of the reference's
 * pybind11 module `pointnet2._ext` (lib/pointnet2/_ext_src/src/bindings.cpp:6-19); the
 * reference-side file:line it stands in for is cited per function.  Differences by design:
 *   - plain pointers + sizes, no torch types; the CALLER allocates every output and workspace;
 *   - the stream is explicit (the reference uses at::cuda::getCurrentCUDAStream());
 *   - a failed launch returns a non-zero status and sets spc_last_error(); it never calls
 *     exit(-1) (reference: include/cuda_utils.h:30-39);
 *   - outputs need NOT be zero-initialised by the caller: every element is written
 *     (the reference relies on torch::zeros, e.g. ball_query.cpp:19-21).
 * All pointers are DEVICE pointers on the current device.  float = IEEE fp32, indices = int32.
 * All tensors are dense, row-major ("contiguous") in the layouts given below.
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * Thread-safety: no mutable global state except a thread-local error string.
 */
#ifndef SPACAP3D_OPS_H
#define SPACAP3D_OPS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPC_OK 0
#define SPC_ERR_INVALID_ARG 1
#define SPC_ERR_CUDA 2
#define SPC_ERR_UNSUPPORTED 3

/* ABI version of this header (bumped on any signature change). */
int spc_abi_version(void);
/* Thread-local, NUL-terminated description of the last non-zero status on this thread. */
const char *spc_last_error(void);

/* furthest_point_sampling(points, nsamples)              sampling.cpp:66-87, sampling_gpu.cu:69-229
 * xyz (B,N,3) -> idx (B,npoint).  Bit-exact with the reference including its tie-breaking
 * (bit-reversed thread id of a 512-thread tree) and its |p|^2 <= 1e-3 skip.
 * new_xyz (B,npoint,3) is optional (may be NULL): the sampled coordinates, i.e. the fused
 * gather_points that always follows FPS in the SA modules (pointnet2_modules.py:237-242).
 * No global workspace: running min-distances live in registers / distributed shared memory. */
int spc_furthest_point_sampling(const float *xyz, int B, int N, int npoint, int32_t *idx,
                                float *new_xyz, void *stream);

/* Same operator with an exact shortcut for FPS-ORDERED inputs (SA2..SA4 of the detector sample
 * from the previous layer's FPS output, where the reference's result is 0..npoint-1 unless exact
 * distance ties interfere -- the reference model relies on that, models/backbone_module.py:107-127).
 * With hint_ordered != 0 and a workspace of spc_fps_workspace_bytes(B,N,npoint) bytes, two fully
 * parallel kernels PROVE per scene whether FPS(xyz)[0:npoint] == 0..npoint-1 (every round's winner
 * is the strict unique maximum, same fp32 arithmetic); proven scenes skip the npoint-1 sequential
 * rounds, all others run the normal kernel.  Results are identical to spc_furthest_point_sampling
 * in every case; the hint only affects speed. */
size_t spc_fps_workspace_bytes(int B, int N, int npoint);
/* Sampler selection, PER CALL (spc_furthest_point_sampling_ex2; the library keeps no mutable state).  Results are
 * identical for every choice.
 *   SPC_FPS_AUTO     the library decides for a call that runs alone: the cluster sampler (small clouds: a single
 *                    CTA), the lowest latency.
 *   SPC_FPS_CLUSTER  one thread-block cluster per scene; coordinates and running min-distances of every point in
 *                    registers / distributed shared memory, per-round arg-max over warp shuffles + DSMEM
 *                    (needs no workspace; holds 4 SMs per 40 k-point scene while it runs).
 *   SPC_FPS_BUCKET   one 512-thread CTA per scene; Hilbert-sorted points parked in L2 (workspace), per-bucket
 *                    bounding boxes and candidates on chip, only the buckets a new centre can change are updated
 *                    (two scenes share an SM; ~2.5x the latency of the cluster sampler, 1/6 of its instructions and
 *                    1/8 of its SM-time: the choice for pipelines with several batches in flight).  Needs a workspace and
 *                    4096 <= N <= 40960, else SPC_ERR_UNSUPPORTED. */
#define SPC_FPS_AUTO 0
#define SPC_FPS_CLUSTER 1
#define SPC_FPS_BUCKET 2
int spc_furthest_point_sampling_ex(const float *xyz, int B, int N, int npoint, int32_t *idx,
                                   float *new_xyz, int hint_ordered, void *workspace,
                                   size_t workspace_bytes, void *stream);
/* Same, with the "strict sequence" side channel that lets a chain of samplers (SA1 -> SA2 -> SA3 -> SA4 each
 * sample from the previous output, models/backbone_module.py:107-127) skip even the proof kernels:
 *   strict_out    (B) int32 device, nullable: 1 = every pick of THIS call was the strict unique maximum of the
 *                 min-distances (implied by a successful proof; the samplers themselves report 0 = unknown), so FPS over
 *                 any prefix of the output is provably the identity; 0 = a tie occurred or it was not tracked.
 *   known_ordered (B) int32 device, nullable: strict_out of the call that produced `xyz` (npoint <= N);
 *                 scenes flagged 1 skip the proof and the sequential rounds, the others behave as with
 *                 hint_ordered alone. */
int spc_furthest_point_sampling_ex2(const float *xyz, int B, int N, int npoint, int32_t *idx,
                                    float *new_xyz, int hint_ordered, const int32_t *known_ordered,
                                    int32_t *strict_out, void *workspace, size_t workspace_bytes,
                                    int algo, void *stream);

/* gather_points(points, idx)                             sampling.cpp:15-38, sampling_gpu.cu:8-30
 * points (B,C,N), idx (B,M) -> out (B,C,M) */
int spc_gather_points(const float *points, const int32_t *idx, int B, int C, int N, int M,
                      float *out, void *stream);

/* gather_points_grad(grad_out, idx, n)                   sampling.cpp:40-65, sampling_gpu.cu:34-57
 * grad_out (B,C,M), idx (B,M) -> grad_points (B,C,N) (zeroed here, then scatter-added) */
int spc_gather_points_grad(const float *grad_out, const int32_t *idx, int B, int C, int N, int M,
                           float *grad_points, void *stream);

/* ball_query(new_xyz, xyz, radius, nsample)              ball_query.cpp:8-32, ball_query_gpu.cu:9-54
 * new_xyz (B,M,3), xyz (B,N,3) -> idx (B,M,nsample): first nsample indices (ascending) with
 * d2 < radius*radius, padded with the first hit; all zeros when the ball is empty. */
int spc_ball_query(const float *new_xyz, const float *xyz, int B, int N, int M, float radius,
                   int nsample, int32_t *idx, void *stream);

/* Same operator, grid-accelerated for large clouds: with a workspace of
 * spc_ball_query_workspace_bytes(B,N) bytes the scene is binned into cells of edge >= radius and
 * each centre only visits its 3x3x3 neighbourhood; the hits are then ordered by point index, so
 * the output is bit-identical to spc_ball_query (same distance arithmetic, same first-nsample /
 * padding contract).  Small problems (and workspace == NULL) use the all-pairs kernel. */
size_t spc_ball_query_workspace_bytes(int B, int N);
int spc_ball_query_ex(const float *new_xyz, const float *xyz, int B, int N, int M, float radius,
                      int nsample, int32_t *idx, void *workspace, size_t workspace_bytes,
                      void *stream);

/* group_points(points, idx)                              group_points.cpp:12-36, group_points_gpu.cu:8-39
 * points (B,C,N), idx (B,npoint,nsample) -> out (B,C,npoint,nsample) */
int spc_group_points(const float *points, const int32_t *idx, int B, int C, int N, int npoint,
                     int nsample, float *out, void *stream);

/* group_points_grad(grad_out, idx, n)                    group_points.cpp:38-62, group_points_gpu.cu:43-75
 * grad_out (B,C,npoint,nsample), idx (B,npoint,nsample) -> grad_points (B,C,N) */
int spc_group_points_grad(const float *grad_out, const int32_t *idx, int B, int C, int N,
                          int npoint, int nsample, float *grad_points, void *stream);
/* Same result (up to fp32 summation order), atomic-free: with a workspace of
 * spc_group_points_grad_workspace_bytes(B,N,npoint,nsample) bytes the index tensor is inverted once into
 * per-point position lists shared by all C channels and every output element is summed by one thread
 * (or one warp) from grad_out rows staged in shared memory.  Bit-reproducible from run to run when
 * npoint*nsample <= 49152; the reference's RED.ADD order is not (SURVEY a6).  Falls back to the
 * entry above when workspace is NULL/too small or C < 4. */
size_t spc_group_points_grad_workspace_bytes(int B, int N, int npoint, int nsample);
int spc_group_points_grad_ex(const float *grad_out, const int32_t *idx, int B, int C, int N,
                             int npoint, int nsample, float *grad_points, void *workspace,
                             size_t workspace_bytes, void *stream);

/* bf16 storage (torch.autocast(dtype=torch.bfloat16) training) of the three entries above: the same operators and
 * argument lists with points / out / grad_out as __nv_bfloat16 device tensors (void pointers).
 *   spc_group_points_bf16        group_points(points, idx)        bf16 in, bf16 out (a copy: no rounding);
 *                                rows of up to ~100 k points are staged (the budget counts bytes)
 *   spc_group_points_grad_bf16   group_points_grad(grad_out, idx, n)   bf16 grad_out in, FP32 grad_points out,
 *   spc_group_points_grad_ex_bf16                                       fp32 accumulation, same kernel choice
 * The gradient stays fp32 (it is nsample times smaller than grad_out): no bf16 atomics, one rounding by the caller. */
int spc_group_points_bf16(const void *points, const int32_t *idx, int B, int C, int N, int npoint,
                          int nsample, void *out, void *stream);
int spc_group_points_grad_bf16(const void *grad_out, const int32_t *idx, int B, int C, int N,
                               int npoint, int nsample, float *grad_points, void *stream);
int spc_group_points_grad_ex_bf16(const void *grad_out, const int32_t *idx, int B, int C, int N,
                                  int npoint, int nsample, float *grad_points, void *workspace,
                                  size_t workspace_bytes, void *stream);

/* three_nn(unknowns, knows)                              interpolate.cpp:14-40, interpolate_gpu.cu:9-68
 * unknown (B,n,3), known (B,m,3) -> dist2 (B,n,3) SQUARED distances ascending, idx (B,n,3).
 * m < 3 leaves +inf / index 0 in the unfilled slots, like the reference. */
int spc_three_nn(const float *unknown, const float *known, int B, int n, int m, float *dist2,
                 int32_t *idx, void *stream);

/* three_interpolate(points, idx, weight)                 interpolate.cpp:42-70, interpolate_gpu.cu:72-111
 * points (B,C,m), idx (B,n,3), weight (B,n,3) -> out (B,C,n) */
int spc_three_interpolate(const float *points, const int32_t *idx, const float *weight, int B,
                          int C, int m, int n, float *out, void *stream);

/* three_interpolate_grad(grad_out, idx, weight, m)       interpolate.cpp:71-99, interpolate_gpu.cu:116-154
 * grad_out (B,C,n), idx (B,n,3), weight (B,n,3) -> grad_points (B,C,m) */
int spc_three_interpolate_grad(const float *grad_out, const int32_t *idx, const float *weight,
                               int B, int C, int n, int m, float *grad_points, void *stream);

/* bf16 storage of the two entries above (same argument lists; idx and weight stay int32 / fp32):
 *   spc_three_interpolate_bf16       three_interpolate(points, idx, weight)        bf16 points -> bf16 out
 *                                    (fp32 arithmetic, one rounding per output)
 *   spc_three_interpolate_grad_bf16  three_interpolate_grad(grad_out, idx, weight, m)  bf16 grad_out -> FP32 grad_points */
int spc_three_interpolate_bf16(const void *points, const int32_t *idx, const float *weight, int B,
                               int C, int m, int n, void *out, void *stream);
int spc_three_interpolate_grad_bf16(const void *grad_out, const int32_t *idx, const float *weight,
                                    int B, int C, int n, int m, float *grad_points, void *stream);


/* Fused set-abstraction forward, eval mode (no reference C++ counterpart: it replaces the whole
 * Python/ATen/cuDNN sequence of PointnetSAModuleVotes.forward after the ball query --
 * pointnet2_utils.py:351-362 (2x group_points, sub, div, cat), pytorch_utils.py:11-36 (SharedMLP =
 * 3 x [1x1 conv, BN, ReLU]) and pointnet2_modules.py:256-271 (max-pool over nsample)).
 *   xyz (B,n,3), new_xyz (B,npoint,3), idx (B,npoint,nsample) from spc_ball_query.
 *   Layer 0, one of two forms (BatchNorm folded into weights/bias by the caller):
 *     in-line  : G_f16 == NULL; feat (B,Cf,n) raw features (Cf <= 13, NULL when Cf == 0),
 *                W0 (C1,3+Cf), b0 (C1);  h1 = relu(W0 . [(p-c)/radius, f] + b0), on the tensor cores with
 *                inputs and weights as fp16 (hi, lo) pairs and three partial products: fp32-grade
 *     projected: G_f16 (B,n,C1) FP16 = W0[:,3:] . f per POINT (one plain GEMM by the caller, conv0 is
 *                linear), Cf == 0, W0 (C1,3) = the xyz columns, b0 (C1);
 *                h1 = relu(G[idx] + W0 . (p-c)/radius + b0), the xyz term evaluated in fp32 here
 *   Layers 1,2: W1 (C2,C1), W2 (C3,C2) row-major FP16 (device pointers to 16-bit data), b1, b2 f32;
 *   run on tcgen05 tensor cores, fp32 accumulation in TMEM.
 *   out (B,C3,npoint) f32 = max over nsample of relu(layer2); out_pm_f16 (optional, may be NULL):
 *   the same values as (B,npoint,C3) FP16, point-major (input of the next layer's projection GEMM).
 * Returns SPC_ERR_UNSUPPORTED (nothing launched) for shapes without a kernel: supported are
 * (C1,C2,C3) in {(64,64,128),(128,128,128),(128,128,256)}, nsample in {16,32,64},
 * npoint*nsample % 128 == 0. */
int spc_sa_fused_forward(const float *xyz, const float *new_xyz, const int32_t *idx,
                         const void *G_f16, const float *feat, const float *W0, const float *b0,
                         int Cf, float radius, const void *W1_f16, const float *b1,
                         const void *W2_f16, const float *b2, int B, int n, int npoint, int nsample,
                         int C1, int C2, int C3, float *out, void *out_pm_f16, void *stream);
/* Same, with a per-call launch hint.  W0_host / b0_host (host copies of the folded layer-0 weights, or NULL) fed a
 * constant-bank FFMA path that no longer exists: they are accepted and ignored.
 * min_tiles_per_cta: PER-CALL launch hint (0 = one CTA per SM, the latency optimum): give every CTA at least this
 * many 128-row tiles, i.e. launch fewer CTAs for the small layers.  Results do not change.  With several batches in
 * flight the freed SMs run other streams' kernels: +4.5 % scenes/s at 16 on B200 (12 streams), -6 % for one stream. */
int spc_sa_fused_forward_ex(const float *xyz, const float *new_xyz, const int32_t *idx, const void *G_f16,
                            const float *feat, const float *W0, const float *b0, const float *W0_host,
                            const float *b0_host, int Cf, float radius, const void *W1_f16, const float *b1,
                            const void *W2_f16, const float *b2, int B, int n, int npoint, int nsample, int C1,
                            int C2, int C3, float *out, void *out_pm_f16, int min_tiles_per_cta, void *stream);

/* ---- point-major (FP16) eval path of the feature-propagation and voting stages ------------------
 * These have no C++ counterpart in the reference; each replaces a chain of small ATen launches. */

/* three_nn + inverse-distance weights (pointnet2_modules.py:398-402): idx (B,n,3) bit-identical to
 * spc_three_nn; weight (B,n,3) = normalised 1/(dist+1e-8).  Needs m >= 3. */
int spc_three_nn_weights(const float *unknown, const float *known, int B, int n, int m, int32_t *idx,
                         float *weight, void *stream);

/* three_interpolate + torch.cat with the skip features (pointnet2_modules.py:404-416), FP16
 * point-major: known_pm (B,m,C2), skip_pm (B,n,C1) -> X (B,n,C2+C1).  C2, C1 multiples of 8. */
int spc_interp_cat_pm(const void *known_pm_f16, const int32_t *idx, const float *weight,
                      const void *skip_pm_f16, int B, int n, int m, int C2, int C1, void *X_f16,
                      void *stream);

/* One 1x1-conv layer of the point-major eval path on tcgen05 tensor cores (csrc/pm_linear.cu): Y = act(X . W^T + b).
 * Replaces the library GEMMs + layout / elementwise kernels of PointnetFPModule's SharedMLP
 * (pointnet2_modules.py:412-421), VotingModule (models/voting_module.py:34-61, plus the L2 normalisation of
 * models/SpaCapNet.py:66-67) and the proposal head (models/proposal_module.py:46-54,73).
 *   X_hi (M,K) FP16 point-major rows, X_lo (M,K) FP16 or NULL (x = hi + lo);  K % 8 == 0
 *   W_hi, W_lo (N,K) FP16: the BatchNorm-folded fp32 weights as a pair (w = hi + lo);  bias (N) f32;  N <= 272
 *   three MMAs per product (hi.hi + lo.hi + hi.lo), fp32 accumulation: fp32-grade results
 *   points_per_scene: rows per scene (M = B * points_per_scene), used by the channel-major outputs
 * mode:
 *   SPC_PM_HIDDEN    y = relu(.)            -> Y_hi, Y_lo (M,N) FP16 pair (the next layer's X);  N % 32 == 0
 *   SPC_PM_OUT_CM    y = relu(.)            -> out (B,N,points) f32 channel-major (the reference's layout) and
 *                                              Y_hi (and Y_lo if not NULL) (M,N) FP16 point-major;  N % 32 == 0
 *   SPC_PM_OUT_PM32  y = .  (no activation) -> out (M,N) f32 point-major (proposal head scores)
 *   SPC_PM_LINEAR    y = .  (no activation) -> Y_hi (and Y_lo if not NULL) (M,N) FP16 (the per-point projection G of
 *                                              the fused set-abstraction kernel, conv0 hoisted out of the grouping)
 *   SPC_PM_VOTE      net = . (N = D + 3; the caller moves conv3's three xyz-offset rows BEHIND its D feature
 *                    rows; D % 32 == 0)     -> v = seed_cm (B,D,points) + net[0:D];  out (B,D,points) = v / ||v||_2,
 *                                              Y_hi (and Y_lo) (M,D) the same point-major;
 *                                              vote_xyz (B,points,3) = seed_xyz + net[D:D+3]
 * n_tile: PER-CALL launch hint, 0 or a multiple of 16: output channels per CTA (0 = 128).  Results do not change.
 *   128 splits a 256-wide layer over two CTAs per row tile (lowest latency alone); 256 keeps it in one, which loads
 *   X once and occupies fewer SMs: +2 % scenes/s with 32 batches in flight on B200.
 * tiles_per_cta: PER-CALL launch hint (0 = 1): consecutive 128-row tiles one CTA works through.  With more than one
 *   the accumulator is double-buffered in TMEM and the epilogue of a tile overlaps the loads of the next; fewer,
 *   longer-lived CTAs (higher latency alone, less SM time in a saturated pipeline).  Results do not change. */
#define SPC_PM_HIDDEN 0
#define SPC_PM_OUT_CM 1
#define SPC_PM_OUT_PM32 2
#define SPC_PM_VOTE 3
#define SPC_PM_LINEAR 4
int spc_pm_linear(const void *X_hi, const void *X_lo, int M, int K, const void *W_hi, const void *W_lo,
                  const float *bias, int N, int mode, int points_per_scene, void *Y_hi, void *Y_lo, float *out,
                  const float *seed_cm, const float *seed_xyz, float *vote_xyz, int n_tile, int tiles_per_cta,
                  void *stream);


/* ---- training-mode BatchNorm + ReLU of a shared-MLP block -------------------------------------------
 * Replaces nn.BatchNorm2d(training) + nn.ReLU(inplace=True) of the reference's Conv2d block
 * (lib/pointnet2/pytorch_utils.py:11-36,39-64,67-120) on y (B,C,S) fp32, S = npoint*nsample:
 *   forward : batch statistics (biased variance), z = relu((y-mean)*invstd*gamma+beta), running statistics
 *             updated in place with `momentum` and the unbiased variance (pass NULL to skip), mean / invstd
 *             saved for backward;
 *   backward: dy, dgamma, dbeta from dz (gradient w.r.t. z), y and the saved statistics; the ReLU mask is
 *             recomputed from y.
 * Any B >= 1 and 1 <= C <= 65535 (no B*C limit).  workspace: spc_bn_relu_workspace_bytes(C) bytes, 8-byte aligned. */
size_t spc_bn_relu_workspace_bytes(int C);
int spc_bn_relu_train_forward(const float *y, const float *gamma, const float *beta, int B, int C, int S,
                              float eps, float momentum, float *running_mean, float *running_var, float *z,
                              float *save_mean, float *save_invstd, void *workspace, size_t workspace_bytes,
                              void *stream);
int spc_bn_relu_train_backward(const float *dz, const float *y, const float *gamma, const float *beta,
                               const float *save_mean, const float *save_invstd, int B, int C, int S,
                               float *dy, float *dgamma, float *dbeta, void *workspace, size_t workspace_bytes,
                               void *stream);

/* Last block of a set-abstraction MLP in training mode: BatchNorm + ReLU + max over the nsample neighbours
 * (pytorch_utils.py:11-36 followed by F.max_pool2d(kernel=[1,nsample]), pointnet2_modules.py:256-259).
 * y (B,C,npoint,nsample) -> pooled (B,C,npoint); the normalised activation is never materialised.
 * argmax (B,C,npoint) uint8 = winning slot (lowest slot on ties, like ATen), ymax = y at that slot; both
 * are consumed by the backward, which produces dy (B,C,npoint,nsample), dgamma, dbeta from dpool.
 * nsample must be 16, 32 or 64 (SPC_ERR_UNSUPPORTED otherwise: nothing launched); any B >= 1 and 1 <= C <= 65535. */
int spc_bn_relu_maxpool_train_forward(const float *y, const float *gamma, const float *beta, int B, int C,
                                      int npoint, int nsample, float eps, float momentum,
                                      float *running_mean, float *running_var, float *pooled,
                                      uint8_t *argmax, float *ymax, float *save_mean, float *save_invstd,
                                      void *workspace, size_t workspace_bytes, void *stream);
int spc_bn_relu_maxpool_train_backward(const float *dpool, const uint8_t *argmax, const float *ymax,
                                       const float *y, const float *gamma, const float *beta,
                                       const float *save_mean, const float *save_invstd, int B, int C,
                                       int npoint, int nsample, float *dy, float *dgamma, float *dbeta,
                                       void *stream);

/* ---- synchronised training-mode BatchNorm (+ ReLU, + max-pool) across the ranks of a process group -------------
 * torch.nn.SyncBatchNorm semantics on the kernels above: the statistics and the backward sums of dm and dm*xhat are
 * taken over the elements of every rank; dgamma / dbeta stay the local sums (the gradient all-reduce adds them).
 * Each pass is split at its one cross-rank reduction.  A rank writes its row `stats` (C, SPC_BN_SYNC_K) fp64:
 *   forward : (n, mean, M2) of its B*S elements per channel       (spc_bn_relu_sync_stats, both variants)
 *   backward: (n, sum dm, sum dm * xhat) per channel              (..._sync_backward_reduce)
 * The caller gathers the rows of all `world` ranks into `stats_all` (world, C, SPC_BN_SYNC_K), rank r at row r (a SUM
 * all-reduce of a zero-initialised buffer does that exactly), and the next call combines them in rank order on the
 * device: every rank gets bit-identical statistics, whatever the collective's reduction order.  The global count
 * comes from the rows, so ranks may hold different B.  No host synchronisation; any B >= 0 (no B*C limit; with
 * B = 0, an empty shard, the rank still takes part: its rows have n = 0 and its tensor pointers may be NULL).
 * The backward apply calls use the workspace (spc_bn_relu_workspace_bytes(C) bytes) as scratch. */
#define SPC_BN_SYNC_K 3
int spc_bn_relu_sync_stats(const float *y, int B, int C, int S, double *stats, void *workspace,
                           size_t workspace_bytes, void *stream);
int spc_bn_relu_sync_forward(const float *y, const float *gamma, const float *beta, int B, int C, int S, int world,
                             const double *stats_all, float eps, float momentum, float *running_mean,
                             float *running_var, float *z, float *save_mean, float *save_invstd, void *stream);
int spc_bn_relu_sync_backward_reduce(const float *dz, const float *y, const float *gamma, const float *beta,
                                     const float *save_mean, const float *save_invstd, int B, int C, int S,
                                     float *dgamma, float *dbeta, double *stats, void *workspace,
                                     size_t workspace_bytes, void *stream);
int spc_bn_relu_sync_backward(const float *dz, const float *y, const float *gamma, const float *beta,
                              const float *save_mean, const float *save_invstd, int B, int C, int S, int world,
                              const double *stats_all, float *dy, void *workspace, size_t workspace_bytes,
                              void *stream);
/* max-pool variant; its statistics phase is the plain one with S = npoint*nsample */
int spc_bn_relu_maxpool_sync_forward(const float *y, const float *gamma, const float *beta, int B, int C, int npoint,
                                     int nsample, int world, const double *stats_all, float eps, float momentum,
                                     float *running_mean, float *running_var, float *pooled, uint8_t *argmax,
                                     float *ymax, float *save_mean, float *save_invstd, void *stream);
int spc_bn_relu_maxpool_sync_backward_reduce(const float *dpool, const float *ymax, const float *gamma,
                                             const float *beta, const float *save_mean, const float *save_invstd,
                                             int B, int C, int npoint, int nsample, float *dgamma, float *dbeta,
                                             double *stats, void *stream);
int spc_bn_relu_maxpool_sync_backward(const float *dpool, const uint8_t *argmax, const float *ymax, const float *y,
                                      const float *gamma, const float *beta, const float *save_mean,
                                      const float *save_invstd, int B, int C, int npoint, int nsample, int world,
                                      const double *stats_all, float *dy, void *workspace, size_t workspace_bytes,
                                      void *stream);

/* ---- bf16 storage of the eleven training-mode BatchNorm + ReLU entries above ---------------------------------------
 * The same passes and argument lists (each `_bf16` entry replaces the same reference code as its fp32 twin) with
 * y, z, dz, dy, dpool, pooled and ymax as __nv_bfloat16 device tensors (void pointers): what
 * nn.BatchNorm2d + nn.ReLU + F.max_pool2d compute on the bf16 output of a 1x1 convolution under
 * torch.autocast(dtype=torch.bfloat16).  gamma, beta, save_mean / save_invstd, dgamma / dbeta and the running
 * statistics stay fp32, the partial sums and the exchanged (world, C, SPC_BN_SYNC_K) rows fp64, and the arithmetic
 * fp32; each bf16 output is rounded once (to nearest even).  The ReLU gradient passes where the bf16 output is > 0,
 * and the max-pool compares the bf16-ROUNDED values of relu(bn(y)): slots that round to the same value tie and the
 * lowest one wins, as F.max_pool2d on the bf16 tensor.  Vector kernels need 8-byte (not 16-byte) alignment. */
int spc_bn_relu_train_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C, int S,
                                   float eps, float momentum, float *running_mean, float *running_var, void *z,
                                   float *save_mean, float *save_invstd, void *workspace, size_t workspace_bytes,
                                   void *stream);
int spc_bn_relu_train_backward_bf16(const void *dz, const void *y, const float *gamma, const float *beta,
                                    const float *save_mean, const float *save_invstd, int B, int C, int S,
                                    void *dy, float *dgamma, float *dbeta, void *workspace, size_t workspace_bytes,
                                    void *stream);
int spc_bn_relu_maxpool_train_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C,
                                           int npoint, int nsample, float eps, float momentum,
                                           float *running_mean, float *running_var, void *pooled,
                                           uint8_t *argmax, void *ymax, float *save_mean, float *save_invstd,
                                           void *workspace, size_t workspace_bytes, void *stream);
int spc_bn_relu_maxpool_train_backward_bf16(const void *dpool, const uint8_t *argmax, const void *ymax,
                                            const void *y, const float *gamma, const float *beta,
                                            const float *save_mean, const float *save_invstd, int B, int C,
                                            int npoint, int nsample, void *dy, float *dgamma, float *dbeta,
                                            void *stream);
int spc_bn_relu_sync_stats_bf16(const void *y, int B, int C, int S, double *stats, void *workspace,
                                size_t workspace_bytes, void *stream);
int spc_bn_relu_sync_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C, int S, int world,
                                  const double *stats_all, float eps, float momentum, float *running_mean,
                                  float *running_var, void *z, float *save_mean, float *save_invstd, void *stream);
int spc_bn_relu_sync_backward_reduce_bf16(const void *dz, const void *y, const float *gamma, const float *beta,
                                          const float *save_mean, const float *save_invstd, int B, int C, int S,
                                          float *dgamma, float *dbeta, double *stats, void *workspace,
                                          size_t workspace_bytes, void *stream);
int spc_bn_relu_sync_backward_bf16(const void *dz, const void *y, const float *gamma, const float *beta,
                                   const float *save_mean, const float *save_invstd, int B, int C, int S, int world,
                                   const double *stats_all, void *dy, void *workspace, size_t workspace_bytes,
                                   void *stream);
int spc_bn_relu_maxpool_sync_forward_bf16(const void *y, const float *gamma, const float *beta, int B, int C,
                                          int npoint, int nsample, int world, const double *stats_all, float eps,
                                          float momentum, float *running_mean, float *running_var, void *pooled,
                                          uint8_t *argmax, void *ymax, float *save_mean, float *save_invstd,
                                          void *stream);
int spc_bn_relu_maxpool_sync_backward_reduce_bf16(const void *dpool, const void *ymax, const float *gamma,
                                                  const float *beta, const float *save_mean, const float *save_invstd,
                                                  int B, int C, int npoint, int nsample, float *dgamma, float *dbeta,
                                                  double *stats, void *stream);
int spc_bn_relu_maxpool_sync_backward_bf16(const void *dpool, const uint8_t *argmax, const void *ymax, const void *y,
                                           const float *gamma, const float *beta, const float *save_mean,
                                           const float *save_invstd, int B, int C, int npoint, int nsample, int world,
                                           const double *stats_all, void *dy, void *workspace, size_t workspace_bytes,
                                           void *stream);

/* ---- detection post-processing (SURVEY row N3): device side of parse_predictions, lib/ap_helper.py:44-160 ----
 * spc_box_point_counts: counts[b,k] = number of points of scene b inside predicted box k (the reference's
 *   extract_pc_in_box3d / scipy Delaunay hull test per box, ap_helper.py:69-79, data/scannet/model_util_scannet.py:
 *   13-22).  points (B,N,point_stride) f32 (xyz first), corners (B,K,8,3) f64 in get_3d_box_batch order
 *   (utils/box_util.py:360-383; rotated boxes are handled).
 * spc_nms_boxes: pick[b,k] = 1 for the boxes kept by nms_2d_faster (mode 0), nms_3d_faster (mode 1) or
 *   nms_3d_faster_samecls (mode 2) of utils/nms.py:39-147 applied to the boxes with valid[b,k] != 0 (NULL = all),
 *   scores (B,K) f32, classes (B,K) int64 (mode 2), fp64 arithmetic in numpy's expression order; equal scores are
 *   ordered as by a stable sort.  K <= 512. */
int spc_box_point_counts(const float *points, int point_stride, const double *corners, int B, int N, int K,
                         int32_t *counts, void *stream);
int spc_nms_boxes(const double *corners, const float *score, const int64_t *cls, const int32_t *valid, int B,
                  int K, int mode, int old_type, double iou_threshold, int32_t *pick, void *stream);

/* ---- input pipeline (SURVEY row N4): device side of ScannetReferenceDataset.__getitem__, lib/dataset.py:291-531 ----
 * The pre-processed scenes live in HBM as ONE packed vertex table verts (total_rows, vstride) f32 -- columns
 * x y z r g b nx ny nz as written by data/scannet/batch_load_scannet_data.py:75-80 -- plus, optionally, a packed
 * multiview table (total_rows, n_mv) f32 (the ENet features the reference reads per item from an h5py file,
 * lib/dataset.py:321-328) and packed int32 instance / semantic label columns.  Batch item b refers to the scene whose
 * first row is row0[b]; choices (B,P) int32 are row numbers RELATIVE to that scene (np.random.choice of
 * utils/pc_utils.py:32-40, drawn on the host so that the reference's RNG stream is preserved).
 *
 * spc_scene_floor_height: out[0] = np.percentile(verts[:M, col], 100*quantile) with numpy >= 2.0 float32 semantics
 *   (`quantile` is the float32 value np.float32(0.99)/np.float32(100) for lib/dataset.py:331); one CTA, radix select.
 *   Call once per scene when it is loaded and cache the value.  Finite inputs only.
 * spc_prepare_point_clouds: out (B,P,C_out) f32, C_out = 3 [+3 colour] [+3 normal] [+n_mv] [+1 height], in the
 *   reference's channel order (lib/dataset.py:309-333).  colour = (rgb - mean)/256 in fp64 -> fp32 (:314);
 *   height = z - floor_height[b] (fp32, BEFORE augmentation, :330-333; floor_height NULL = no height channel);
 *   aug (B,32) f64 per item = [flip_x, flip_y, rotx(9), roty(9), rotz(9), translation(3)] (:366-404; NULL = no
 *   augmentation): xyz is negated / multiplied by each 3x3 matrix in fp64 and ROUNDED TO fp32 after every step, as
 *   numpy does when assigning into the float32 cloud; normals are not rotated (neither does the reference).
 * spc_vote_labels: vote_label (B,P,9) f32 and vote_label_mask (B,P) int64 of lib/dataset.py:421-431 from the prepared
 *   clouds (B,P,C): per instance id the bounding box of its sampled points, centre = 0.5*(min+max), vote = centre - x,
 *   tiled 3x; an instance votes iff the semantic label of its first sampled point is in sem_mask (bit i = label i,
 *   DC.nyu40ids).  Instance ids must be in [0, max_instances); others get no vote and set *overflow = 1 (nullable).
 *   workspace: spc_vote_labels_workspace_bytes(B, max_instances) bytes.
 * spc_augment_boxes: the same flips / rotations / translation applied to axis-aligned boxes (B,K,6) f64 =
 *   centre + lengths (lib/dataset.py:369-404, rotate_aligned_boxes_along_axis,
 *   data/scannet/model_util_scannet.py:47-82), fp64 throughout. */
int spc_scene_floor_height(const float *verts, int M, int stride, int col, float quantile, float *out,
                           void *stream);
int spc_prepare_point_clouds(const float *verts, int vstride, const float *multiview, int n_mv,
                             const int64_t *row0, const int32_t *choices, const float *floor_height,
                             const double *aug, double mean_r, double mean_g, double mean_b, int B, int P,
                             int use_color, int use_normal, float *out, void *stream);
size_t spc_vote_labels_workspace_bytes(int B, int max_instances);
int spc_vote_labels(const float *point_clouds, int C, const int32_t *instance_labels,
                    const int32_t *semantic_labels, const int64_t *row0, const int32_t *choices, int B, int P,
                    int max_instances, uint64_t sem_mask, float *vote_label, int64_t *vote_label_mask,
                    int32_t *overflow, void *workspace, size_t workspace_bytes, void *stream);
int spc_augment_boxes(const double *boxes, const double *aug, int B, int K, double *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SPACAP3D_OPS_H */
