/*
 * pointdae_b200.h -- C ABI of libpointdae_b200.so: Point-DAE's point-cloud geometry hot path
 * (FPS + gather, kNN + Group, DGCNN kNN / graph feature, Chamfer fwd/bwd) as sm_100a CUDA.
 *
 * Conventions (all entry points):
 *   - plain device pointers, sizes as int; no torch / C++ types.  fp32 data, int32 indices for
 *     FPS / gather / Chamfer / ball-query, int64 for kNN (they feed `idx + idx_base`).
 *   - the caller owns every buffer (inputs, outputs, workspace); nothing is allocated inside.
 *   - work is enqueued on `stream` (a cudaStream_t / CUstream) of the CURRENT device and the
 *     call returns without synchronising: safe under CUDA-graph capture, re-entrant, and
 *     callable from several host threads (one per device) at once.
 *   - return value: 0 on success, a positive cudaError_t when the CUDA runtime refused a
 *     launch, a negative PDAE_E_* for an invalid argument.  Never exit(), never print and
 *     continue (the reference does both: cuda_utils.h:32-41, chamfer.cu:166-169).
 *
 * "replaces" cites the reference (YBZh/Point-DAE) interface each symbol stands in for.
 */
#ifndef POINTDAE_B200_H
#define POINTDAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDAE_ABI_VERSION 1

#define PDAE_E_INVALID (-1)     /* bad size / null pointer */
#define PDAE_E_UNSUPPORTED (-2) /* shape outside what the kernels implement (message via pdae_strerror) */
#define PDAE_E_WORKSPACE (-3)   /* workspace too small */

typedef void *pdae_stream_t; /* cudaStream_t */

int pdae_abi_version(void);
/* human-readable text for a code returned by any entry point (cudaGetErrorString for >0). */
const char *pdae_strerror(int code);

/* ---- FPS ------------------------------------------------------------------------------------
 * replaces: pointnet2_ops / extensions/pointnet2 `furthest_point_sampling(points, nsamples)`
 *           _ext_src/src/sampling.cpp:67-88 -> sampling_gpu.cu:72-176 (bindings.cpp:12).
 * xyz (b,n,3) dense; idx (b,m) int32.  Bit-exact with the reference including the
 * |p|^2 <= 1e-3 skip and the bit-reversed-slot tie rule (block size from pdae_fps_block_size).
 * Needs no workspace for n <= 12288 (state lives in registers / shared memory); larger n uses
 * `workspace` (pdae_fps_workspace_bytes, may be 0) for the running min-distances.            */
int pdae_fps_block_size(int n); /* replaces opt_n_threads, cuda_utils.h:15-21 */
size_t pdae_fps_workspace_bytes(int b, int n, int m);
int pdae_fps_f32(const float *xyz, int b, int n, int m, int *idx, void *workspace, size_t workspace_bytes,
                 pdae_stream_t stream);

/* fused utils/misc.py:13-20 `fps(data, number)`: data (b,n,c) with c >= 3 (xyz first),
 * idx (b,m) int32, centers (b,m,c) = data[idx] -- one launch instead of FPS + 2 transposes +
 * gather + transpose.                                                                         */
int pdae_fps_gather_f32(const float *data, int b, int n, int c, int m, int *idx, float *centers, void *workspace,
                        size_t workspace_bytes, pdae_stream_t stream);

/* ---- gather ---------------------------------------------------------------------------------
 * replaces: `gather_points` sampling.cpp:17-40 / sampling_gpu.cu:11-33 and `gather_points_grad`
 *           sampling.cpp:42-66 / sampling_gpu.cu:37-60 (bindings.cpp:10-11).
 * feat (b,c,n), idx (b,m) int32 -> out (b,c,m).  grad: gout (b,c,m) -> gfeat (b,c,n),
 * overwritten (zero-filled inside, then scatter-added).                                       */
int pdae_gather_f32(const float *feat, const int *idx, int b, int c, int n, int m, float *out, pdae_stream_t stream);
int pdae_gather_grad_f32(const float *gout, const int *idx, int b, int c, int n, int m, float *gfeat,
                         pdae_stream_t stream);

/* ---- kNN ------------------------------------------------------------------------------------
 * replaces: knn_cuda.KNN(k, transpose_mode).forward(ref, query) (KNN_CUDA 0.2, un-vendored;
 *           call sites models/PointCAE_transformer.py:59,76, models/MaskSurf_v2.py:79,124).
 * ref (b,r,dim), query (b,q,dim) row-major (the facade transposes for transpose_mode=False).
 * Outputs ascending by (distance, index): dist = sqrt(squared distance) or NULL,
 * idx int64.  out_kq = 0: (b,q,k) layout; 1: (b,k,q) layout (transpose_mode=False).
 * Requires 1 <= k <= min(r, 128).                                                             */
int pdae_knn_f32(const float *ref, const float *query, int b, int r, int q, int dim, int k, int out_kq, float *dist,
                 int64_t *idx, pdae_stream_t stream);

/* Same searches with a caller-owned workspace (pdae_knn_workspace_bytes; may return 0): shapes with few queries and a
 * long reference cloud (scene scale, e.g. 2048 queries x 100 000 points) are cut along the reference cloud into chunks
 * that fill the GPU; each chunk's k best keys land in the workspace and a merge launch finishes.  Same results bit for
 * bit; a NULL / too small workspace runs the unchunked form.                                                       */
size_t pdae_knn_workspace_bytes(int b, int r, int q, int dim, int k);
int pdae_knn_ws_f32(const float *ref, const float *query, int b, int r, int q, int dim, int k, int out_kq, float *dist,
                    int64_t *idx, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
int pdae_group_ws_f32(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx,
                      float *neighborhood, void *workspace, size_t workspace_bytes, pdae_stream_t stream);

/* fused Group.forward tail, models/PointCAE_transformer.py:76-85: kNN of `center` (b,g,3) in
 * xyz (b,n,3) + gather + centre-subtract.  idx (b,g,m) int64 (may be NULL),
 * neighborhood (b,g,m,3).                                                                     */
int pdae_group_f32(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx,
                   float *neighborhood, pdae_stream_t stream);

/* same search, neighbours NOT re-centred: patches (b,g,m,3) = xyz[idx].  The patch gather of
 * datasets/corrupt_util_tensor.py:592-616 `dropout_patch_random` (FPS 64 + KNN 32 + advanced indexing).            */
int pdae_group_gather_f32(const float *xyz, const float *center, int b, int n, int g, int m, int64_t *idx,
                          float *patches, pdae_stream_t stream);

/* the whole patchifier of `Group.forward` (models/PointCAE_transformer.py:61-86) in one call: utils/misc.py:13-20 `fps`
 * (FPS + centre gather) followed by the Group tail above.  xyz (b,n,3); fps_idx (b,g) int32; center (b,g,3);
 * idx (b,g,m) int64 (may be NULL); neighborhood (b,g,m,3).  Batches of >= 48 clouds of 512..2048 points with m <= 32 and g <= 1024 run as
 * ONE launch (a CTA per cloud: four FPS warps post each centre to shared memory, consumer warps search it while the
 * sampling goes on); other shapes run pdae_fps_gather_f32 + pdae_group_ws_f32 (workspace: pdae_fps_group_workspace_bytes,
 * may be 0).  Same results bit for bit either way.  pdae_tune_patchify(enabled, centres per consumer task, consumer warps)
 * is the A/B hook (enabled = 0: always the two-launch form, 1: automatic, 2: one launch for every eligible shape).                                                        */
size_t pdae_fps_group_workspace_bytes(int b, int n, int g, int m);
int pdae_fps_group_f32(const float *xyz, int b, int n, int g, int m, int *fps_idx, float *center, int64_t *idx,
                       float *neighborhood, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
/* same call with launch flags.  PDAE_LAUNCH_OVERLAP_PREVIOUS: the caller vouches that the kernel queued before this call on
 * `stream` does not produce xyz (e.g. the Chamfer forward of the same training step); the single-launch form is then
 * queued with programmatic stream serialization, so its CTAs start as the previous kernel's CTAs exit (that kernel must
 * have triggered its dependents -- the tensor-core Chamfer forward does -- or the launch simply waits for it to end).
 * Ignored by the two-launch form.                                                                                   */
#define PDAE_LAUNCH_OVERLAP_PREVIOUS 1u
int pdae_fps_group_ex_f32(const float *xyz, int b, int n, int g, int m, int *fps_idx, float *center, int64_t *idx,
                          float *neighborhood, void *workspace, size_t workspace_bytes, unsigned flags, pdae_stream_t stream);
int pdae_tune_patchify(int enabled, int qw, int ncw);
/* diagnostics: while `device_buffer` (>= 1 + g + 8 * g int64, caller-zeroed) is set, CTA 0 of every single-launch
 * patchifier call stamps clock64 there: [0] start, [1 + j] centre j posted, [1 + g + 8 t + p] phases of search task t.
 * NULL switches the stamps off (the default).                                                                       */
int pdae_patchify_trace(long long *device_buffer);

/* ---- the hot path as one call ---------------------------------------------------------------------------------------
 * One training step of the path (the model's order: models/PointCAE_transformer.py:1010-1066) enqueued natively with its
 * launch choreography: on `stream` the Chamfer forward of `pred` against `cloud` (both (b,n,3)), then the patchifier of
 * `cloud` (g centres, m neighbours; g = 0 skips it) as a programmatic dependent launch -- it reads only the cloud, so its
 * CTAs start where a forward CTA exits; on two library-owned helper streams, after the forward only: the fused mean loss
 * (loss3, see pdae_chamfer_loss_f32) and the gradients of that loss scaled by the device scalar *gloss (gpred, gcloud,
 * see pdae_chamfer_loss_bwd_f32).  `stream` waits for both before the call returns; the call is capturable.
 * Outputs as in pdae_fps_group_f32 / pdae_chamfer_fwd_f32 (dist1 / idx1 belong to pred's points); same bits.
 * Six launches, a few microseconds of host time; workspace: pdae_step_workspace_bytes.                              */
size_t pdae_step_workspace_bytes(int b, int n, int g, int m);
int pdae_step_f32(const float *cloud, const float *pred, int b, int n, int g, int m, int *fps_idx, float *center,
                  float *neighborhood, float *dist1, float *dist2, int *idx1, int *idx2, float *loss3, const float *gloss,
                  float *gpred, float *gcloud, void *workspace, size_t workspace_bytes, pdae_stream_t stream);

/* ---- DGCNN kNN + graph feature --------------------------------------------------------------
 * replaces: models/dgcnn_util.py:7-12 `knn(x, k)` and :15-36 `get_graph_feature`.
 * x (b,c,n) channel-major.  idx (b,n,k) int64 nearest-first, self included, direct-form
 * distance accumulated in channel order, ties -> lower index.
 * graph_feature: out physical (b,n,k,2c): [0:c] = x[:,idx]-x_i, [c:2c] = x_i (the reference's
 * permuted view).  grad: gout same layout -> gx (b,c,n) overwritten.                          */
int pdae_feat_knn_f32(const float *x, int b, int c, int n, int k, int64_t *idx, pdae_stream_t stream);
/* Same search with a caller-owned workspace (pdae_feat_knn_workspace_bytes, up to 1 GiB): for c >= 8 and k <= 32 the
 * distances go through a materialised (n x n) matrix per cloud and a threshold pre-pass, which is faster than the
 * streaming selection of pdae_feat_knn_f32 (same result bit for bit); other shapes ignore the workspace.          */
size_t pdae_feat_knn_workspace_bytes(int b, int c, int n, int k);
int pdae_feat_knn_ws_f32(const float *x, int b, int c, int n, int k, int64_t *idx, void *workspace,
                         size_t workspace_bytes, pdae_stream_t stream);
/* workspace for graph_feature / _grad: one (b,n,c) fp32 transposed copy. */
size_t pdae_graph_feature_workspace_bytes(int b, int c, int n);
int pdae_graph_feature_f32(const float *x, const int64_t *idx, int b, int c, int n, int k, float *out,
                           void *workspace, size_t workspace_bytes, pdae_stream_t stream);
int pdae_graph_feature_grad_f32(const float *gout, const int64_t *idx, int b, int c, int n, int k, float *gx,
                                void *workspace, size_t workspace_bytes, pdae_stream_t stream);

/* ---- Chamfer --------------------------------------------------------------------------------
 * replaces: `chamfer.forward(xyz1, xyz2)` chamfer_cuda.cpp:22-25 -> chamfer.cu:147-171 and
 *           `chamfer.backward(...)` chamfer_cuda.cpp:27-34 -> chamfer.cu:203-229.
 * xyz1 (b,n,3), xyz2 (b,m,3) read as dense storage exactly like the reference's raw data_ptr
 * access.  dist1 (b,n), dist2 (b,m) squared distances; idx1, idx2 int32, lowest index on ties.
 * backward: gx1 (b,n,3), gx2 (b,m,3) overwritten.                                             */
/* Optional workspace (pdae_chamfer_fwd_workspace_bytes, 8 bytes per point of both clouds): when given,
 * every point pair is evaluated ONCE and feeds both directions (the squared distance is symmetric bit for
 * bit), halving the arithmetic; with workspace == NULL each direction is scanned separately.  With at least
 * 8 bytes per point of the smaller cloud the symmetric kernel runs; with the full size it may also cut every
 * row block's sweep into column chunks merged through packed keys, which evens out the load of the SMs when
 * the batch gives fewer than ~8 CTAs per SM.  Results are identical in all cases.                          */
size_t pdae_chamfer_fwd_workspace_bytes(int b, int n, int m);
int pdae_chamfer_fwd_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2,
                         int *idx1, int *idx2, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
/* The same forward in two calls, so that the caller can put a stream event between them: phase 1 = the scan (the
 * FMA-bound part: every output of the larger cloud final, the other cloud's minima parked in the workspace), phase 2 =
 * the recovery of the other cloud's dist / idx from the workspace.  Work that should overlap the latency-bound tail of
 * the step rather than the scan (the patchifier's kNN in bench.py) waits on that event.  Same arguments in both
 * calls; phase 1 then phase 2 is identical to pdae_chamfer_fwd_f32.                                                  */
int pdae_chamfer_fwd_phase_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2,
                               int *idx1, int *idx2, void *workspace, size_t workspace_bytes, int phase,
                               pdae_stream_t stream);
int pdae_chamfer_bwd_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2, const float *gd1,
                         const float *gd2, int b, int n, int m, float *gx1, float *gx2, pdae_stream_t stream);

/* Fused mean losses on top of the forward's outputs (SURVEY.md 8f row 2).
 * replaces: the torch arithmetic of ChamferDistanceL2.forward `mean(dist1) + mean(dist2)`
 *           (extensions/chamfer_dist/__init__.py:43), ChamferDistanceL2_split (:394-395) and ChamferDistanceL1
 *           `(mean(sqrt(dist1)) + mean(sqrt(dist2))) / 2` (:413-417), and their autograd backward into
 *           chamfer.backward.
 * pdae_chamfer_loss_f32: loss3[0] = the loss (l1 = 0: L2, 1: L1), loss3[1], loss3[2] = the two mean terms;
 *   deterministic two-launch reduction; workspace of pdae_chamfer_loss_workspace_bytes().
 * pdae_chamfer_loss_bwd_f32: gradients of  w1 * mean(f(dist1)) + w2 * mean(f(dist2))  scaled by the device scalar
 *   *gloss (f = identity or sqrt): gx1 (b,n,3), gx2 (b,m,3) overwritten.  dist1/dist2 are read only when l1 != 0. */
size_t pdae_chamfer_loss_workspace_bytes(void);
int pdae_chamfer_loss_f32(const float *dist1, const float *dist2, int b, int n, int m, int l1, float *loss3,
                          void *workspace, size_t workspace_bytes, pdae_stream_t stream);
int pdae_chamfer_loss_bwd_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2, const float *dist1,
                              const float *dist2, const float *gloss, float w1, float w2, int b, int n, int m, int l1,
                              float *gx1, float *gx2, pdae_stream_t stream);

/* ---- "next" rows: the dense consumers on the tensor cores (SURVEY.md 8f row 4) --------------------------------------
 * replaces: the 1x1 convolutions of `dgcnn_encoder` (nn.Conv2d(2C, Co, 1, bias=False) over the graph feature,
 *           models/dgcnn_util.py:96-128 -- through the identity W [x_j - x_i ; x_i] = W1 x_j + (W2 - W1) x_i it is
 *           one Conv1d-shaped product per layer) and of the patch `Encoder` (nn.Conv1d, models/PointCAE_transformer.py:
 *           24-35).
 * z[b][j][n] = sum_c w[j][c] * x[b][c][n]:  x (b,c,n), w (j,c), z (b,j,n), fp32 in and out.  tcgen05.mma kind::tf32 with
 * the 3xTF32 operand split (fp32 accuracy, ~1e-6 relative), accumulator in tensor memory.  The workspace holds the
 * weights' hi / lo shared-memory images (pdae_conv1x1_workspace_bytes).                                            */
size_t pdae_conv1x1_workspace_bytes(int c, int j);
int pdae_conv1x1_tf32x3_f32(const float *x, const float *w, const float *bias, int b, int c, int n, int j,
                            int in_point_major, int out_point_major, float *z, void *workspace, size_t workspace_bytes,
                            pdae_stream_t stream);
/* bias (j) or NULL is added in the epilogue (nn.Conv1d's bias).  in_point_major / out_point_major: x is (b,n,c) / z is
 * (b,n,j) instead of the channel-major layouts above.
 *
 * One EdgeConv layer on the point-major product z = [P | Q] (b,n,ld >= 2*co) of the call above with the stacked weight
 * [W1 ; W2 - W1] (W = [W1 | W2] the layer's (co,2c) convolution weight): y[i][j] = P[idx(i,j)] + Q[i] is the layer's
 * convolution output for edge (i,j) without the (b,2c,n,k) graph feature or the (b,co,n,k) tensor ever existing.
 *   pdae_edge_stats_f64     per-CTA partial sums (pdae_edge_partial_count(b,n), co, 2) of sum y and sum y^2 -> BatchNorm
 *                           batch statistics (training mode); summed by the caller in a fixed order.
 *   pdae_edge_forward_f32   out (b,co,n) = LeakyReLU(scale (ext_j P[idx] + Q) + shift), ext = max where scale >= 0, min
 *                           where scale < 0 (BatchNorm + LeakyReLU is monotone per channel); jstar (b,n,co) uint8 = the
 *                           neighbour slot selected (NULL: not wanted).
 *   pdae_edge_backward_f32  partial != NULL: per-CTA partial sums of dbeta / dgamma from g (b,n,co), the upstream
 *                           gradient point-major.  dz != NULL: dz (b,n,ld) = [dP | dQ], zero-filled by the caller
 *                           (dP is scatter-added); train = 1 adds the two per-channel terms training-mode BatchNorm
 *                           spreads over every edge (ca, cb = gamma dbeta / M, gamma dgamma / M, M = b n k).
 *                           LeakyReLU's derivative is 1 where the BatchNorm output is > 0 and the slope elsewhere, at 0
 *                           too (torch's convention); the same in the two-phase backward below.                    */
size_t pdae_edge_partial_count(int b, int n);
int pdae_edge_stats_f64(const float *z, int ld, const int64_t *idx, int b, int n, int k, int co, double *partial, float *s1,
                        pdae_stream_t stream);  /* s1 (b,n,co) or NULL: sum_j P[idx(i,j)], kept for the backward */
/* The same sums of v = y - c_o instead of y, c_o = P[0][o] + Q[0][o] of cloud 0 rounded to fp32 (one sample of the
 * channel); s1 unchanged.  sum y^2 / M - mean^2 loses the digits a channel's mean has above its spread; the shifted sums
 * keep the statistics at the accuracy of P and Q themselves (what ops.edge_conv uses; finish with
 * pdae_edge_bn_prepare_shifted_f32 on the same z).                                                                    */
int pdae_edge_stats_shifted_f64(const float *z, int ld, const int64_t *idx, int b, int n, int k, int co, double *partial,
                                float *s1, pdae_stream_t stream);
int pdae_edge_forward_f32(const float *z, int ld, const int64_t *idx, const float *scale, const float *shift, float slope,
                          int b, int n, int k, int co, float *out, unsigned char *jstar, pdae_stream_t stream);
int pdae_edge_backward_f32(const float *z, int ld, const int64_t *idx, const unsigned char *jstar, const float *g,
                           const float *scale, const float *shift, const float *mean, const float *invstd,
                           const float *gamma, const float *ca, const float *cb, float slope, int train, int b, int n, int k,
                           int co, double *partial, float *dz, pdae_stream_t stream);

/* ---- "next" rows: index consumers of the match (SURVEY.md 8f row 2) ---------------------------------------------------
 * replaces: the torch.gather / normalize / difference / mean chains of the normal, curvature and position terms of
 *           ChamferDistanceL2_withnormal* (extensions/chamfer_dist/__init__.py:95-120, 143-165, 206-376).
 * One term  mean_j metric(a_j, b[idx1[j]]) + mean_j metric(b_j, a[idx2[j]]),  a (bs,n,d), b (bs,m,d), d <= 8, idx from
 * pdae_chamfer_fwd_f32; metric 0 dis_l2, 1 dis_normalized_l2 (orientation-free), 2 dis_normalized_l1, 3
 * dis_normalized_l2_strict.  fwd: per-CTA fp64 partial sums (pdae_pair_loss_partial_count(bs,n,m), 2), summed by the
 * caller in a fixed order.  bwd: ga / gb overwritten with gloss * (w1 d(side 1) + w2 d(side 2)), w = 1/(bs n), 1/(bs m). */
size_t pdae_pair_loss_partial_count(int bs, int n, int m);
int pdae_pair_loss_fwd_f64(const float *a, const float *b, const int *idx1, const int *idx2, int bs, int n, int m, int d,
                           int metric, double *partial, pdae_stream_t stream);
int pdae_pair_loss_bwd_f32(const float *a, const float *b, const int *idx1, const int *idx2, const float *gloss, float w1,
                           float w2, int bs, int n, int m, int d, int metric, float *ga, float *gb, pdae_stream_t stream);

/* tuning hook, no reference counterpart: number of column chunks every 512-row block of the symmetric forward is cut
 * into (ids as the PDAE_CHAMFER_SPLIT environment variable: 0 = automatic, 1 = never split; nc < 0 only queries).
 * Returns the previous setting.  Results do not depend on it.  Not thread-safe.                                 */
int pdae_tune_chamfer_split(int nc);
/* Chamfer forward, both clouds >= 512 points (above 2048 points: with the workspace, column chunks merged through keys): the tensor cores (tcgen05.mma kind::tf32, hi/lo split operands) evaluate
 * approximate distances, the 32-column groups that can hold a row's minimum within the error bound are re-evaluated with the
 * reference's exact expression (chamfer.cu:42-79) -- same bits as the FP32-pipe kernels (csrc/chamfer_tc.cu).
 * Tuning / test hook: mode 0 = FP32-pipe kernels only, 1 / 2 = tf32 operands (two K = 8 MMAs per tile) with 128- / 256-column
 * accumulators, 3 = fp16 operands of power-of-two scaled coordinates (one K = 16 MMA per tile; the default; environment
 * PDAE_CHAMFER_TC); eps_rel > 0 sets the filter's error bound relative to max|a - c|^2 + max|b - c|^2, eps_rel < 0 restores
 * the mode's default (2^-17 tf32, 2^-16 fp16; PDAE_CHAMFER_TC_EPS).  mode < 0 only queries.  Returns the previous mode.    */
int pdae_tune_chamfer_tc(int mode, float eps_rel);
/* host-only diagnostic: the cost-balanced shares of the tensor-core forward's persistent CTAs (a CTA pays for its
 * 128-row blocks and for every operand image it builds) for b clouds of n against m points on `grid` CTAs.
 * bounds_out[0..grid]: first unit of every CTA; returns grid + 1, or 0 when equal block counts are used.            */
int pdae_chamfer_tc_shares(int b, int n, int m, int grid, long long *bounds_out, long long *units_out);
/* probe: the tensor-core forward regardless of the mode, plus filter statistics in stats4 (4 x uint64, zeroed by the caller):
 * [0] float bits of the largest |approximate - exact| group minimum relative to the bound's scale, [1] rows decided by the
 * literal scan (list overflow / no finite candidate), [2] 32-column groups evaluated exactly, [3] rows written.
 * trace: optional 256 x 6 int64 of clock64 stamps of CTA 0's first tiles (pipeline timeline), or NULL.                     */
int pdae_chamfer_tc_probe(const float *xyz1, const float *xyz2, int b, int n, int m, float *dist1, float *dist2, int *idx1,
                          int *idx2, unsigned long long *stats4, long long *trace, pdae_stream_t stream);
/* tuning / test hook of kNN / Group (dim 3, k <= 64): form = (queries per warp, warps per CTA) of the kernel: 0 = (4, 8)
 * warp-specialised (7 compute warps + a producer warp), 1 = (4, 8), 2 = (4, 4), 3 = (2, 4); tile points per
 * shared-memory tile, nz chunks along the reference cloud (needs the workspace), tma 0/1.  -1 = automatic.  Same results
 * for every setting (tests/test_gpu_knn4.py).  Returns 0, or PDAE_E_INVALID for a form outside -1..3 (the setting is
 * then unchanged).  Not thread-safe.                                                                                 */
int pdae_tune_knn(int form, int tile, int nz, int tma);

/* reference-set sharding (scene-scale clouds, SURVEY.md 8e; new, no reference counterpart):
 * one direction, queries (b,nq,3) against the local slice refs (b,nr,3) whose first point has
 * global index `ref_offset`; emits keys[b,nq] = (float_bits(min d) << 32) | global argmin, an
 * order-preserving packing so a uint64/int64 MIN all-reduce across ranks yields the global
 * (min, lowest argmin).  pdae_chamfer_unpack_keys splits reduced keys into dist / idx.        */
int pdae_chamfer_min_keys_u64(const float *queries, const float *refs, int b, int nq, int nr, int ref_offset,
                              uint64_t *keys, pdae_stream_t stream);
int pdae_chamfer_unpack_keys(const uint64_t *keys, long long count, float *dist, int *idx, pdae_stream_t stream);
/* one rank's whole share in a single pass (each pair evaluated once): xyz1 (b,n,3) replicated, xyz2_local
 * (b,m_local,3) = points [ref_offset, ref_offset+m_local) of xyz2.  keys1 (b,n): packed row minima for the MIN
 * all-reduce; dist2_local / idx2_local (b,m_local): final for the slice.  workspace: 8*b*m_local bytes.          */
int pdae_chamfer_sharded_f32(const float *xyz1, const float *xyz2_local, int b, int n, int m_local, int ref_offset,
                             uint64_t *keys1, float *dist2_local, int *idx2_local, void *workspace,
                             size_t workspace_bytes, pdae_stream_t stream);

/* kNN with the reference set sharded across ranks (scene-scale clouds, SURVEY.md 8e; new, no reference counterpart).
 * pdae_knn_keys_u64: this rank's k best candidates per query from its slice ref_local (b,r_local,dim), whose first
 *   point has global index ref_offset: keys (b,q,k) ascending, (squared-distance bits << 32 | global index);
 *   slots beyond r_local hold 0xffff...f.  The ranks all-gather their lists into (w,b,q,k).
 * pdae_knn_merge_keys_u64: W-way merge of the gathered lists -> the same dist / idx pdae_knn_f32 returns on the whole
 *   reference cloud (Euclidean distances, int64 indices, (b,q,k) or (b,k,q) layout).  w <= 16.                     */
int pdae_knn_keys_u64(const float *ref_local, const float *query, int b, int r_local, int q, int dim, int k,
                      long long ref_offset, uint64_t *keys, pdae_stream_t stream);
int pdae_knn_merge_keys_u64(const uint64_t *keys_all, int w, int b, int q, int k, int out_kq, float *dist, int64_t *idx,
                            pdae_stream_t stream);

/* The same backward in two phases without one float atomic per edge and channel (the default of ops.edge_backward):
 *   pdae_edge_backward_select_f32  per-CTA partial sums of dbeta / dgamma AND the selected edges' term gamma*dbn stored into
 *                                  the Q half / scatter-added into the P half of dz (b,n,ld), zero-filled by the caller
 *                                  (b*n*co atomics); with train = 0 (eval-mode BatchNorm) dz is then complete.
 *   pdae_edge_backward_dense_f32   training mode: the two per-channel terms BatchNorm spreads over every edge, as a gather
 *                                  of Q rows along the reversed graph (built here in the int workspace,
 *                                  pdae_edge_reverse_workspace_ints) + s1 of the forward; dz finished in place.       */
size_t pdae_edge_reverse_workspace_ints(int b, int n, int k);
int pdae_edge_backward_select_f32(const float *z, int ld, const int64_t *idx, const unsigned char *jstar, const float *g,
                                  const float *scale, const float *shift, const float *mean, const float *invstd,
                                  const float *gamma, float slope, int train, int b, int n, int k, int co, double *partial,
                                  float *dz, pdae_stream_t stream);
int pdae_edge_backward_dense_f32(const float *z, int ld, const int64_t *idx, const float *s1, const float *mean,
                                 const float *invstd, const float *ca, const float *cb, int b, int n, int k, int co,
                                 int *workspace, size_t workspace_ints, float *dz, pdae_stream_t stream);

/* The per-channel BatchNorm arithmetic around those kernels, one launch each: partial sums -> batch statistics (training:
 * running buffers updated like nn.BatchNorm2d; train = 0: the running buffers ARE the statistics) -> invstd and the folded
 * scale / shift; and the backward's partial sums -> dgamma, dbeta and the two per-channel terms ca, cb.               */
int pdae_edge_bn_prepare_f32(const double *partial, int np, int co, double m, const float *gamma, const float *beta,
                             float *running_mean, float *running_var, float momentum, float eps, int train, float *mean,
                             float *invstd, float *scale, float *shift, pdae_stream_t stream);
/* partial sums of pdae_edge_stats_shifted_f64: mean = c_o + sum v / M with c_o read from z (b,n,ld), variance
 * sum v^2 / M - (sum v / M)^2.  z may be NULL when train = 0.                                                         */
int pdae_edge_bn_prepare_shifted_f32(const double *partial, int np, int co, double m, const float *z, int ld, const float *gamma,
                                     const float *beta, float *running_mean, float *running_var, float momentum, float eps,
                                     int train, float *mean, float *invstd, float *scale, float *shift, pdae_stream_t stream);
int pdae_edge_bn_backward_f32(const double *partial, int np, int co, double m, const float *gamma, float *dgamma, float *dbeta,
                              float *ca, float *cb, pdae_stream_t stream);

/* The exchange of the sharded forward as one kernel over NVLink peer memory (no collective call): every rank's packed
 * row keys live in a symmetric buffer; rank r reduces rows [lo, hi) (its share) over all ranks' buffers and writes the
 * unpacked (distance, index) pairs into every rank's result buffers.  keys / dist / idx: host arrays of `world` peer-mapped
 * device pointers.  _multimem: the same through the multicast address of the allocation -- the NVSwitch reduces the keys
 * (multimem.ld_reduce.min.u64) and broadcasts the results (multimem.st).  The caller brackets the call with cross-rank
 * barriers.  Results equal pdae_chamfer_unpack_keys of an all-reduce(MIN) bit for bit.                             */
int pdae_chamfer_exchange_keys_peer(const void *const *keys, void *const *dist, void *const *idx, int world, long long lo,
                                    long long hi, pdae_stream_t stream);
int pdae_chamfer_exchange_keys_multimem(const void *mc_keys, void *mc_dist, void *mc_idx, long long lo, long long hi,
                                        pdae_stream_t stream);

/* ---- "next" rows: ball query + grouping (3DETR / PointNet++ configs) ------------------------
 * replaces: `ball_query` ball_query_gpu.cu:12-57, `group_points` / `_grad`
 *           group_points_gpu.cu:11-78 (bindings.cpp:18-21).                                    */
int pdae_ball_query_f32(const float *new_xyz, const float *xyz, int b, int n, int m, float radius, int nsample,
                        int *idx, pdae_stream_t stream);
int pdae_group_points_f32(const float *points, const int *idx, int b, int c, int n, int npoints, int nsample,
                          float *out, pdae_stream_t stream);
int pdae_group_points_grad_f32(const float *gout, const int *idx, int b, int c, int n, int npoints, int nsample,
                               float *gpoints, pdae_stream_t stream);

/* ---- feature propagation: three_nn / three_interpolate (PointNet++ decoder) ------------------
 * replaces: `three_nn` interpolate.cpp:17-46 -> interpolate_gpu.cu:12-72, `three_interpolate` /
 *           `three_interpolate_grad` interpolate.cpp:48-106 -> interpolate_gpu.cu:76-158 (bindings.cpp:14-16).
 * unknown (b,n,3), known (b,m,3) -> dist2 (b,n,3) SQUARED distances ascending (ties -> lower index; +inf and
 * index 0 in slots that never fill when m < 3), idx (b,n,3) int32.
 * points (b,c,m), idx / weight (b,n,3) -> out (b,c,n); grad: gout (b,c,n) -> gpoints (b,c,m) overwritten.   */
int pdae_three_nn_f32(const float *unknown, const float *known, int b, int n, int m, float *dist2, int *idx,
                      pdae_stream_t stream);
int pdae_three_interpolate_f32(const float *points, const int *idx, const float *weight, int b, int c, int m, int n,
                               float *out, pdae_stream_t stream);
int pdae_three_interpolate_grad_f32(const float *gout, const int *idx, const float *weight, int b, int c, int n, int m,
                                    float *gpoints, pdae_stream_t stream);

/* ---- affine corruptions between the patchifier and the encoder (SURVEY.md 8f row 3) ----------------------
 * replaces: the torch chains of `corrupt_scale_nonorm`, `corrupt_tranlate`, `corrupt_rotate_360`,
 *           `corrupt_rotate_z_360`, `corrupt_reflection`, `corrupt_shear` (datasets/corrupt_util_tensor.py:59-343)
 *           as composed by `corrupt_data` (:706-728) and used in models/PointCAE_transformer.py:1011-1017.
 * mats (b,t,3,3): the per-cloud matrices in the order the reference would apply them; a point is a ROW vector,
 * p <- p @ mats[cloud][s] for s = 0..t-1 (fp32, one fma chain per output coordinate, no composition of the
 * matrices, so diagonal steps equal the reference's elementwise products bit for bit).  0 <= t <= 8.
 *
 * pdae_affine_points_f32: points (b,p,3) and center (b,g,3) -> out_points, out_center (may alias the inputs).
 * pdae_group_affine_f32:  the Group tail (see pdae_group_f32) that ALSO emits what the reference's forward
 *   derives from it: neighborhood = ((x - c) + c) - c, t_center = affine(c),
 *   t_neighborhood = affine((x - c) + c) - affine(c), each rounded as the reference's separate kernels round. */
#define PDAE_AFFINE_MAX_CHAIN 8
int pdae_affine_points_f32(const float *points, const float *center, const float *mats, int b, int p, int g, int t,
                           float *out_points, float *out_center, pdae_stream_t stream);
int pdae_group_affine_f32(const float *xyz, const float *center, const float *mats, int b, int n, int g, int m, int t,
                          int64_t *idx, float *neighborhood, float *t_neighborhood, float *t_center,
                          pdae_stream_t stream);
/* FPS + centre gather + the call above in one call (one launch for the shapes of pdae_fps_group_f32): the first seven
 * lines of the reference model's forward, models/PointCAE_transformer.py:1010-1017.  fps_idx (b,g) int32, center (b,g,3). */
int pdae_fps_group_affine_f32(const float *xyz, const float *mats, int b, int n, int g, int m, int t, int *fps_idx,
                              float *center, int64_t *idx, float *neighborhood, float *t_neighborhood, float *t_center,
                              void *workspace, size_t workspace_bytes, pdae_stream_t stream);

/* ---- EdgeConv, eval mode (SURVEY.md 8f row 4; first stage: parity verified on B200, not yet timed) ----------------------
 * replaces: the tail of one EdgeConv layer of `dgcnn_encoder`, models/dgcnn_util.py:114-126: Conv2d(2C,Co,1) over the
 *           graph feature -> BatchNorm2d (running statistics) -> LeakyReLU -> max over the k neighbours, once the
 *           convolution has been split into p = x^T W1^T and q = x^T (W2 - W1)^T (two GEMMs, caller's).
 * p, q (b,n,co) row-major, idx (b,n,k) int64 per-cloud neighbour indices, scale / shift (co) = BatchNorm folded to
 * y*scale + shift, slope = LeakyReLU negative slope.
 * out (b,co,n): out[b][o][i] = act(scale[o] * (ext_j p[b][idx[b][i][j]][o] + q[b][i][o]) + shift[o]),
 * ext = max where scale[o] >= 0, min where scale[o] < 0.                                                        */
int pdae_edge_gather_extremum_f32(const float *p, const float *q, const int64_t *idx, const float *scale,
                                  const float *shift, float slope, int b, int n, int k, int co, float *out,
                                  pdae_stream_t stream);

/* ---- deterministic gradients -------------------------------------------------------------------------------------
 * Twins of the scatter-add gradients whose result is a pure function of the inputs (independent of grid, batch
 * composition, stream and concurrent load): every gradient element starts from its own term (+0 where the op has none)
 * and adds the scattered contributions one by one in ascending order of the source slot's linear index within the
 * cloud, each contribution formed by the same expression as the atomic form, with rounded fp32 products and adds.
 * Each takes a workspace of its own *_workspace_bytes query, builds ordered reverse maps there and writes every
 * target once; no float atomics, no allocation, no host synchronisation (capturable).  Same argument rules and
 * outputs as the atomic forms.  Orders:
 *   chamfer (both forms)  point i of cloud 1: g_i (a_i - b[idx1[i]]), then -v_j for every j of cloud 2 with
 *                         idx2[j] == i, j ascending; cloud 2 symmetric
 *   pair loss             the own term, then the matched rows' terms, source ascending
 *   gather grad           source j ascending
 *   group_points grad     source slot q * nsample + k ascending
 *   three_interpolate     slot i * 3 + s ascending (terms rn(gout * weight))
 *   graph feature grad    the centre term of row j (p ascending), then G[i][p][0:c] for every edge with
 *                         idx[i][p] == j, slot i * k + p ascending                                                   */
size_t pdae_chamfer_bwd_det_workspace_bytes(int b, int n, int m); /* both Chamfer forms */
int pdae_chamfer_bwd_det_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2, const float *gd1,
                             const float *gd2, int b, int n, int m, float *gx1, float *gx2, void *workspace,
                             size_t workspace_bytes, pdae_stream_t stream);
int pdae_chamfer_loss_bwd_det_f32(const float *xyz1, const float *xyz2, const int *idx1, const int *idx2, const float *dist1,
                                  const float *dist2, const float *gloss, float w1, float w2, int b, int n, int m, int l1,
                                  float *gx1, float *gx2, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_pair_loss_bwd_det_workspace_bytes(int bs, int n, int m);
int pdae_pair_loss_bwd_det_f32(const float *a, const float *b, const int *idx1, const int *idx2, const float *gloss, float w1,
                               float w2, int bs, int n, int m, int d, int metric, float *ga, float *gb, void *workspace,
                               size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_gather_grad_det_workspace_bytes(int b, int n, int m);
int pdae_gather_grad_det_f32(const float *gout, const int *idx, int b, int c, int n, int m, float *gfeat, void *workspace,
                             size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_group_points_grad_det_workspace_bytes(int b, int n, int npoints, int nsample);
int pdae_group_points_grad_det_f32(const float *gout, const int *idx, int b, int c, int n, int npoints, int nsample,
                                   float *gpoints, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_three_interpolate_grad_det_workspace_bytes(int b, int n, int m);
int pdae_three_interpolate_grad_det_f32(const float *gout, const int *idx, const float *weight, int b, int c, int n, int m,
                                        float *gpoints, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_graph_feature_grad_det_workspace_bytes(int b, int c, int n, int k);
int pdae_graph_feature_grad_det_f32(const float *gout, const int64_t *idx, int b, int c, int n, int k, float *gx,
                                    void *workspace, size_t workspace_bytes, pdae_stream_t stream);

/* The reverse index those gradients gather through, on its own: idx (b,s) int32 or int64 with targets in [0,t) ->
 * ptr (b,t+1) bucket offsets within the cloud, slot (b,s) the source slots of each bucket in ascending order, i.e. a
 * stable argsort of each cloud's targets.  Sources outside [0,t) are left out (ptr[t] counts the others; slot entries
 * past it are not written).  Buckets are sorted by one thread up to 32 slots, by one CTA in shared memory up to 8192,
 * by one CTA's ordered compaction of the cloud beyond.  Workspace: pdae_reverse_index_workspace_bytes.              */
size_t pdae_reverse_index_workspace_bytes(int b, int s, int t);
int pdae_reverse_index_i32(const int32_t *idx, int b, int s, int t, int *ptr, int *slot, void *workspace,
                           size_t workspace_bytes, pdae_stream_t stream);
int pdae_reverse_index_i64(const int64_t *idx, int b, int s, int t, int *ptr, int *slot, void *workspace,
                           size_t workspace_bytes, pdae_stream_t stream);

/* pdae_step_f32 with a flags word (pdae_step_f32 is this call with flags = 0).  PDAE_STEP_DETERMINISTIC: the backward on
 * the side stream is pdae_chamfer_loss_bwd_det_f32; everything else is unchanged.  Workspace:
 * pdae_step_ex_workspace_bytes with the same flags.                                                                  */
#define PDAE_STEP_DETERMINISTIC 1u
size_t pdae_step_ex_workspace_bytes(int b, int n, int g, int m, unsigned flags);
int pdae_step_ex_f32(const float *cloud, const float *pred, int b, int n, int g, int m, int *fps_idx, float *center,
                     float *neighborhood, float *dist1, float *dist2, int *idx1, int *idx2, float *loss3, const float *gloss,
                     float *gpred, float *gcloud, void *workspace, size_t workspace_bytes, unsigned flags,
                     pdae_stream_t stream);

/* ---- Earth Mover's Distance (approxmatch / matchcost / matchcostgrad) -------------------------------------------
 * replaces: the reference's extensions/emd (`emd_cuda`: approxmatch_forward, matchcost_forward, matchcost_backward;
 *           Fan et al. 2017, tf_approxmatch_g.cu), which includes THC and does not build with current torch.
 * xyz1 (b,n,3), xyz2 (b,m,3) fp32; 1 <= n, m <= 65536 (PDAE_E_UNSUPPORTED beyond).  Per cloud:
 *   masses     n >= m: remainL = 1, remainR = n / m; else remainL = m / n, remainR = 1 (integer divisions)
 *   levels     j = 0..9: level = -4^(7-j) for j < 9, 0 for j = 9; c_j = rn(level * 1.44269504f)
 *   distance   d(k,l) = fma(dz,dz, fma(dy,dy, rn(dx*dx))), dx = x2_l - x1_k (rounded fp32 differences)
 *   pair term  e = ex2.approx.ftz(rn(c_j * d))
 *   pass 1     ratioL[k] = remainL[k] / s,  s = fma(e, remainR[l], s) for l ascending from s = 1e-9f
 *   pass 2     t = fma(e, ratioL[k], t) for k ascending from +0; sumr = rn(t * remainR[l]);
 *              ratioR[l] = rn(fminf(remainR[l] / (sumr + 1e-9f), 1) * remainR[l]); remainR[l] = fmaxf(0, remainR[l] - sumr)
 *   pass 3     w(k,l) = rn(rn(e * ratioL[k]) * ratioR[l]); u = u + w for l ascending from +0; remainL[k] = fmaxf(0, remainL[k] - u)
 *   match      match[l][k] = sum_j w_j(k,l) added in level order from +0, layout (b,m,n)
 *   cost       rowcost[l] = fma(sqrtf(d), match[l][k], .) for k ascending from +0; then per cloud, thread t < 256 of
 *              one CTA adds rowcost[t + 256 i] for ascending i from +0 and the 256 partials reduce as
 *              p[t] = p[t] + p[t + s] for s = 128, 64, ..., 1; cost = p[0] (no normalisation)
 *   gradient   match held constant: grad1[k] = rn(g_b * a), a = fma(rn(match[l][k] * rsqrtf(fmaxf(d, 1e-20))), x1_k - x2_l, a)
 *              per coordinate for l ascending from +0; grad2[l] likewise over k ascending with x2_l - x1_k
 * Every row and column sum is one sequential chain, so the results do not depend on the grid, the batch or the stream
 * and need no atomics (bit-reproducible with or without torch.use_deterministic_algorithms).
 * pdae_emd_match_f32 stores the per-level ratios ratio_l (b,10,n) and ratio_r (b,10,m) instead of the (b,m,n) match;
 * `match` may be null, else the match is also written (one pass from the ratios, 64-bit offsets).  Cost and gradient
 * read the caller's `match` when it is non-null (the ratios are then ignored and may be null) and rebuild it from the
 * ratios, bit for bit, otherwise.  Workspace: pdae_emd_workspace_bytes (match and cost; the gradient needs none).     */
size_t pdae_emd_workspace_bytes(int b, int n, int m);
int pdae_emd_match_f32(const float *xyz1, const float *xyz2, int b, int n, int m, float *ratio_l, float *ratio_r, float *match,
                       void *workspace, size_t workspace_bytes, pdae_stream_t stream);
int pdae_emd_cost_f32(const float *xyz1, const float *xyz2, int b, int n, int m, const float *match, const float *ratio_l,
                      const float *ratio_r, float *cost, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
int pdae_emd_cost_grad_f32(const float *grad_cost, const float *xyz1, const float *xyz2, int b, int n, int m,
                           const float *match, const float *ratio_l, const float *ratio_r, float *grad1, float *grad2,
                           pdae_stream_t stream);

/* ---- variable-size clouds in one batch: segment FPS and segment kNN (parity unpinned) --------------------------
 * replaces: the reference's extensions/pointops (`pointops_cuda`: furthestsampling_cuda, knnquery_cuda; published
 *           PointTransformer lib/pointops), which includes THC and does not build with current torch.  The reference
 *           source is not in this tree: the semantics below restate the published kernels.
 * Packed layout: xyz (n_total,3) fp32 holds the clouds back to back; offset (b,) int32 holds the cumulative ends,
 * segment s = [offset[s-1], offset[s]) with offset[-1] = 0; new_offset (b,) likewise for samples / queries.  Offsets
 * are device pointers and are only read on the device (no call synchronises with the host); they are expected to be
 * non-decreasing and every value is clamped into [0, n_total] / [0, m_total], so no access leaves the tensors.
 * Every index written is global (a row of the packed xyz).
 * FPS (pdae_seg_fps_f32; idx (m_total,) int32, tmp (n_total,) fp32 or null):
 *   first sample of segment s: idx[start_m] = start_n; sample j folds d = fma(dz,dz, fma(dx,dx, rn(dy*dy))),
 *   dx = x_k - x_prev, into tmp[k] = fminf(d, tmp[k]) and takes the arg-max over the segment: a point counts when
 *   tmp[k] > -1 (the reference's `d2 > best` from best = -1; there is no |p|^2 <= 1e-3 skip).  Ties go to the smallest
 *   bitrev_lg(bs)((k - start_n) mod bs), then to the smaller k, bs = min(1024, 2^floor(log(n)/log(2))) (1 for n = 0).
 *   `n` (the reference passes the largest segment size) sets the tie rule and the kernel form only: segments larger
 *   than n are still exact.  tmp starts from the caller's contents (the reference fills 1e10) and on exit holds the
 *   minima folded with every sample but the last; tmp = null starts from 1e10, writes nothing back and needs
 *   pdae_seg_fps_workspace_bytes(n_total) of workspace.  A segment without points writes start_n for all of its
 *   samples; a segment without samples writes nothing.  PDAE_E_UNSUPPORTED when n_total >> log2(bs) >= 2^22.
 * kNN (pdae_seg_knn_f32; new_xyz (m,3), idx / dist2 (m, nsample) int32 / fp32, 1 <= nsample <= 100):
 *   query p belongs to the first segment s with p < new_offset[s] and searches the points of that segment only;
 *   d^2 = fma(dz,dz, fma(dy,dy, rn(dx*dx))), dx = x_k - x_p (the rounding of pdae_knn_f32).  The row holds the
 *   nsample smallest (d^2, index) pairs with d^2 < 1e10, ascending; the rest of the row is (1e10, start_n).  (The
 *   reference's heap can resolve exact ties at the k-th distance differently; this order is the definition here.)
 *   Rows p >= max(new_offset) hold idx -1 and dist2 1e10.  Workspace: pdae_seg_knn_workspace_bytes(b, m).
 * No atomics: the results depend on the inputs only, not on the launch shape or the stream.                      */
size_t pdae_seg_fps_workspace_bytes(int n_total);
int pdae_seg_fps_f32(const float *xyz, int n_total, const int *offset, const int *new_offset, int b, int n, int m_total,
                     float *tmp, int *idx, void *workspace, size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_seg_knn_workspace_bytes(int b, int m);
int pdae_seg_knn_f32(const float *xyz, int n_total, const float *new_xyz, int m, const int *offset, const int *new_offset,
                     int b, int nsample, int *idx, float *dist2, void *workspace, size_t workspace_bytes,
                     pdae_stream_t stream);

/* ---- Chamfer distance over variable-size clouds in one batch (segment forward, gradients, mean losses) -----------
 * xyz1 (n_total,3), xyz2 (m_total,3) fp32 packed as above; offset1 / offset2 (b,) int32 cumulative ends (device).
 * Segments: row p of xyz1 belongs to the first segment s with p < offset1[s] after clamping into [0, n_total] (the rule
 * of the segment kNN's queries), i.e. segment s = [end1[s-1], end1[s]) with end1[s] = max(offset1[0..s]) clamped; for
 * non-decreasing offsets that is [offset1[s-1], offset1[s]).  Likewise xyz2.  Segments never overlap, whatever the
 * offsets.  Segment s of xyz1 is matched only against segment s of xyz2.
 * Forward (pdae_seg_chamfer_fwd_f32): dist1 (n_total,) / dist2 (m_total,) fp32 squared distances, idx1 / idx2 int32
 *   GLOBAL row indices.  d = fma(dz,dz, fma(dx,dx, rn(dy*dy))), d* = b - a, minimum over the opposite segment, ties to
 *   the lowest index: the rounding and tie rule of pdae_chamfer_fwd_f32, so equal segments give its (b,n,3) result bit
 *   for bit with idx + s*m.  A point whose opposite segment is empty, or that lies past the last segment, gets dist 0
 *   and idx -1.  Workspace: pdae_seg_chamfer_fwd_workspace_bytes(b, n_total, m_total).
 * Backward (pdae_seg_chamfer_bwd_f32 / _det_f32): the equal-size backward at b = 1 over the packed arrays (same terms,
 *   same orders; _det adds the terms of the points that chose a point in ascending source order); a row with idx -1
 *   has no own term.  _det workspace: pdae_seg_chamfer_bwd_det_workspace_bytes(n_total, m_total).
 * Mean losses (pdae_seg_chamfer_loss_f32): S = the segments with both sides non-empty.  loss3 = [loss, term1, term2],
 *   term1 = (1/|S|) sum_{s in S} mean_s f(dist1), term2 likewise, f = identity (L2) or sqrt (L1); loss = term1 + term2
 *   (L2) or (term1 + term2) / 2 (L1), sqrt in fp32.  |S| = 0 gives 0 everywhere.  Per-segment sums in float64 in a
 *   fixed order, then one fixed-order float64 pass over the segments: deterministic.  state (4b + 1,) int32 receives
 *   [|S|, end1 (b), end2 (b), weight1 (b), weight2 (b)] (weights as fp32 bits, see below) for the backward.
 *   Workspace: pdae_seg_chamfer_loss_workspace_bytes(b).
 * Loss backward (pdae_seg_chamfer_loss_bwd_f32 / _det_f32, `state` from the loss): the backward above with
 *   d(loss)/d(dist) of a point of segment s = rn(gloss * weight_s), weight_s = rn(w / (float)(|S| * size_s)),
 *   w = 1 (L2) or 0.5 (L1), |S| * size_s formed in 64 bits
 *   (the rounding of pdae_chamfer_loss_bwd_f32, where it is b * n), divided by 2 sqrt(dist) for L1 (dist 0 gives inf,
 *   NaN after the multiply by 0, like SqrtBackward).  _det workspace: pdae_seg_chamfer_bwd_det_workspace_bytes.
 * b = 0: the forward, the loss and the loss backward return 0 and write nothing.  No call synchronises with the host;
 * the forward and the loss use no float atomics, so their results depend on the inputs only.                      */
size_t pdae_seg_chamfer_fwd_workspace_bytes(int b, int n_total, int m_total);
int pdae_seg_chamfer_fwd_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                             const int *offset2, int b, float *dist1, float *dist2, int *idx1, int *idx2, void *workspace,
                             size_t workspace_bytes, pdae_stream_t stream);
int pdae_seg_chamfer_bwd_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1, const int *idx2,
                             const float *gd1, const float *gd2, float *gx1, float *gx2, pdae_stream_t stream);
size_t pdae_seg_chamfer_bwd_det_workspace_bytes(int n_total, int m_total);
int pdae_seg_chamfer_bwd_det_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1,
                                 const int *idx2, const float *gd1, const float *gd2, float *gx1, float *gx2, void *workspace,
                                 size_t workspace_bytes, pdae_stream_t stream);
size_t pdae_seg_chamfer_loss_workspace_bytes(int b);
int pdae_seg_chamfer_loss_f32(const float *dist1, int n_total, const float *dist2, int m_total, const int *offset1,
                              const int *offset2, int b, int l1, float *loss3, int *state, void *workspace,
                              size_t workspace_bytes, pdae_stream_t stream);
int pdae_seg_chamfer_loss_bwd_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1,
                                  const int *idx2, const float *dist1, const float *dist2, const int *state, int b,
                                  const float *gloss, int l1, float *gx1, float *gx2, pdae_stream_t stream);
int pdae_seg_chamfer_loss_bwd_det_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *idx1,
                                      const int *idx2, const float *dist1, const float *dist2, const int *state, int b,
                                      const float *gloss, int l1, float *gx1, float *gx2, void *workspace,
                                      size_t workspace_bytes, pdae_stream_t stream);

/* ---- Earth Mover's Distance over variable-size clouds in one batch (segment approxmatch, cost, gradient) --------
 * xyz1 (n_total,3), xyz2 (m_total,3) fp32 packed; offset1 / offset2 (b,) int32 cumulative ends (device).  Segments:
 * the rule of the segment Chamfer above (end[s] = max(clamp(offset[0..s]))); segment s of xyz1 is matched only against
 * segment s of xyz2.  Per segment with n_s, m_s >= 1: exactly the arithmetic and orders of pdae_emd_* above at b = 1
 * (masses from the integer divisions of n_s and m_s, the ten levels with ex2.approx.ftz, the three passes, the cost as a
 * per-column chain then 256 strided chains and the fixed pairwise tree, the gradient chains with rsqrtf times
 * grad_cost[s]), indices relative to the segment start.  So every segment's ratios, cost and gradients equal those of
 * pdae_emd_* on that segment's slices at b = 1, bit for bit, and equal segments give the batched (b,n,3) results.
 * Ratios: ratio_l (10, n_total), ratio_r (10, m_total), level-major: level j of point p at j * n_total + p (equal
 * segments: ratio_l viewed (10,b,n) and transposed to (b,10,n) is the equal-size layout).  There is no match output:
 * cost and gradient rebuild it from the ratios.
 * A segment with an empty side has cost 0, and every point of it gets ratios 0 and gradient 0; so do the points past
 * the last segment.  b = 0: return 0 and write nothing.  No per-segment size cap (the equal-size 65536 stays there):
 * one segment runs on one cluster of at most 8 CTAs, so its time grows with n_s * m_s.  n_total, m_total above
 * 2^31 / 10 give PDAE_E_UNSUPPORTED.  Each call runs its own pre-pass over the offsets; none synchronises with the host.
 * No atomics: the results depend on the inputs only, not on the launch shape, the stream or the deterministic flag.
 * Workspace (all three calls): pdae_seg_emd_workspace_bytes(b, n_total, m_total).                                */
size_t pdae_seg_emd_workspace_bytes(int b, int n_total, int m_total);
int pdae_seg_emd_match_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                           const int *offset2, int b, float *ratio_l, float *ratio_r, void *workspace, size_t workspace_bytes,
                           pdae_stream_t stream);
int pdae_seg_emd_cost_f32(const float *xyz1, int n_total, const float *xyz2, int m_total, const int *offset1,
                          const int *offset2, int b, const float *ratio_l, const float *ratio_r, float *cost, void *workspace,
                          size_t workspace_bytes, pdae_stream_t stream);
int pdae_seg_emd_cost_grad_f32(const float *grad_cost, const float *xyz1, int n_total, const float *xyz2, int m_total,
                               const int *offset1, const int *offset2, int b, const float *ratio_l, const float *ratio_r,
                               float *grad1, float *grad2, void *workspace, size_t workspace_bytes, pdae_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* POINTDAE_B200_H */
