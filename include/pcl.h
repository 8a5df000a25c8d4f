/*
 * pcl.h -- C ABI of libpcl_b200.so: the point-cloud reconstruction-loss hot path
 * (Chamfer distance and auction EMD, forward + backward) for NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the native layer the reference reaches through
 *   - the pybind11 module `emd` (pointcloud_vision/loss/emd/emd.cpp:28-31: forward/backward,
 *     implemented in loss/emd/emd_cuda.cu:228-316) and
 *   - pytorch3d's `_C.knn_points_idx` / `_C.knn_points_backward` under
 *     `pytorch3d.loss.chamfer_distance` (call sites pointcloud_vision/utils.py:211,228).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless its name ends in `_host`;
 *     the library never allocates or frees device memory (reference: caller-allocates,
 *     emd_module.py:45-56) -- scratch is one opaque workspace sized by *_workspace_bytes();
 *   - point arrays are (B, P, D) with element strides (batch_stride, row_stride) and unit
 *     channel stride, so strided views such as pred[:, :, :3] (utils.py:254) need no copy;
 *     `dtype` selects the element type of such an input: PCL_F32, PCL_F16 or PCL_BF16 (the
 *     kernels up-cast exactly like `.float()`, emd_module.py:43-44); outputs are fp32 / int32;
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream, which is what the reference uses, emd_cuda.cu:257-269);
 *   - return value: 0 = ok, negative = error (PCL_E_*), text via pcl_last_error() (thread-local).
 *     The reference printf()s and returns -1/0/1 (emd_cuda.cu:236-249,276-281); no printf here.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef PCL_B200_H
#define PCL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCL_VERSION 100 /* major*100 + minor */

#if defined(__GNUC__)
#define PCL_API __attribute__((visibility("default")))
#else
#define PCL_API
#endif

enum { PCL_F32 = 0, PCL_F16 = 1, PCL_BF16 = 2 };

enum {
    PCL_OK = 0,
    PCL_E_SHAPE = -1,     /* bad sizes (reference: emd_cuda.cu:236-249 returns -1) */
    PCL_E_ARG = -2,       /* null pointer / bad enum */
    PCL_E_CUDA = -3,      /* a CUDA call or launch failed (reference returns 0, emd_cuda.cu:276-281) */
    PCL_E_WORKSPACE = -4, /* workspace too small */
    PCL_E_UNSUPPORTED = -5
};

/* Chamfer arithmetic: how one squared distance is rounded (see DESIGN.md "Chamfer arithmetic"). */
enum {
    PCL_CHAMFER_UNFUSED = 0, /* ((dx*dx)+dy*dy)+dz*dz -- pytorch3d CPU build; the default */
    PCL_CHAMFER_FMA = 1      /* fma(dz,dz,fma(dy,dy,dx*dx)) -- what nvcc makes of pytorch3d's knn.cu */
};

PCL_API int pcl_version(void);
PCL_API const char *pcl_last_error(void);
/* Number of SMs / compute capability of the current device, for sizing and for the bench roofline. */
PCL_API int pcl_device_info(int *sm_count, int *cc_major, int *cc_minor, int *max_smem_optin);

/* ------------------------------------------------------------------ Chamfer ------------------------------- */
/*
 * Replaces pytorch3d.loss.chamfer_distance(x, y, x_lengths, y_lengths)[0] forward
 * (utils.py:211,228): two directed K=1 nearest-neighbour searches with squared L2, lowest index
 * on exact ties, padded rows ignored, then point mean and batch mean.
 *   x (B,P1,D), y (B,P2,D); x_len / y_len: nullable int64[B] (entries in [0,P]); 1 <= D <= 8.
 *   dist_x,idx_x: (B,P1)  dist_y,idx_y: (B,P2)   (padded rows: 0 / 0)
 *   loss_xy[4] = { sum_n mean_i dist_x / max(B,1), same for y,  sum_n mean_i dist_x, same for y }
 *   (loss = loss_xy[0]+loss_xy[1]; [2..3] are the un-normalised batch sums a batch-sharded caller all-reduces)
 */
/*
 * D == 3 has two forward implementations with identical results: a brute-force scan of all P1*P2 pairs, and -- for clouds of at
 * least `min_points` (default 6144) and at most 16384 points -- a spatially pruned one (both clouds in Morton order, 32-point tiles
 * with bounding boxes, only the tiles that can hold a nearer point are scanned).  pcl_chamfer_set_prune_min moves the switch-over
 * (0: never prune, < 0: default); a tuning knob, process-wide.
 */
PCL_API int pcl_chamfer_set_prune_min(int min_points);
PCL_API size_t pcl_chamfer_workspace_bytes(int B, int P1, int P2);
PCL_API int pcl_chamfer_fwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                    const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len,
                    int B, int P1, int P2, int D, int mode,
                    float *dist_x, int32_t *idx_x, float *dist_y, int32_t *idx_y, float *loss_xy,
                    void *workspace, size_t workspace_bytes, void *stream);
/*
 * Replaces pytorch3d's knn_points_backward applied to both directions plus the mean reductions:
 *   gdx = g[0] / max(B,1) / clamp(x_len,1);  grad_x[i] += 2*gdx*(x_i - y[idx_x[i]]);  grad_y[idx_x[i]] -= same
 *   and symmetrically for the y direction with g[1].  `grad_out` is a DEVICE float[2]: the upstream
 * gradients of loss_xy[0] and loss_xy[1] (no host sync).  grad_x (B,P1,D), grad_y (B,P2,D) are dense
 * fp32 and are overwritten.
 */
PCL_API int pcl_chamfer_bwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                    const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len,
                    int B, int P1, int P2, int D, const int32_t *idx_x, const int32_t *idx_y,
                    const float *grad_out, float *grad_x, float *grad_y, void *stream);

/* ------------------------------------------------------------------ EMD (auction) ------------------------- */
/*
 * Replaces emd.forward (emd.cpp:14-18 -> emd_cuda_forward, emd_cuda.cu:228-282): `iters` rounds of
 * {list unassigned, Bid, GetMax, Assign} then CalcDist, all inside ONE persistent kernel.
 *   xyz1 = prediction (B,N,3) (receives the gradient), xyz2 = target (B,N,3), both in [0,1]^3.
 *   dist (B,N) fp32 = squared distance to the matched target, assignment (B,N) int32.
 *   stats: nullable int32[B*8] = { sum_t U_t, iterations run, GetMax multi-bidder events, cluster size,
 *          executed pair evaluations (lo, hi 32 bits; tiles skipped by the spatial pruning are not counted),
 *          launch flags, tiles per cloud }.
 * Constraints: 1 <= N <= pcl_emd_max_points() (8192: the reference's own demo size, emd_module.py:82), B >= 0
 * (the reference needs N%1024==0 and B<=512, emd_cuda.cu:241-249; both are accepted here, neither is required).
 * Up to 3584 points the whole auction state lives in shared memory; above, half of it lives in `workspace`
 * (>= pcl_emd_workspace_bytes(B, N), which then is tens of MB).
 * The GetMax race of the reference (emd_cuda.cu:188-191) is resolved deterministically: the
 * largest bidder index inside the +-1e-6 window wins.
 *
 * Three paths implement the same auction bit for bit (stats[3] tells which kind ran: cluster size, or 0 for the team path):
 *   cluster path: one thread-block cluster of 1..16 CTAs per cloud for the whole auction (pcl_emd.cu);
 *   team path:    one owner CTA per cloud + worker CTAs on all other SMs that execute Bid tasks of whichever cloud is
 *                 furthest behind (pcl_emd_team.cu);
 *   tickets path: the cluster kernel, whose many-bidder iterations are shared as tasks with worker CTAs on the SMs the
 *                 clusters leave free and with the clusters that are already done (pcl_emd.cu + pcl_emd_team.cu).
 * The team and tickets paths need N <= 3584, B < SM count and a workspace of pcl_emd_workspace_bytes.  Where they are possible,
 * AUTO takes the team path for N >= 3072 and B >= 8, else the tickets path for N >= 1536 when the clusters have at most 2 CTAs,
 * else the cluster path.  pcl_emd_set_path forces one path for the calls that follow (process-wide; for parity tests and A/B
 * timing); a forced team or tickets path that is not possible fails with PCL_E_UNSUPPORTED.
 */
enum { PCL_EMD_PATH_AUTO = 0, PCL_EMD_PATH_CLUSTER = 1, PCL_EMD_PATH_TEAM = 2, PCL_EMD_PATH_TICKETS = 3 };
PCL_API int pcl_emd_set_path(int path);
PCL_API int pcl_emd_max_points(void);
PCL_API size_t pcl_emd_workspace_bytes(int B, int N);
PCL_API int pcl_emd_fwd(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1,
                const void *xyz2, int dtype2, int64_t bs2, int64_t rs2,
                int B, int N, float eps, int iters,
                float *dist, int32_t *assignment, int32_t *stats,
                void *workspace, size_t workspace_bytes, void *stream);
/*
 * pcl_emd_fwd with the loss epilogue of the UNWEIGHTED EarthMoverDistance fused into the same kernel (utils.py:304 with
 * weights == 1 -- the Autoencoder loss, train.py:82 -- followed by emdFunction.backward, emd_module.py:63-72):
 *   sums (nullable, device float[3]) = { sum_{b,j} sqrt(dist), B*N, their ratio = the reference's point_l };
 *   grad_xyz1 (nullable, (B,N,3) fp32) = grad_scale * d(sum sqrt(dist)) / d xyz1
 *             = 2 * (grad_scale / (2*sqrt(dist))) * (xyz1 - xyz2[assignment])   (torch's sqrt backward, then emd_cuda.cu:284-300),
 *   so grad_scale = upstream gradient / (B_global*N) yields the final gradient of the loss and no backward kernel is left.
 * The sum is formed in fp64 in a fixed order (per-CTA partials + last-CTA ticket inside `workspace`, which is then
 * required: >= pcl_emd_workspace_bytes(B, N)); dist == 0 gives inf/nan exactly like the reference's dists.sqrt().
 */
PCL_API int pcl_emd_fwd_fused(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1,
                      const void *xyz2, int dtype2, int64_t bs2, int64_t rs2,
                      int B, int N, float eps, int iters,
                      float *dist, int32_t *assignment, int32_t *stats,
                      float grad_scale, float *grad_xyz1, float *sums,
                      void *workspace, size_t workspace_bytes, void *stream);
/*
 * Replaces emd.backward (emd.cpp:20-23 -> NmDistanceGradKernel, emd_cuda.cu:284-316):
 *   grad_xyz1[j] = (2*graddist[j]) * (xyz1[j] - xyz2[assignment[j]]);  the target gets no gradient
 *   (emd_module.py:69,72).  grad_xyz1 (B,N,3) dense fp32, overwritten (no zero-fill needed).
 */
PCL_API int pcl_emd_bwd(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1,
                const void *xyz2, int dtype2, int64_t bs2, int64_t rs2,
                int B, int N, const int32_t *assignment, const float *graddist,
                float *grad_xyz1, void *stream);

/*
 * Loss epilogue of EarthMoverDistance (utils.py:257-304), fused.
 * pcl_emd_match_hist: hist[c] += #{(b,j): label(target[b, assignment[b,j]]) == c}  (utils.py:271-275;
 *   the histogram of the PERMUTED target).  target_label: the channel holding the class id as a float
 *   (target[..., 3]) given as pointer + strides; hist: int64[C], zeroed by the callee.
 *   matched_label (nullable, B*N int32) receives the permuted labels for the cross-entropy term.
 * pcl_emd_weighted_reduce: sums[0] = sum w*sqrt(dist), sums[1] = sum w, with
 *   w = class_weights[matched_label] (or 1 when class_weights == NULL)  (utils.py:292,304).
 */
PCL_API int pcl_emd_match_hist(const void *target_label, int dtype, int64_t bs, int64_t rs,
                       const int32_t *assignment, int B, int N, int C,
                       int64_t *hist, int32_t *matched_label, void *stream);
PCL_API int pcl_emd_weighted_reduce(const float *dist, const int32_t *matched_label, const float *class_weights,
                            int B, int N, int C, float *sums,
                            void *workspace /* >= pcl_emd_workspace_bytes(B,N) */, size_t workspace_bytes, void *stream);
/*
 * Backward of point_l = sums[0]/sums[1] through sqrt and the auction distance, fused with pcl_emd_bwd:
 *   graddist = g * w / (2*sqrt(dist)) / sums[1]   =>   grad_xyz1 = 2*graddist*(xyz1 - xyz2[assignment]).
 * dist == 0 gives inf/nan exactly like the reference's dists.sqrt() (utils.py:304).
 */
PCL_API int pcl_emd_weighted_bwd(const void *xyz1, int dtype1, int64_t bs1, int64_t rs1,
                         const void *xyz2, int dtype2, int64_t bs2, int64_t rs2,
                         int B, int N, const int32_t *assignment, const float *dist,
                         const int32_t *matched_label, const float *class_weights, int C,
                         const float *sums, const float *grad_out, float *grad_xyz1, void *stream);

/*
 * Feature term of EarthMoverDistance, fused (replaces the torch ops of pointcloud_vision/utils.py:278-279,293-301;
 * SURVEY.md 8f row 2).  Both forward calls return (numerator, denominator) in sums[0..1] so that a batch-sharded caller
 * can all-reduce them before dividing; accumulation is fp64 in a fixed order.  workspace >= pcl_emd_feature_workspace_bytes().
 *
 * pcl_emd_seg_ce_fwd (Segmenter, utils.py:293-295): logits (B,N,C) given as pointer + strides (pred[..., 3:]),
 *   matched_label = labels of the matched targets (pcl_emd_match_hist), class_weights float[C]:
 *   sums[0] = sum_i w_i * (logsumexp(logits_i) - logits_i[label_i]), sums[1] = sum_i w_i, w_i = class_weights[label_i]
 *   (F.cross_entropy(..., weight=class_weights) == sums[0] / sums[1]).  pred_hist (nullable int64[C], zeroed by the
 *   callee) receives the histogram of argmax_c logits (first maximum), the input of the logged KL term (utils.py:278-279).
 *   C <= 64.
 * pcl_emd_seg_ce_bwd: grad_logits (B,N,C) dense fp32 = grad_sums[0] * w_i * (softmax(logits_i) - onehot(label_i));
 *   grad_sums is a DEVICE pointer (the upstream gradient of sums[0]).
 * pcl_emd_feat_mse_fwd (Autoencoder, utils.py:257-258,301): sums[0] = sum (feat[b,i,f] - tfeat[b,assignment[b,i],f])^2,
 *   sums[1] = B*N*F  (F.mse_loss of the prediction against the permuted target == sums[0] / sums[1]).
 * pcl_emd_feat_mse_bwd: grad_feat (B,N,F) dense fp32 = grad_sums[0] * 2 * (feat - tfeat[assignment]).
 */
PCL_API size_t pcl_emd_feature_workspace_bytes(void);
PCL_API int pcl_emd_seg_ce_fwd(const void *logits, int dtype, int64_t bs, int64_t rs, const int32_t *matched_label,
                       const float *class_weights, int B, int N, int C, float *sums, int64_t *pred_hist,
                       void *workspace, size_t workspace_bytes, void *stream);
PCL_API int pcl_emd_seg_ce_bwd(const void *logits, int dtype, int64_t bs, int64_t rs, const int32_t *matched_label,
                       const float *class_weights, int B, int N, int C, const float *grad_sums, float *grad_logits,
                       void *stream);
PCL_API int pcl_emd_feat_mse_fwd(const void *feat, int dtype1, int64_t bs1, int64_t rs1,
                         const void *tfeat, int dtype2, int64_t bs2, int64_t rs2,
                         const int32_t *assignment, int B, int N, int F, float *sums,
                         void *workspace, size_t workspace_bytes, void *stream);
PCL_API int pcl_emd_feat_mse_bwd(const void *feat, int dtype1, int64_t bs1, int64_t rs1,
                         const void *tfeat, int dtype2, int64_t bs2, int64_t rs2,
                         const int32_t *assignment, int B, int N, int F,
                         const float *grad_sums, float *grad_feat, void *stream);

/*
 * Per-cloud class filter of a labelled target for FilteringChamferDistance (utils.py:110-124,222-226; SURVEY.md 8f row 4):
 * for every cloud the rows whose label -- target[..., label_channel] truncated to an integer, as `.long()` -- is one of
 * `labels` (a HOST array of n_labels <= 16 values) are copied, in order, to the front of out_xyz[b] ((B,N,3) fp32, the rest
 * zero-filled like F.pad) and lengths[b] (int64, device) receives their number: the (points, y_lengths) pair
 * chamfer_distance takes, without the reference's per-cloud Python loop and without a host synchronisation.
 */
PCL_API int pcl_class_filter(const void *target, int dtype, int64_t bs, int64_t rs, int B, int N, int label_channel,
                     const int64_t *labels, int n_labels, float *out_xyz, int64_t *lengths, void *stream);

/* ------------------------------------------------------------------ sampling (SURVEY.md 8f rows 1, 3) ------ */
/*
 * Farthest point sampling: replaces pointnet2_ops._ext.furthest_point_sampling (models/pointnet2_utils.py:6,89-90)
 * and pytorch3d.ops.sample_farthest_points (utils.py:10,90; models/pointmlp.py:158) -- third-party code that is not
 * part of the reference tree; semantics = the torch algorithm kept as a comment in pointnet2_utils.py:64-86 with
 * start index 0 (or start_idx[b]) and the lowest index on ties.  idx_out: int32 (B, npoint).
 * skip_origin != 0: points with x*x+y*y+z*z <= 1e-3 are never selected (pointnet2_ops' padding convention).
 */
PCL_API int pcl_fps_max_points(void);
PCL_API int pcl_fps(const void *xyz, int dtype, int64_t bs, int64_t rs, int B, int N, int npoint,
            const int32_t *start_idx /* nullable */, int skip_origin, int32_t *idx_out, void *stream);
/*
 * Ball query: replaces query_ball_point(radius, nsample, xyz, new_xyz) (models/pointnet2_utils.py:93-113): for every
 * centroid the first `nsample` point indices (ascending) with squared distance <= radius2, padded with the first
 * hit; N when nothing is inside.  group_idx: int32 (B, S, nsample).  radius2 = (float)(radius**2).
 */
PCL_API int pcl_ball_query(const void *xyz, int dtype, int64_t bs, int64_t rs,
                   const void *new_xyz, int ndtype, int64_t nbs, int64_t nrs,
                   int B, int N, int S, float radius2, int nsample, int32_t *group_idx, void *stream);

/* ------------------------------------------------------------------ composite step ------------------------ */
/*
 * One pass of the whole hot path over a batch that is already on the device: Chamfer fwd+bwd (upstream gradient 1)
 * and EMD fwd + sqrt-mean (utils.py:304, weights == 1) + bwd -- three kernels: the auction with its fused epilogue
 * (pcl_emd_fwd_fused), the Chamfer forward and the Chamfer backward.  Chamfer is forked onto a library-owned side stream
 * and runs next to the auction kernel (which leaves 20 of the 148 SMs free); it is joined back into `stream` before the
 * call's work completes.  losses: device float[8] = {chamfer_x, chamfer_y (batch means), chamfer_x, chamfer_y (batch sums),
 * sum sqrt(dist), B*N, EMD mean = [4]/[5], unused} -- a batch-sharded caller all-reduces the contiguous [2..5];
 * grad_pred_chamfer / grad_pred_emd: device (B,N,3) fp32 (d loss / d pred with the batch-mean denominators of THIS batch:
 * B for Chamfer, B*N for EMD).
 */
PCL_API size_t pcl_chamfer_emd_step_scratch_bytes(int B, int N);
PCL_API int pcl_chamfer_emd_step(const void *pred, int dtype1, int64_t bs1, int64_t rs1,
                         const void *target, int dtype2, int64_t bs2, int64_t rs2,
                         int B, int N, float eps, int iters, int chamfer_mode,
                         float *losses, float *grad_pred_chamfer, float *grad_pred_emd,
                         void *scratch, size_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------ host-buffer entry points -------------- */
/*
 * End-to-end calls with HOST buffers (what a non-torch caller binds; also bench.py's e2e leg).
 * Inputs are dense fp32 host arrays (pinned memory recommended), outputs are host arrays; the
 * device staging buffer `dev_scratch` (>= *_host_scratch_bytes) is caller-allocated device memory.
 * The calls enqueue H2D copies, kernels and D2H copies on `stream` and return without
 * synchronising; the caller synchronises the stream before reading the outputs.
 */
PCL_API size_t pcl_loss_host_scratch_bytes(int B, int N);
PCL_API int pcl_chamfer_emd_step_host(const float *pred_host, const float *target_host, int B, int N,
                              float eps, int iters, int chamfer_mode,
                              float *loss_host /* 8: the `losses` vector of pcl_chamfer_emd_step ([0]+[1] = Chamfer loss, [6] = EMD mean sqrt(dist)) */,
                              float *grad_pred_chamfer_host /* nullable B*N*3 */,
                              float *grad_pred_emd_host /* nullable B*N*3 */,
                              void *dev_scratch, size_t dev_scratch_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PCL_B200_H */
