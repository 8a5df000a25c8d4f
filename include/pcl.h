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
/*
 * pcl_chamfer_fwd plus what the rest of pytorch3d's chamfer_distance needs: per-cloud results (weights, batch_reduction None /
 * "sum") and the normal-consistency term (x_normals / y_normals).  pcl_chamfer_fwd is this call with every new pointer NULL.
 *   cloud_sums: nullable DEVICE float[2*B]: cloud_sums[d*B + n] = sum_{i < len} dist (d = 0: x -> y, d = 1: y -> x),
 *     un-normalised, the per-cloud sums loss_xy is made of.
 *   x_nrm / y_nrm: (B,P1,3) / (B,P2,3) normals, strided like the points (pointer, dtype, batch stride, row stride); read only
 *     when normal_sums is not NULL, and then both are required.
 *   normal_sums: nullable DEVICE float[2*B]: normal_sums[d*B + n] = sum_{i < len} (1 - |cos(n_i, n'_{idx[i]})|), the cosine as
 *     F.cosine_similarity(eps=1e-6) forms it; a query whose target cloud is empty adds 1 (its neighbour's normal is taken as 0).
 * It still writes dist / idx and loss_xy, and uses the same workspace (pcl_chamfer_workspace_bytes).  With normal_sums a second
 * kernel runs after the search.
 */
PCL_API int pcl_chamfer_cloud_fwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                    const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len,
                    int B, int P1, int P2, int D, int mode,
                    float *dist_x, int32_t *idx_x, float *dist_y, int32_t *idx_y, float *loss_xy, float *cloud_sums,
                    const void *x_nrm, int x_nrm_dtype, int64_t x_nrm_bs, int64_t x_nrm_rs,
                    const void *y_nrm, int y_nrm_dtype, int64_t y_nrm_bs, int64_t y_nrm_rs, float *normal_sums,
                    void *workspace, size_t workspace_bytes, void *stream);
/*
 * Backward of pcl_chamfer_cloud_fwd.  grad_cloud: DEVICE float[2*B] (may be NULL when B = 0), the upstream gradients of cloud_sums:
 *   grad_x[i] += 2*grad_cloud[n]*(x_i - y[idx_x[i]]);  grad_y[idx_x[i]] -= same;  symmetrically with grad_cloud[B + n].
 * grad_normal: nullable DEVICE float[2*B], the upstream gradients of normal_sums; when given, x_nrm / y_nrm are required and
 * grad_x_nrm (B,P1,3), grad_y_nrm (B,P2,3) receive the normal term's gradient (each query's own normal and, scattered, its
 * neighbour's; 0 where the target cloud is empty).  All gradient outputs are dense fp32 and are overwritten.  No host sync.
 */
PCL_API int pcl_chamfer_cloud_bwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                    const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len,
                    int B, int P1, int P2, int D, const int32_t *idx_x, const int32_t *idx_y,
                    const float *grad_cloud, float *grad_x, float *grad_y,
                    const void *x_nrm, int x_nrm_dtype, int64_t x_nrm_bs, int64_t x_nrm_rs,
                    const void *y_nrm, int y_nrm_dtype, int64_t y_nrm_bs, int64_t y_nrm_rs,
                    const float *grad_normal, float *grad_x_nrm, float *grad_y_nrm, void *stream);

/* ------------------------------------------------------------------ EMD (auction) ------------------------- */
/*
 * Replaces emd.forward (emd.cpp:14-18 -> emd_cuda_forward, emd_cuda.cu:228-282): `iters` rounds of
 * {list unassigned, Bid, GetMax, Assign} then CalcDist, all inside ONE persistent kernel.
 *   xyz1 = prediction (B,N,3) (receives the gradient), xyz2 = target (B,N,3).  Results equal the CPU oracle's bit for bit
 *   for any finite coordinates whose pairwise distances stay below 1e9 (the reference's initial bid value is -1e9);
 *   [0,1]^3 is only the range for which the reference tuned eps.
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
 * start_idx[b] is clamped to [0, N-1].  npoint > N is allowed: once every running minimum is 0, index 0 repeats.
 * N may be up to pcl_fps_max_points() = 262144: one thread-block cluster of 1..16 CTAs per cloud keeps the cloud
 * and its running minima on chip (16384 points per CTA); the cluster size is chosen per launch (pcl_sampling.cu).
 * N above the bound gives PCL_E_UNSUPPORTED.
 */
PCL_API int pcl_fps_max_points(void);
PCL_API int pcl_fps(const void *xyz, int dtype, int64_t bs, int64_t rs, int B, int N, int npoint,
            const int32_t *start_idx /* nullable */, int skip_origin, int32_t *idx_out, void *stream);
/*
 * Farthest point sampling of a ragged batch (pytorch3d's sample_farthest_points(points, lengths, K)).  For cloud b:
 * n_b = lengths[b] clamped to [0, N] (N without lengths), k_b = K[b] clamped to [0, npoint] (npoint without K),
 * s_b = min(n_b, k_b).  idx_out[b, j < s_b] is the FPS sequence over the first n_b points only (the arithmetic, start
 * (start_idx[b] clamped to [0, n_b-1]), skip_origin and tie rule of pcl_fps; points at index >= n_b never influence
 * it); idx_out[b, s_b <= j < npoint] = -1.  Without lengths and K the result equals pcl_fps whenever npoint <= N.
 * lengths and K are int64 DEVICE arrays of B entries, read on the device (no host synchronisation).
 * cluster: 0 = the automatic cluster size; 1, 2, 4, 8 or 16 force one (tests and timing only; a cluster of c CTAs
 * holds at most 16384 * c points, larger N gives PCL_E_UNSUPPORTED).  Other values give PCL_E_ARG.
 */
PCL_API int pcl_fps_ragged(const void *xyz, int dtype, int64_t bs, int64_t rs, const int64_t *lengths /* nullable */,
            int B, int N, const int64_t *K /* nullable */, int npoint, const int32_t *start_idx /* nullable */,
            int skip_origin, int cluster, int32_t *idx_out /* (B, npoint) */, void *stream);
/*
 * Ball query: replaces query_ball_point(radius, nsample, xyz, new_xyz) (models/pointnet2_utils.py:93-113): for every
 * centroid the first `nsample` point indices (ascending) with squared distance <= radius2, padded with the first
 * hit; N when nothing is inside.  group_idx: int32 (B, S, nsample).  radius2 = (float)(radius**2).
 */
PCL_API int pcl_ball_query(const void *xyz, int dtype, int64_t bs, int64_t rs,
                   const void *new_xyz, int ndtype, int64_t nbs, int64_t nrs,
                   int B, int N, int S, float radius2, int nsample, int32_t *group_idx, void *stream);

/* ------------------------------------------------------------------ k nearest neighbours ------------------ */
/*
 * Replaces pytorch3d.ops.knn_points(p1, p2, lengths1, lengths2, norm=2, K) forward and knn_points_backward (third-party
 * code, restated from memory: parity with pytorch3d itself is unpinned).  p1 (B,P1,D) queries, p2 (B,P2,D) targets,
 * 1 <= D <= 8, len1 / len2 nullable int64[B] (entries clamped to [0,P]); 1 <= K <= pcl_knn_max_k() (64); K > P2 is allowed.
 *   dists (B,P1,K) fp32: squared L2 distances, rounded as `mode` says (PCL_CHAMFER_UNFUSED or PCL_CHAMFER_FMA);
 *   idx (B,P1,K) int32.
 * For a query i < len1[n] the result is the K smallest targets j < len2[n] under the key (distance, index), sorted
 * ascending by that key: exact ties go to the lower index, and a NaN distance ranks after +inf (its dists entry is the
 * NaN 0x7fffffff).  Slots k >= min(K, len2[n]) and rows i >= len1[n] are dist 0, idx 0.  The result does not depend on
 * the order in which the kernel visits the targets; for finite inputs K = 1 is bit-identical to dist_x / idx_x of
 * pcl_chamfer_fwd.
 * No workspace.
 */
PCL_API int pcl_knn_max_k(void);
PCL_API int pcl_knn_fwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                int B, int P1, int P2, int D, int K, int mode,
                float *dists, int32_t *idx, void *stream);
/*
 * Backward through dists (idx is not differentiable): for every i < len1[n] and k < min(K, len2[n]), with j = idx[n,i,k],
 *   diff = 2*grad_dists[n,i,k] * (p1[n,i] - p2[n,j]);  grad_p1[n,i] += diff;  grad_p2[n,j] -= diff.
 * grad_dists is a DEVICE (B,P1,K) fp32 array (no host sync).  grad_p1 (B,P1,D) and grad_p2 (B,P2,D) are dense fp32 and are
 * overwritten: grad_p1 is summed over k in ascending order by one thread, grad_p2 is accumulated with fp32 atomics.
 * A slot whose idx is -1 contributes nothing (pcl_knn_fwd never writes -1; pcl_ball_query_fwd pads with it).
 */
PCL_API int pcl_knn_bwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                int B, int P1, int P2, int D, int K, const int32_t *idx,
                const float *grad_dists, float *grad_p1, float *grad_p2, void *stream);

/* ------------------------------------------------------------------ ball query ---------------------------- */
/*
 * Replaces pytorch3d.ops.ball_query(p1, p2, lengths1, lengths2, K, radius) forward and its backward (third-party code,
 * restated from memory [3P-memory]: parity with pytorch3d itself is unpinned).  Inputs as for pcl_knn_fwd: p1 (B,P1,D)
 * queries, p2 (B,P2,D) targets, 1 <= D <= 8, len1 / len2 nullable int64[B] (entries clamped to [0,P]); K >= 1 with no
 * upper bound (K > P2 is allowed); radius2 is the fp32 comparison value.
 *   dists (B,P1,K) fp32, idx (B,P1,K) int32.
 * For a query i < len1[n], the targets j = 0, 1, ..., len2[n]-1 are visited in ascending order and j is kept when
 * d(i,j) < radius2 (strict; a NaN or infinite d is never kept).  The first c <= K kept targets fill slots 0..c-1 with
 * (d, j); slots c..K-1 are dist 0, idx -1.  Rows i >= len1[n] are dist 0, idx -1 (pcl_knn_fwd writes 0 / 0 there).
 * d is the arithmetic of `mode` (PCL_CHAMFER_UNFUSED or PCL_CHAMFER_FMA), so a kept distance is bit-identical to the one
 * pcl_knn_fwd reports for the same pair.  The result does not depend on how the kernel splits the scan.
 * Unlike pcl_ball_query (pointnet2's query_ball_point: xyz only, <=, padding with the first hit) this takes lengths,
 * D <= 8, returns distances and has a backward.  No workspace.
 */
PCL_API int pcl_ball_query_fwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                int B, int P1, int P2, int D, int K, float radius2, int mode,
                float *dists, int32_t *idx, void *stream);
/*
 * Backward through dists: pcl_knn_bwd's formula and kernel (the -1 pads contribute nothing) without its bound on K.
 */
PCL_API int pcl_ball_query_bwd(const void *p1, int dtype1, int64_t bs1, int64_t rs1, const int64_t *len1,
                const void *p2, int dtype2, int64_t bs2, int64_t rs2, const int64_t *len2,
                int B, int P1, int P2, int D, int K, const int32_t *idx,
                const float *grad_dists, float *grad_p1, float *grad_p2, void *stream);

/* ------------------------------------------------------------------ normals and local frames -------------- */
/*
 * Replaces pytorch3d.ops.estimate_pointcloud_local_coord_frames / estimate_pointcloud_normals (0.7.2) forward and their
 * autograd backward (third-party code, restated from memory [3P-memory]: parity with pytorch3d itself is unpinned).
 * p (B,P,3) strided fp32 / fp16 / bf16 points, len nullable int64[B] (entries clamped to [0,P]), 1 <= K <= pcl_knn_max_k(),
 * knn_idx (B,P,K) int32: what pcl_knn_fwd(p, p, len, len, K) wrote (read only; an entry outside [0, n_b) is clamped into it).
 * For cloud b with n_b = len[b] points (P without len) and n_b > K, every point i < n_b with neighbours N_i = knn_idx[b,i,:]:
 *   mu = mean_{j in N_i} p_j,  C = mean_{j in N_i} (p_j - mu)(p_j - mu)^T,  C = V diag(lam) V^T with lam ascending;
 *   curvatures[b,i,:] = lam (B,P,3) fp32;  frames[b,i,:,c] = v_c (B,P,3,3) fp32, column c = eigenvector of lam_c.
 *   disambiguate != 0: v0 and v2 are each negated when 2 * #{j in N_i : v . (p_j - p_i) > 0} < K, and column 1 is v0 x v2.
 * All of it runs in fp64 on the up-cast coordinates (cyclic Jacobi until the off-diagonal is <= 2^-52 ||C||_F) and is
 * rounded to fp32 once.  Rows i >= n_b, and every row of a cloud with n_b <= K, are 0.  Repeated eigenvalues give a finite,
 * orthonormal, deterministic frame.  No atomics: results are bit-reproducible.  No workspace, no host synchronisation.
 */
PCL_API int pcl_frames_fwd(const void *p, int dtype, int64_t bs, int64_t rs, const int64_t *len,
                int B, int P, int K, int disambiguate, const int32_t *knn_idx,
                float *curvatures, float *frames, void *stream);
/*
 * Backward from the saved curvatures and frames and the upstream gradients grad_curvatures (B,P,3) and grad_frames (B,P,3,3)
 * (DEVICE fp32, each nullable: NULL = zero).  With V = frames[b,i], lam = curvatures[b,i], M = V^T grad_frames[b,i] and
 * F_ij = 1 / (lam_j - lam_i) for i != j, 0 on the diagonal (a term whose M_ij is exactly 0 is 0):
 *   Cbar = V (diag(grad_curvatures[b,i]) + F o M) V^T,  grad_p[b,j] += (Cbar + Cbar^T) (p_j - mu) / K  for every j in N_i.
 * The sign flips carry no gradient; column 1 of a disambiguated frame is the unit eigenvector of lam_1 and is treated as one.
 * Equal eigenvalues whose vectors carry gradient give a non-finite gradient, as torch.linalg.eigh's backward does.
 * grad_p (B,P,3) fp32 is overwritten: zero-filled on `stream`, then accumulated with fp32 atomics.
 */
PCL_API int pcl_frames_bwd(const void *p, int dtype, int64_t bs, int64_t rs, const int64_t *len,
                int B, int P, int K, const int32_t *knn_idx, const float *curvatures, const float *frames,
                const float *grad_curvatures, const float *grad_frames, float *grad_p, void *stream);

/* ------------------------------------------------------------------ points alignment and ICP ---------------- */
/*
 * Replaces pytorch3d.ops.corresponding_points_alignment and iterative_closest_point (0.7.2, third-party code restated from
 * memory [3P-memory]: parity with pytorch3d itself is unpinned).  D = 3.  Row-vector convention: apply(X; R, T, s) = s (X R) + T.
 * In fp32, with every step rounded and no contraction:  apply_d = fl(fl(s * fl(fl(fl(x0 R0d) + fl(x1 R1d)) + fl(x2 R2d))) + T_d).
 *
 * Alignment of cloud b, points i < n_b = len[b] (P without len) with weight w_i = weights[b,i] (1 without weights; rows
 * i >= n_b weigh 0, and a point of weight exactly 0 contributes nothing at all):
 *   xm = sum w x / max(sum w, eps),  ym likewise,  a_i = w_i (x_i - xm),  b_i = w_i (y_i - ym)   (pytorch3d's w^2 quirk)
 *   Wt = max(sum w, eps) with weights or len, max(n_b, 1) without either;  M = sum a b^T / Wt,  Xcov = sum |a|^2 / Wt
 *   M = U diag(sig) V^T with det U = det V = +1: one-sided Jacobi SVD of M in fp64, v3 negated if det V < 0,
 *   u1 = M v1 / |M v1|, u2 = M v2 orthogonalised against u1, u3 = u1 x u2; sig_i = u_i^T M v_i (sig3 may be negative).
 *   allow_reflection: u3 and sig3 negated when sig3 < 0.  R = U V^T, tr(ES) = sig1 + sig2 + sig3.
 *   s = tr(ES) / max(Xcov, eps) with estimate_scale, else 1;  T = ym - s (xm R).
 * Rank <= 1 (u2 from the coordinate axis least aligned with u1) and M = 0 (R = I) give deterministic proper rotations.
 * P = 0 (x and y may then be NULL) is M = 0: R = I, T = 0, s = 1 (0 with estimate_scale).
 * Everything runs in fp64 (moments per 32-point block, summed in a fixed order: no atomics, bit-reproducible, independent
 * of the launch); R (B,3,3), T (B,3), s (B) are fp32, rounded once.  pytorch3d's warning on ambiguous rotations is not
 * issued (it needs a host read).
 * record (nullable, B x PCL_ALIGN_RECORD doubles): what the backward reads.  Workspace: pcl_points_alignment_workspace_bytes.
 * Two launches, no host synchronisation.
 */
#define PCL_ALIGN_RECORD 40
PCL_API size_t pcl_points_alignment_workspace_bytes(int B, int P);
PCL_API int pcl_points_alignment_fwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs,
                const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *len, const float *weights,
                int B, int P, int estimate_scale, int allow_reflection, double eps,
                float *R, float *T, float *s, double *record, void *workspace, size_t workspace_bytes, void *stream);
/*
 * Backward from the forward's record and the upstream gradients grad_R (B,3,3), grad_T (B,3), grad_s (B) (DEVICE fp32, each
 * nullable: NULL = zero; grad_s is ignored without estimate_scale).  The polar factor's closed form: with G = U^T Rbar V,
 * Mbar = U H V^T + tr(ES)bar R, H_ij = (G_ij - G_ji) / (sig_i + sig_j), H_ii = 0 (the sign choices are locally constant);
 * then the chain through a_i, b_i, the means and the clamps (an active clamp, value < eps, passes nothing).  Finite for
 * repeated singular values; non-finite only where sig_i + sig_j = 0.  grad_x, grad_y (B,P,3) and grad_weights (B,P,
 * nullable) fp32 are overwritten, one writer per element (rows of weight 0 get 0 for x and y).  One launch.
 */
PCL_API int pcl_points_alignment_bwd(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs,
                const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *len, const float *weights,
                int B, int P, int estimate_scale, double eps, const double *record,
                const float *grad_R, const float *grad_T, const float *grad_s,
                float *grad_x, float *grad_y, float *grad_weights, void *stream);
/*
 * The whole ICP loop in one cooperative launch (plus a memset of the barrier words).  X (B,P1,3), Y (B,P2,3), strided,
 * x_len / y_len nullable.  init_R / init_T / init_s: all NULL (start from X) or all given (DEVICE fp32 (B,3,3), (B,3), (B)).
 * For it = 0 .. max_iterations-1, with Xt the current transformed X (X itself, or apply(X; init), at it = 0):
 *   nn_i = knn K=1 of Xt_i in Y (pcl_knn_fwd's arithmetic for `mode` and its (distance, index) tie rule; Ynn_i = 0 when
 *   y_len[b] = 0);  (R, T, s) = alignment of the ORIGINAL X to Ynn with weights = the 0/1 mask of x_len, eps = 1e-9;
 *   Xt = apply(X; R, T, s);  rmse_b = fl32(sqrt(sum_{i < n_b} |Xt_i - Ynn_i|^2 / max(n_b, 1e-9))), summed in fp64;
 *   rel_b = 1 at it = 0, else fl32((prev_b - rmse_b) / prev_b);  stop when rel_b <= relative_rmse_thr for EVERY b.
 * So a cloud's result depends on its batch, and 0 / 0 (an exact or empty cloud) never passes.
 * P1 = 0 or P2 = 0 is allowed (that input may then be NULL).
 * Outputs, all overwritten: Xt (B,P1,3) fp32, every row (rows past x_len transformed too); R_hist (max_iterations,B,3,3),
 * T_hist (max_iterations,B,3), s_hist and rmse_hist (max_iterations,B): slots past the iterations run are 0;
 * status int32[2] = {iterations run, converged}.  The number of launches does not depend on max_iterations, nothing
 * synchronises with the host and the call can be captured in a CUDA graph.  Workspace: pcl_icp_workspace_bytes (its barrier
 * words are zeroed on `stream` by the call).
 */
PCL_API size_t pcl_icp_workspace_bytes(int B, int P1, int P2, int max_iterations);
PCL_API int pcl_icp(const void *x, int x_dtype, int64_t x_bs, int64_t x_rs, const int64_t *x_len,
                const void *y, int y_dtype, int64_t y_bs, int64_t y_rs, const int64_t *y_len, int B, int P1, int P2,
                const float *init_R, const float *init_T, const float *init_s, int max_iterations, float relative_rmse_thr,
                int estimate_scale, int allow_reflection, int mode, float *Xt, float *R_hist, float *T_hist, float *s_hist,
                float *rmse_hist, int32_t *status, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------ points to volumes -------------------- */
/*
 * Replaces pytorch3d.ops.add_points_features_to_volume_densities_features (0.7.2) forward, unscaled, and its autograd backward
 * (third-party code, restated from memory [3P-memory]: parity with pytorch3d itself is unpinned; tests/volumes_ref.py is
 * the specification).  points (B,P,3) and features (B,P,C), C >= 1, strided fp32 / fp16 / bf16 (pointer, dtype, batch
 * stride, row stride); mask nullable fp32 (B,P), used as a weight m (1 without); grid_sizes nullable DEVICE int64 (B,3)
 * = (D_b, H_b, W_b) (the padded D, H, W without); 0 <= D, H, W <= 2^24.  mode PCL_P2V_TRILINEAR or PCL_P2V_NEAREST.
 * Per axis (x -> W, y -> H, z -> D) with cloud size S, in fp32 with every operation rounded:
 *   t = ((p + 1) * (S - s) - o) * 0.5,   (s, o) = (1, 0) with align_corners, (0, 1) without.
 * Trilinear: f = floor(t), r = t - f; corner f + d (d in {0,1}^3) has weight w = m * (wz * wy) * wx, w_a = d_a ? r_a : 1 - r_a.
 * Nearest: the voxel roundf(t) (half away from zero), weight m.  A vote lands at [b, :, z, y, x] when 0 <= index <
 * min(S_axis, padded axis) on every axis (tested in float: non-finite coordinates and 0 or oversize grid_sizes never index
 * out of bounds) and w != 0; a point with m == 0 is skipped entirely.
 *   volume_densities (B,1,D,H,W) += w;  volume_features (B,C,D,H,W)[c] += w * feature[c]
 * Both volumes are contiguous fp32 and are accumulated into in place with fp32 reductions (red.global.add, subnormals
 * flushed) in no fixed order: not bit-reproducible.  One launch; B = 0, P = 0 or an empty grid launch nothing.
 */
enum { PCL_P2V_TRILINEAR = 0, PCL_P2V_NEAREST = 1 };
PCL_API int pcl_points_to_volumes_fwd(const void *points, int p_dtype, int64_t p_bs, int64_t p_rs,
                const void *features, int f_dtype, int64_t f_bs, int64_t f_rs, const float *mask, const int64_t *grid_sizes,
                int B, int P, int C, int D, int H, int W, int mode, int align_corners,
                float *volume_densities, float *volume_features, void *stream);
/*
 * Backward.  grad_densities (B,1,D,H,W) and grad_features (B,C,D,H,W): contiguous DEVICE fp32, each nullable (NULL = zero).
 * grad_points (B,P,3) and grad_point_features (B,P,C): dense fp32, each nullable (NULL = not computed), overwritten.
 * With the forward's in-bounds corners v_k and weights w_k (zero-weight corners included):
 *   grad_point_features[c] = sum_k w_k grad_features[c, v_k];
 *   grad_points[a] = (S_a - s)/2 * sum_k dw_k/dt_a * (grad_densities[v_k] + sum_c feature[c] grad_features[c, v_k])
 * (trilinear, floor convention dr/dt = 1); 0 in nearest mode.  Points with m == 0 get 0.  One thread per point sums in a
 * fixed order in fp32 with no atomics: bit-reproducible, and a cloud's gradients do not depend on the rest of the batch.
 * One launch, none when both outputs are NULL.
 */
PCL_API int pcl_points_to_volumes_bwd(const void *points, int p_dtype, int64_t p_bs, int64_t p_rs,
                const void *features, int f_dtype, int64_t f_bs, int64_t f_rs, const float *mask, const int64_t *grid_sizes,
                int B, int P, int C, int D, int H, int W, int mode, int align_corners,
                const float *grad_densities, const float *grad_features, float *grad_points, float *grad_point_features,
                void *stream);

/* ------------------------------------------------------------------ rasterize points / compositing -------- */
/*
 * Replaces pytorch3d.renderer.points.rasterize_points (0.7.2) forward and its autograd backward (third-party code, restated
 * from memory [3P-memory]: parity with pytorch3d itself is unpinned; tests/raster_ref.py is the specification).
 * points (B,P,3) strided fp32 / fp16 / bf16 in NDC (+X left, +Y up, +Z away); lengths nullable int64[B] (entries clamped to
 * [0,P]); radius nullable DEVICE fp32 (B,P) contiguous, one radius per point, else radius_scalar for every point.
 * B*P < 2^31, B <= 65535, 1 <= H, W <= 16384, 1 <= K <= pcl_raster_max_k() (150).
 * Pixel (row r, column c) has the fp32 centre xf = ndc(W-1-c, W, H), yf = ndc(H-1-r, H, W), with
 *   ndc(i, S1, S2) = -off + (range*i + off) / S1,  range = S1 > S2 ? (S1*2)/S2 : 2,  off = range/2,
 * every operation rounded (no contraction).  Point i of cloud b hits it when i < lengths[b], x, y, z and r are finite,
 * z >= 0 and d2 = (xf-x)*(xf-x) + (yf-y)*(yf-y) <= r*r (fp32, every operation rounded).  The pixel keeps the K hits of
 * smallest key (z + 0, i) (so -0.0 ties +0.0 and the index decides), ascending:
 *   idx (B,H,W,K) int32 = offset_b + i with offset_b = sum of lengths[0..b-1] (b*P without lengths): pytorch3d's packed index;
 *   zbuf (B,H,W,K) fp32 = z;  dists (B,H,W,K) fp32 = d2;  unused slots -1 in all three.
 * The key is a total order, so the outputs are bit-identical whatever bin_size and max_points_per_bin are, and a cloud's
 * outputs do not depend on the rest of the batch (apart from offset_b).
 * bin_size = 0: one launch; each 16 x TH pixel block scans its whole cloud.  bin_size > 0 (a multiple of 16, else PCL_E_ARG):
 * a memset and two launches; a coarse pass puts every point into each bin_size x bin_size pixel bin its conservative box
 * reaches, at most max_points_per_bin per (cloud, bin) (<= 0: max(10000, P/5), as pytorch3d; never more than P), and the
 * fine pass reads its bin -- or, when the bin overflowed, the whole cloud.  Overflow costs time only: no error, no host read.
 * Workspace: pcl_rasterize_points_workspace_bytes(B, P, H, W, bin_size, max_points_per_bin) (0 for bin_size = 0), else
 * PCL_E_WORKSPACE.  The call can be captured in a CUDA graph.
 */
PCL_API int pcl_raster_max_k(void);
PCL_API size_t pcl_rasterize_points_workspace_bytes(int B, int P, int H, int W, int bin_size, int max_points_per_bin);
PCL_API int pcl_rasterize_points_fwd(const void *points, int dtype, int64_t bs, int64_t rs, const int64_t *lengths,
                const float *radius, float radius_scalar, int B, int P, int H, int W, int K, int bin_size,
                int max_points_per_bin, int32_t *idx, float *zbuf, float *dists, void *workspace, size_t workspace_bytes,
                void *stream);
/*
 * Backward through zbuf and dists (each grad nullable = zero; DEVICE fp32 (B,H,W,K) contiguous): for every slot whose idx is
 * offset_b + i with 0 <= i < lengths[b] (other values, -1 included, are skipped),
 *   grad_points[b,i,2] += grad_zbuf;  grad_points[b,i,0:2] += 2*grad_dists*(p_xy - pixel_xy)
 * with the forward's fp32 pixel centre.  grad_points (B,P,3) dense fp32 is zero-filled (one memset) and accumulated with
 * fp32 red.add by one thread per (pixel, slot): not bit-reproducible.  A memset and at most one launch.
 */
PCL_API int pcl_rasterize_points_bwd(const void *points, int dtype, int64_t bs, int64_t rs, const int64_t *lengths, int B,
                int P, int H, int W, int K, const int32_t *idx, const float *grad_zbuf, const float *grad_dists,
                float *grad_points, void *stream);
/*
 * Replaces pytorch3d.renderer.compositing's alpha_composite / norm_weighted_sum / weighted_sum and their backward
 * [3P-memory].  idx (N,K,H,W) int32 (idx_int64 = 0) or int64 (1), alphas (N,K,H,W) fp32 and features (C, P_total) fp32 are
 * read through their element strides (idx_strides_host / alpha_strides_host: 4 HOST int64, feature_strides_host: 2 HOST
 * int64), so permuted views need no copy.  out (N,C,H,W) contiguous fp32.  A slot with idx < 0 or idx >= P_total
 * contributes nothing.  Sums in fp32 in slot order, every operation rounded:
 *   WEIGHTED:       out = sum_k a_k F[:, idx_k]
 *   NORM_WEIGHTED:  out = sum_k (a_k F[:, idx_k]) / w,  w = max(sum of the valid a_k, 1e-4)
 *   ALPHA:          out = sum_k ((T_k a_k) F[:, idx_k]),  T_0 = 1, T_{k+1} = T_k (1 - a_k) over every slot, valid or not.
 * One launch, one thread per (pixel, 4 channels): bit-reproducible.
 */
enum { PCL_COMPOSITE_ALPHA = 0, PCL_COMPOSITE_NORM_WEIGHTED = 1, PCL_COMPOSITE_WEIGHTED = 2 };
PCL_API int pcl_composite_fwd(int mode, const void *idx, int idx_int64, const int64_t *idx_strides_host, const float *alphas,
                const int64_t *alpha_strides_host, const float *features, const int64_t *feature_strides_host, int N, int K,
                int H, int W, int C, int64_t P_total, float *out, void *stream);
/*
 * Backward: grad_out (N,C,H,W) contiguous fp32.  grad_alphas (N,K,H,W) contiguous fp32, nullable, written by one thread per
 * pixel with no atomics (the alpha derivative is formed from products of (1 - a_t), never by dividing by 1 - a_k, so a = 1
 * stays finite); grad_features (C, P_total) contiguous fp32, nullable, zero-filled (one memset) and accumulated with fp32
 * red.add.  At most a memset and one launch.
 */
PCL_API int pcl_composite_bwd(int mode, const void *idx, int idx_int64, const int64_t *idx_strides_host, const float *alphas,
                const int64_t *alpha_strides_host, const float *features, const int64_t *feature_strides_host, int N, int K,
                int H, int W, int C, int64_t P_total, const float *grad_out, float *grad_alphas, float *grad_features,
                void *stream);

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
