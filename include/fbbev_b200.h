/*
 * fbbev_b200.h -- C ABI of libfbbev_b200.so: the B200 (sm_100a) implementation
 * of the FB-BEV / FB-OCC forward-backward view-transformation hot path.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the parameter name ends in `_host`;
 *   - the caller owns every buffer including workspaces; nothing is allocated,
 *     no host<->device synchronisation happens inside a call, and all work is
 *     enqueued on `stream` (a cudaStream_t; NULL = legacy default stream);
 *   - return value: 0 on success, a negative FBBEV_ERR_* for argument errors,
 *     or a positive cudaError_t raised while enqueuing.  Nothing throws.
 *   - re-entrant per stream; no global mutable state.
 *
 * Each entry point names the reference interface it replaces (paths relative
 * to the NVlabs/FB-BEV checkout).  INTEGRATION.md shows the reference-side
 * binding for each.
 */
#ifndef FBBEV_B200_H_
#define FBBEV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FBBEV_OK 0
#define FBBEV_ERR_INVALID_ARGUMENT (-1)
#define FBBEV_ERR_WORKSPACE_TOO_SMALL (-2)
#define FBBEV_ERR_UNSUPPORTED (-3)

#define FBBEV_ABI_VERSION 4

typedef void* fbbev_stream_t; /* cudaStream_t */

int fbbev_abi_version(void);
/* Diagnostics: cumulative number of kernel launches issued by this library. */
long long fbbev_debug_launch_count(void);
/* Static string for a return code of any entry point. */
const char* fbbev_error_string(int code);

/* =====================================================================
 * F -- lift-splat voxel pooling (bev_pool_v2)
 * ===================================================================== */

/*
 * Drop-in for `bev_pool_v2_ext.bev_pool_v2_forward`
 *   mmdet3d/ops/bev_pool_v2/src/bev_pool.cpp:28-55 (launcher
 *   bev_pool_cuda.cu:120-128, kernel :18-45).
 * depth (B,N,D,H,W) fp32; feat (B,N,H,W,C) fp32; index arrays int32;
 * out (B,Z,Y,X,C) fp32, ZERO-FILLED BY THE CALLER as in bev_pool.py:25.
 * Semantics identical to the reference for arbitrary interval lists: one
 * plain store of the interval sum to voxel ranks_bev[interval_starts[i]].
 * Differences: 64-bit offsets (the reference overflows int32 when
 * B*Z*Y*X*C >= 2^31) and the caller's stream instead of the legacy stream.
 */
int fbbev_bev_pool_v2_fwd(const float* depth, const float* feat,
                          const int32_t* ranks_depth,
                          const int32_t* ranks_feat, const int32_t* ranks_bev,
                          const int32_t* interval_starts,
                          const int32_t* interval_lengths, int32_t n_intervals,
                          int32_t c, float* out, fbbev_stream_t stream);

/*
 * Fused replacement for the whole reference op
 *   `bev_pool_v2()` = QuickCumsumCuda.forward + permute(0,4,1,2,3).contiguous()
 *   mmdet3d/ops/bev_pool_v2/bev_pool.py:15-39, 84-90.
 * Writes EVERY element of out exactly once, directly in the op's final
 * (B,C,Z,Y,X) layout: no caller-side memset, no transpose pass.
 *
 * Precondition (what voxel_pooling_prepare_v2 always produces,
 * view_transformer.py:590-602): intervals are listed in non-decreasing order
 * of their voxel rank ranks_bev[interval_starts[i]], one interval per voxel.
 * Out-of-range ranks are ignored (memory-safe).
 *
 * n_intervals_dev: optional device int32 holding the live interval count
 *   (<= n_intervals_max); NULL means n_intervals_max is the count.  This lets
 *   the prepare -> pool chain run without a host sync / under CUDA graphs.
 * n_points = number of entries in ranks_bev / ranks_depth / ranks_feat (an
 *   upper bound of the kept points when the buffers are over-allocated).
 * n_voxels_per_sample = Z*Y*X.  Requires B*Z*Y*X < 2^31 (int32 ranks).
 * workspace: >= fbbev_bev_pool_v2_dense_workspace_bytes(...) bytes.
 * Scheduling (the one exception to "all work goes to `stream`"): the zero
 * stream of the EMPTY voxel tiles depends on the plan only and is enqueued on a
 * library-owned side stream (one per host thread, created on first use) that
 * forks from and joins back into `stream` with events inside the call, so it
 * runs beside the interval sums; the caller sees ordinary stream semantics (the
 * call is complete on `stream` when everything is).  Warm up once before
 * capturing a CUDA graph.  FBBEV_POOL_OVERLAP=0 in the environment keeps
 * everything on `stream`.
 */
size_t fbbev_bev_pool_v2_dense_workspace_bytes(int32_t batch,
                                               int64_t n_voxels_per_sample,
                                               int32_t n_intervals_max,
                                               int32_t n_points, int32_t c);
int fbbev_bev_pool_v2_fwd_dense(
    const float* depth, const float* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* interval_lengths,
    int32_t n_intervals_max, const int32_t* n_intervals_dev, int32_t n_points,
    int32_t c, int32_t batch, int64_t n_voxels_per_sample, float* out,
    void* workspace, size_t workspace_bytes, fbbev_stream_t stream);

/*
 * The two halves of fbbev_bev_pool_v2_fwd_dense, for callers that reuse an
 * index (static camera rig, `accelerate=True`, view_transformer.py:261-283):
 * `plan` builds the tile table for a given (index, C) once; `_planned` then
 * runs only the pooling kernels (the workspace doubles as their scratch, so it
 * is written by `_planned` as well; one workspace per concurrent stream).
 */
int fbbev_bev_pool_v2_plan(const int32_t* ranks_bev,
                           const int32_t* interval_starts,
                           const int32_t* interval_lengths,
                           int32_t n_intervals_max,
                           const int32_t* n_intervals_dev, int32_t n_points,
                           int32_t c, int32_t batch,
                           int64_t n_voxels_per_sample, void* workspace,
                           size_t workspace_bytes, fbbev_stream_t stream);
int fbbev_bev_pool_v2_fwd_dense_planned(
    const float* depth, const float* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* interval_lengths,
    int32_t n_intervals_max, int32_t n_points, int32_t c, int32_t batch,
    int64_t n_voxels_per_sample, float* out, void* plan, size_t plan_bytes,
    fbbev_stream_t stream);

/*
 * The dense op in stages, for FBOCC's glue around the two projections
 * (mmdet3d/models/fbbev/detectors/fbocc.py:339, 357-366):
 *     bev_feat = forward_projection(...)                       # dense volume
 *     refined  = backward_projection(..., lss_bev=bev_feat.mean(-1), ...)
 *     bev_feat = refined[..., None] + bev_feat                 # re-add
 * reads the 204.8 MB volume twice and writes it twice.  After
 * fbbev_bev_pool_v2_plan on the same workspace:
 *   _sums_planned   runs the interval-sum stage only (V / X rows in the plan);
 *   _zmean_planned  writes bev_feat.mean(-1) as a TOKEN-major map
 *                   lss_tokens (B, Y*X, C) from the interval sums (the map is
 *                   zero-filled here; red.global.add of <= Z terms per element);
 *                   yx = Y*X;
 *   _write_planned  materialises the (B,C,Z,Y,X) volume, adding `add` (may be
 *                   NULL; (B, C, Y*X), e.g. the refined BEV) to every Z slice
 *                   on the way out -- the volume is written exactly once.
 * Requirements as for the dense op plus C % 4 == 0, (Z*Y*X) % 4 == 0, yx % 4 == 0;
 * FBBEV_ERR_UNSUPPORTED otherwise (use the one-shot op and eager glue).
 */
int fbbev_bev_pool_v2_sums_planned(
    const float* depth, const float* feat, const int32_t* ranks_depth,
    const int32_t* ranks_feat, const int32_t* ranks_bev,
    const int32_t* interval_starts, const int32_t* interval_lengths,
    int32_t n_intervals_max, int32_t n_points, int32_t c, int32_t batch,
    int64_t n_voxels_per_sample, void* plan, size_t plan_bytes,
    fbbev_stream_t stream);
int fbbev_bev_pool_v2_zmean_planned(
    const int32_t* interval_starts, const int32_t* interval_lengths,
    int32_t n_intervals_max, int32_t n_points, int32_t c, int32_t batch,
    int64_t n_voxels_per_sample, int32_t yx, float* lss_tokens, void* plan,
    size_t plan_bytes, fbbev_stream_t stream);
int fbbev_bev_pool_v2_write_planned(
    const int32_t* interval_starts, const int32_t* interval_lengths,
    int32_t n_intervals_max, int32_t n_points, int32_t c, int32_t batch,
    int64_t n_voxels_per_sample, int32_t yx, const float* add, float* out,
    void* plan, size_t plan_bytes, fbbev_stream_t stream);

/*
 * Drop-in for `bev_pool_v2_ext.bev_pool_v2_backward`
 *   mmdet3d/ops/bev_pool_v2/src/bev_pool.cpp:72-102 (kernel
 *   bev_pool_cuda.cu:64-118).  Intervals are runs of equal ranks_feat
 *   (bev_pool.py:45-55).  out_grad (B,Z,Y,X,C); depth_grad / feat_grad
 *   zero-filled by the caller (bev_pool.py:65-66).
 */
int fbbev_bev_pool_v2_bwd(const float* out_grad, const float* depth,
                          const float* feat, const int32_t* ranks_depth,
                          const int32_t* ranks_feat, const int32_t* ranks_bev,
                          const int32_t* interval_starts,
                          const int32_t* interval_lengths, int32_t n_intervals,
                          int32_t c, float* depth_grad, float* feat_grad,
                          fbbev_stream_t stream);

/*
 * Same contract as fbbev_bev_pool_v2_bwd, but out_grad is (B,C,Z,Y,X) -- the
 * layout of the tensor `bev_pool_v2()` returns (bev_pool.py:89), i.e. the
 * gradient as autograd delivers it -- so the full-volume transpose copy the
 * reference performs first (`out_grad.contiguous()`, bev_pool.py:67) is skipped.
 */
int fbbev_bev_pool_v2_bwd_bczyx(
    const float* out_grad, const float* depth, const float* feat,
    const int32_t* ranks_depth, const int32_t* ranks_feat,
    const int32_t* ranks_bev, const int32_t* interval_starts,
    const int32_t* interval_lengths, int32_t n_intervals, int32_t c,
    int64_t n_voxels_per_sample, float* depth_grad, float* feat_grad,
    fbbev_stream_t stream);

/*
 * Device implementation of `voxel_pooling_prepare_v2`
 *   mmdet3d/models/fbbev/view_transformation/forward_projection/
 *   view_transformer.py:547-605  (integer path, bit-exact).
 * coor (B,N,D,H,W,3) fp32 ego-frame points from get_lidar_coor (:458-498).
 * lo/iv/gs: grid lower bound, interval and FLOAT32 grid size (:384-387).
 * Outputs (each sized for B*N*D*H*W entries): ranks_bev / ranks_depth /
 * ranks_feat sorted by voxel rank, ascending point index inside a voxel
 * (a stable sort; the reference's argsort order inside a voxel is
 * unspecified), interval_starts / interval_lengths; counts[0] = n_kept,
 * counts[1] = n_intervals (device int32[2]).
 * Voxel rank is computed in exact integer arithmetic; the reference computes
 * it in float32 (:586-589), which is identical while B*Z*Y*X < 2^24.
 * Requires B*Z*Y*X < 2^31 and B*N*D*H*W < 2^31.
 */
size_t fbbev_voxel_prepare_workspace_bytes(int64_t n_points,
                                           int64_t n_voxels_total);
int fbbev_voxel_prepare(const float* coor, int32_t B, int32_t N, int32_t D,
                        int32_t H, int32_t W, const float* lo_host,
                        const float* iv_host, const float* gs_host,
                        int32_t* ranks_bev, int32_t* ranks_depth,
                        int32_t* ranks_feat, int32_t* interval_starts,
                        int32_t* interval_lengths, int32_t* counts,
                        void* workspace, size_t workspace_bytes, int32_t pool_c,
                        void* pool_plan, size_t pool_plan_bytes,
                        fbbev_stream_t stream);

/*
 * voxel_pooling_prepare_v2 with get_lidar_coor fused in
 *   (view_transformer.py:458-498 + 547-605): the (B,N,D,H,W,3) coordinate tensor
 *   is never materialised.  frustum_u [W], frustum_v [H], frustum_d [D] are the
 *   three axes of the frustum template (create_frustum, :389-411);
 *   inv_post_rots = inverse(post_rots) (B*N,3,3); cam2ego = rots @ inverse(K)
 *   (B*N,3,3) -- the two tiny products the reference also forms before touching
 *   the points (:483-491); post_trans, trans (B*N,3); bda (B,3,3).
 * The per-point chain is evaluated in fp32 in the rounding order the reference's
 * eager chain has on this device (torch broadcast matmul -> cuBLAS): per output
 * row fma(m1, x1, m0*x0) + m2*x2, or -- FBBEV_ORDER_SEQ_* bit set -- the
 * sequential chain fma(m2, x2, fma(m1, x1, m0*x0)) cuBLAS uses when ONE
 * column-major matrix (the layout torch.inverse returns) is broadcast over the
 * whole batch.  order_flags: bit 0 inv_post_rots, bit 1 cam2ego, bit 2 bda.
 * The index is bit-identical to fbbev_voxel_prepare on get_lidar_coor's output.
 *
 * pool_plan (both prepare entry points; may be NULL): a dense-pooling workspace
 * of fbbev_bev_pool_v2_dense_workspace_bytes(B, Z*Y*X, min(n_points, B*Z*Y*X),
 * n_points, pool_c) bytes.  When given, the scan over the voxel histogram also
 * fills the pooling plan (what fbbev_bev_pool_v2_plan computes in a launch of
 * its own), so the index can go straight to fbbev_bev_pool_v2_fwd_dense_planned
 * / _sums_planned with the same workspace and n_intervals_max = min(n_points,
 * B*Z*Y*X).  Needs fbbev_voxel_prepare_can_plan(pool_c, Z*Y*X) != 0, else
 * FBBEV_ERR_UNSUPPORTED.
 */
int fbbev_voxel_prepare_can_plan(int32_t pool_c, int64_t n_voxels_per_sample);
#define FBBEV_ORDER_SEQ_A 1
#define FBBEV_ORDER_SEQ_B 2
#define FBBEV_ORDER_SEQ_C 4
int fbbev_voxel_prepare_cams(
    const float* frustum_u, const float* frustum_v, const float* frustum_d,
    const float* inv_post_rots, const float* post_trans, const float* cam2ego,
    const float* trans, const float* bda, int32_t order_flags, int32_t B,
    int32_t N, int32_t D, int32_t H, int32_t W, const float* lo_host,
    const float* iv_host, const float* gs_host, int32_t* ranks_bev,
    int32_t* ranks_depth, int32_t* ranks_feat, int32_t* interval_starts,
    int32_t* interval_lengths, int32_t* counts, void* workspace,
    size_t workspace_bytes, int32_t pool_c, void* pool_plan,
    size_t pool_plan_bytes, fbbev_stream_t stream);

/*
 * The same two index builders with the depth-threshold sparsification of the
 * BEVDet-lineage transformer
 *   mmdet3d/models/necks/view_transformer.py:520-578 (LSSViewTransformer2.
 *   voxel_pooling_prepare_v2: `kept = kept & (depth.view(-1) > 0.01)`, :556-557)
 *   and its cached-index form (:645-678: the geometric index filtered by
 *   `(depth.view(-1) > 0.01)[self.kept]` on every forward).
 * depth_prob (B,N,D,H,W) fp32 -- the tensor the pooling op will read, indexed
 * by the point index (ranks_depth == arange) -- may be NULL (no threshold);
 * a point is kept when depth_prob[p] > depth_thresh (strict, as the reference).
 * Everything else as fbbev_voxel_prepare / fbbev_voxel_prepare_cams.
 */
int fbbev_voxel_prepare_sparse(
    const float* coor, const float* depth_prob, float depth_thresh, int32_t B,
    int32_t N, int32_t D, int32_t H, int32_t W, const float* lo_host,
    const float* iv_host, const float* gs_host, int32_t* ranks_bev,
    int32_t* ranks_depth, int32_t* ranks_feat, int32_t* interval_starts,
    int32_t* interval_lengths, int32_t* counts, void* workspace,
    size_t workspace_bytes, int32_t pool_c, void* pool_plan,
    size_t pool_plan_bytes, fbbev_stream_t stream);
int fbbev_voxel_prepare_cams_sparse(
    const float* frustum_u, const float* frustum_v, const float* frustum_d,
    const float* inv_post_rots, const float* post_trans, const float* cam2ego,
    const float* trans, const float* bda, int32_t order_flags,
    const float* depth_prob, float depth_thresh, int32_t B, int32_t N,
    int32_t D, int32_t H, int32_t W, const float* lo_host,
    const float* iv_host, const float* gs_host, int32_t* ranks_bev,
    int32_t* ranks_depth, int32_t* ranks_feat, int32_t* interval_starts,
    int32_t* interval_lengths, int32_t* counts, void* workspace,
    size_t workspace_bytes, int32_t pool_c, void* pool_plan,
    size_t pool_plan_bytes, fbbev_stream_t stream);

/*
 * The tail of the depth net as the PRODUCER of the pooling op's inputs
 * (SURVEY.md section 8 f4 / f3):
 *   CM_DepthNet.forward   mmdet3d/models/fbbev/modules/depth_net.py:359-363
 *       depth = depth.softmax(dim=1); context.view(B, N, C, H, W)
 *   LSSViewTransformer / LSSViewTransformer2 / LSSViewTransformerBEVDepth.forward
 *       mmdet3d/models/necks/view_transformer.py:313-321, 710-718, 1094-1096
 *       depth_digit = x[:, :D]; tran_feat = x[:, D:D+C]; depth = softmax(dim=1)
 *   + the `feat.permute(0,1,3,4,2)` / `feat.contiguous()` transposing copy inside
 *     the pooling op (view_transformer.py:530, bev_pool.py:19).
 * depth_logits: image n, bin k, pixel p at [n * logits_image_stride + k*hw + p]
 * (NCHW with its own image stride, so a channel slice of a wider tensor works);
 * context likewise with c channels.  Either may be NULL (that half is skipped).
 * depth_out (bn, d, hw) = softmax over the d bins (max / sum of expf / divide,
 * as torch); feat_out (bn, hw, c) = context transposed to pixel-major -- the
 * (B,N,H,W,C) layout `bev_pool_v2` reads.  One launch.
 */
int fbbev_lift_tail_fwd(const float* depth_logits, int64_t logits_image_stride,
                        const float* context, int64_t context_image_stride,
                        int32_t bn, int32_t d, int32_t c, int32_t hw,
                        float* depth_out, float* feat_out,
                        fbbev_stream_t stream);

/* =====================================================================
 * B -- BEV -> image depth-aware spatial cross-attention (MSDeformAttn)
 * ===================================================================== */

/*
 * One-kernel `bevformer_encoder.point_sampling`
 *   .../backward_projection/bevformer_utils/bevformer_encoder.py:92-120.
 * X [nX], Y [nY], Z [nZ]: voxel-centre coordinates per axis (get_reference_points
 * '3d', :64-70); inv_bda = inverse(bda) (B,3,3); ego2cam = inverse(rots @
 * inverse(K)) (B*N,3,3); trans, post_trans (B*N,3); post_rots (B*N,3,3);
 * (w_in, h_in) = data_config input_size; eps = 1e-5 and one_minus_eps =
 * (float)(1.0 - 1e-5), the two scalars of the visibility test (:113-117).
 * order_flags as for fbbev_voxel_prepare_cams: bit 0 inv_bda, bit 1 ego2cam,
 * bit 2 post_rots.  The image-plane normalisation multiplies by (1 / w_in),
 * (1 / h_in) as torch's CUDA `tensor /= python_scalar` does.
 * Outputs in the reference's layouts: ref_cam (N,B,nY*nX,nZ,2), depth
 * (N,B,nY*nX,nZ), mask (N,B,nY*nX,nZ) uint8; bit-identical to the eager chain.
 */
int fbbev_point_sampling(
    const float* X, const float* Y, const float* Z, int32_t nX, int32_t nY,
    int32_t nZ, const float* inv_bda, const float* trans, const float* ego2cam,
    const float* post_rots, const float* post_trans, int32_t order_flags,
    int32_t B, int32_t N, float w_in, float h_in, float eps,
    float one_minus_eps, float* ref_cam, float* depth, uint8_t* mask,
    fbbev_stream_t stream);

/*
 * BEV queries of `BackwardProjection.forward`
 *   .../backward_projection/backward_projection.py:93-97:
 *   out[b, q, :] = embedding[q, :] + lss_bev[b, :, q]   (lss_bev may be NULL)
 * embedding (nq, E) = bev_embedding.weight; lss_bev (bs, E, bev_h*bev_w) = the
 * lift-splat BEV, channel-major; out (bs, nq, E) contiguous (the reference's
 * (nq, bs, E) tensor is its permuted view).  One pass, one fp32 add per element.
 */
int fbbev_bev_query_init(const float* embedding, const float* lss_bev,
                         int32_t bs, int32_t nq, int32_t E, float* out,
                         fbbev_stream_t stream);

/*
 * out[b, e, q] = tokens[b, q, e]: the last line of `BackwardProjection.forward`
 *   (backward_projection.py:131-133: bev.permute(0, 2, 1).view(bs, -1, bev_h,
 *   bev_w).contiguous()).  tokens (bs, nq, E), out (bs, E, nq), both dense fp32,
 *   16-byte aligned; nq % 4 == 0 and E % 4 == 0, else FBBEV_ERR_UNSUPPORTED.
 */
int fbbev_tokens_to_map(const float* tokens, int32_t bs, int32_t nq, int32_t E,
                        float* out, fbbev_stream_t stream);

/*
 * Drop-in for `ext_module.ms_deform_attn_forward` (mmcv-full 1.5.2 `_ext`)
 *   call site: .../backward_projection/bevformer_utils/
 *   multi_scale_deformable_attn_function.py:127-133.
 * value (bs, n_value, heads, ch) fp32; spatial_shapes (levels,2) and
 * level_start (levels) are DEVICE int64 as in the reference
 * (bevformer.py:108-111); loc (bs,nq,heads,levels,points,2) as (x,y) in
 * [0,1]; attw (bs,nq,heads,levels,points); out (bs,nq,heads*ch).
 * No im2col_step restriction.
 */
int fbbev_msda_fwd(const float* value, const int64_t* spatial_shapes,
                   const int64_t* level_start, const float* loc,
                   const float* attw, int32_t bs, int32_t n_value,
                   int32_t heads, int32_t ch, int32_t levels, int32_t nq,
                   int32_t points, float* out, fbbev_stream_t stream);

/*
 * Drop-in for `ext_module.ms_deform_attn_backward`
 *   call site: multi_scale_deformable_attn_function.py:159-169.
 * grad_value / grad_loc / grad_attw zero-filled by the caller (:155-157).
 */
int fbbev_msda_bwd(const float* value, const int64_t* spatial_shapes,
                   const int64_t* level_start, const float* loc,
                   const float* attw, const float* grad_out, int32_t bs,
                   int32_t n_value, int32_t heads, int32_t ch, int32_t levels,
                   int32_t nq, int32_t points, float* grad_value,
                   float* grad_loc, float* grad_attw, fbbev_stream_t stream);

/*
 * Fused core of mmcv `MultiScaleDeformableAttention.forward` (the encoder
 * layer's self_attn, fbocc-r50 config :176-180): softmax over levels*points,
 * sampling_locations = ref + offsets / (W_l, H_l), bilinear sampling and
 * weighted sum in one kernel -- `loc` / normalised `attw` never touch HBM.
 * ref (bs,nq,levels,2); offsets (bs,nq,heads,levels,points,2) = raw output of
 * the sampling_offsets Linear; logits (bs,nq,heads,levels,points) = raw output
 * of the attention_weights Linear; out (bs,nq,heads*ch).
 * patch_w: 0, or -- for self-attention over the map itself (levels == 1, nq ==
 * n_value, 8 heads) -- the map width W: query q = y * W + x then sits on value
 * pixel (y, x) and blocks own 8x8 query squares (L1-resident footprint) instead
 * of runs of a row.  Results do not depend on it.
 */
int fbbev_msda_fused_fwd(const float* value, const int64_t* spatial_shapes,
                         const int64_t* level_start, const float* ref,
                         const float* offsets, const float* logits, int32_t bs,
                         int32_t n_value, int32_t heads, int32_t ch,
                         int32_t levels, int32_t nq, int32_t points,
                         int32_t patch_w, float* out, fbbev_stream_t stream);

/*
 * Fused depth-aware spatial cross-attention: everything between the three
 * input Linears and `output_proj` of
 *   DA_SpatialCrossAttention.forward   spatial_cross_attention_depth.py:86-223
 *   DA_MSDeformableAttention.forward   spatial_cross_attention_depth.py:465-601
 * i.e. per-camera query selection (:156-169), rebatch (:173-186), depth bin
 * one-hot (:196-199), softmax (:540), sampling locations (:554-570), the depth
 * look-up MSDA launch (:584-591), depth re-weighting (:592), the main MSDA
 * launch (:593-595), scatter-add over cameras (:208-211) and the division by
 * the per-query camera count (:213-216).
 *
 * value      (bs*n_cams, n_value, heads, ch)  value_proj(feat), camera-major
 *            inside a sample (row = b*n_cams + cam), as at :188-191
 * depth_prob (bs*n_cams, H0*W0, DC)  pred_img_depth flattened as at :131-133
 * ref_cam    (n_cams, bs, nq, Z, 2)  reference_points_cam (bevformer_encoder.py:117)
 * ref_depth  (n_cams, bs, nq, Z)     bev_query_depth (:120)
 * mask       (n_cams, bs, nq, Z) uint8   per_cam_mask_list (:118)
 * offsets    (bs, nq, heads, levels, points, 2)  raw sampling_offsets(query)
 * logits     (bs, nq, heads, levels, points)     raw attention_weights(query)
 *   (both Linears act row-wise, so evaluating them once per BEV query equals
 *    the reference's evaluation on the re-batched copies)
 * points = num_points (all Z anchors), Z = num_Z_anchors, point index
 *   = p*Z + z (:563-570, :590).
 * dbound_host = (d_min, d_max, d_step) (:196); DC = depth bins.
 * out        (bs, nq, heads*ch) = slots / clamp(count, 1), the tensor the
 *            reference feeds to output_proj (:219).
 * bev_mask (:156-159): pass the output of fbbev_bev_mask_fold as `mask`.
 * Mask bytes: 0 = not visible; bit 0 set = visible and counted in the camera
 * mean; 2 = visible but not counted (the reference's empty-camera rule).
 *
 * workspace (fbbev_da_sca_workspace_bytes(bs, n_cams) bytes, may be NULL):
 * with it, and when one camera's value map fits in shared memory (n_value *
 * heads * ch * 4 <= ~220 KB; 8 heads x 10 channels, 1 level, 8 points, 4
 * anchors -- the FB-OCC head), the camera-resident kernel of da_sca_smem.cu
 * runs: a CTA stages its camera's map with TMA bulk copies and serves the
 * queries that camera sees from shared memory; contributions of several
 * cameras to one query are combined with red.global.add on the zero-filled
 * output (the order of these <= n_cams additions is not fixed).  Without a
 * workspace, or for other shapes, the one-thread-per-(query, head) kernel
 * gathers from global memory.
 */
size_t fbbev_da_sca_workspace_bytes(int32_t bs, int32_t n_cams);
int fbbev_da_sca_fwd(const float* value, const float* depth_prob,
                     const float* ref_cam, const float* ref_depth,
                     const uint8_t* mask, const float* offsets,
                     const float* logits, const int64_t* spatial_shapes,
                     const int64_t* level_start, const float* dbound_host,
                     int32_t bs, int32_t n_cams, int32_t nq, int32_t n_value,
                     int32_t heads, int32_t ch, int32_t levels, int32_t points,
                     int32_t Z, int32_t DC, float* out, void* workspace,
                     size_t workspace_bytes, int32_t prologue_done,
                     fbbev_stream_t stream);
/* The mask-only part of fbbev_da_sca_fwd's camera-resident path (per-camera
 * visible-query counts into `workspace`, zero-fill of `out`), callable ahead of
 * time -- e.g. on the stream that produced the mask, beside the self-attention.
 * Pass the same `out` / `workspace` to fbbev_da_sca_fwd with prologue_done = 1.
 * FBBEV_ERR_UNSUPPORTED when the shape takes the global-memory kernel. */
int fbbev_da_sca_prologue(const uint8_t* mask, int32_t bs, int32_t n_cams,
                          int32_t nq, int32_t n_value, int32_t heads,
                          int32_t ch, int32_t levels, int32_t points, int32_t Z,
                          float* out, void* workspace, size_t workspace_bytes,
                          fbbev_stream_t stream);

/*
 * `per_cam_mask_list & bev_mask[None, :, :, None]` with the reference's
 * empty-camera rule (spatial_cross_attention_depth.py:156-169, 213-214) as a
 * device-side pass, so a bev_mask no longer forces the per-camera nonzero() /
 * re-batching loops (6*bs host synchronisations per layer in the reference).
 * mask (n_cams, bs, nq, Z) uint8/bool; bev_mask (bs, nq) uint8/bool; mask_out
 * (n_cams, bs, nq, Z) uint8 in the encoding fbbev_da_sca_fwd documents:
 * 1 where mask & bev_mask; for a (sample, camera) pair that sees no query under
 * the masked list, the anchors of the FIRST query it sees at all get 2.
 */
size_t fbbev_bev_mask_fold_workspace_bytes(int32_t bs, int32_t n_cams);
int fbbev_bev_mask_fold(const uint8_t* mask, const uint8_t* bev_mask,
                        int32_t bs, int32_t n_cams, int32_t nq, int32_t Z,
                        uint8_t* mask_out, void* workspace,
                        size_t workspace_bytes, fbbev_stream_t stream);

/* ---- row-wise Linear (+ bias, ReLU, residual, LayerNorm) on tcgen05 ---------
 * Replaces the nn.Linear / LayerNorm / residual chain of the reference's
 * encoder layer for the backward projection: sampling_offsets,
 * attention_weights, value_proj, output_proj
 * (spatial_cross_attention_depth.py:420-427, 226-233; mmcv
 * MultiScaleDeformableAttention), mmcv FFN and the `norm` entries of
 * operation_order (bevformer_encoder.py:251-377), which the reference runs as
 * cuBLAS fp32 GEMMs plus separate elementwise kernels.
 *
 *   y = LN( act( x . W^T + bias ) + residual )
 *
 * x (m, k) fp32 with row stride ldx floats, W (n, k) as in nn.Linear.weight,
 * y (m, n) with row stride ldy (a column block of a wider output is allowed);
 * bias / residual (m, n; row stride ldr) / ln_weight+ln_bias (n) are optional
 * (NULL), relu != 0
 * applies ReLU before the residual.  fp32 in and out; products are formed as
 * 3xTF32 on the tensor cores (error ~1e-6 relative, inside the 1e-4 bar; plain
 * TF32 is not).  Weights are packed once (hi / lo split in the shared-memory
 * layout of the kernel) with fbbev_linear_pack into fbbev_linear_packed_bytes
 * bytes; k % 4 == 0, n % 4 == 0, n <= 192 (split wider layers over n), n <= 80
 * with the LayerNorm epilogue (whole rows stay in shared memory),
 * 16-byte aligned pointers; otherwise FBBEV_ERR_UNSUPPORTED /
 * FBBEV_ERR_INVALID_ARGUMENT.
 */
size_t fbbev_linear_packed_bytes(int32_t n, int32_t k);
int fbbev_linear_pack(const float* weight, int32_t n, int32_t k, float* packed,
                      fbbev_stream_t stream);
int fbbev_linear_fwd(const float* x, int64_t ldx, const float* packed,
                     const float* bias, const float* residual, int64_t ldr,
                     const float* ln_weight, const float* ln_bias, int64_t m,
                     int32_t k, int32_t n, int32_t relu, float ln_eps, float* y,
                     int64_t ldy, fbbev_stream_t stream);

/* Two Linears that read the same x as ONE launch: `packed` / `bias` hold the
 * row-concatenated weight (n = n0 + n1 rows, n <= 192) and bias; output columns
 * [0, n_split) go to y0 (row stride ldy0), [n_split, n) to y1 (ldy1), each dense.
 * This is sampling_offsets + attention_weights of both attention modules
 * (spatial_cross_attention_depth.py:420-424, 533-540): they act on the same
 * query and feed one sampling kernel.  No residual / LayerNorm here.
 * x_add (may be NULL; row stride ldx_add): the GEMM input is x + x_add, formed
 * in the loader with one fp32 add per element -- `query = query + query_pos`
 * of both attention modules (spatial_cross_attention_depth.py:117-118, mmcv
 * MultiScaleDeformableAttention.forward) without a separate pass. */
int fbbev_linear_fwd_split(const float* x, int64_t ldx, const float* x_add,
                           int64_t ldx_add, const float* packed,
                           const float* bias, int64_t m, int32_t k, int32_t n,
                           int32_t n_split, int32_t relu, float* y0,
                           int64_t ldy0, float* y1, int64_t ldy1,
                           fbbev_stream_t stream);

/*
 * The encoder layer's FFN and the LayerNorm after it as ONE kernel:
 *     y = LN( residual + W2 . relu(W1 . x + b1) + b2 )
 * mmcv `FFN` (two Linears, ReLU, identity add; fbocc-r50 config ffn_cfgs) and
 * the following `norm` of operation_order (bevformer_encoder.py:251-377).  The
 * hidden activation (m x hidden) lives in TMEM / shared memory only.
 * w1_packed: hidden / 80 consecutive blocks, block c = fbbev_linear_pack of
 *   rows [80 c, 80 c + 80) of W1 (hidden, embed) -- i.e. fbbev_linear_pack(n = 80,
 *   k = embed) per block, fbbev_linear_packed_bytes(80, embed) bytes each;
 * w2_packed: fbbev_linear_pack(W2 (embed, hidden)).
 * b1 (hidden), b2 (embed), residual (m, embed; row stride ldr), ln_weight /
 * ln_bias (embed) may be NULL.  embed <= 80, embed % 4 == 0, hidden % 80 == 0,
 * hidden <= 320 (fbbev_ffn_supported); FBBEV_ERR_UNSUPPORTED otherwise (use
 * fbbev_linear_fwd per Linear).  Numerics as fbbev_linear_fwd (3xTF32).
 */
int fbbev_ffn_supported(int32_t embed, int32_t hidden);
int fbbev_ffn_fwd(const float* x, int64_t ldx, const float* w1_packed,
                  const float* b1, const float* w2_packed, const float* b2,
                  const float* residual, int64_t ldr, const float* ln_weight,
                  const float* ln_bias, int64_t m, int32_t embed,
                  int32_t hidden, float ln_eps, float* y, int64_t ldy,
                  fbbev_stream_t stream);

/* =====================================================================
 * T -- temporal fusion of the BEV / voxel history (the stage after the path)
 * ===================================================================== */

/*
 * The sampling half of `FBOCC.fuse_history`
 *   mmdet3d/models/fbbev/detectors/fbocc.py:207-319, `generate_grid` :170-205:
 *   grid = rt_flow @ (x, y, z, 1); normalise; F.grid_sample(history, grid,
 *   align_corners=True, bilinear, zeros); torch.cat([curr_bev, sampled], 1)
 * as one pass.  history (n, mc, Z, H, W) fp32 = the T previous frames stacked
 * along channels, samples history_batch_stride floats apart (>= mc*Z*H*W: the
 * history may be a channel slice of the previous step's concatenation buffer); flow (n, 4, 4) row-major = inverse(feat2bev) @ history_augs @
 * curr_to_prev_ego_rt @ inverse(forward_augs) @ feat2bev (:196-197), mapping
 * voxel indices (x, y, z, 1) of the current frame to voxel indices of the
 * history; out (n, c_total, Z, H, W): the warped history is written into
 * channels [ch_offset, ch_offset + mc) -- pass the concatenation buffer and
 * ch_offset = C so that no torch.cat copy is needed.  The 5-D grid tensor is
 * never materialised.
 */
int fbbev_history_warp(const float* history, int64_t history_batch_stride,
                       const float* flow, int32_t n, int32_t mc, int32_t Z,
                       int32_t H, int32_t W, float* out, int32_t c_total,
                       int32_t ch_offset, fbbev_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FBBEV_B200_H_ */
