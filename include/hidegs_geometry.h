/*
 * hidegs_geometry.h — C-ABI of the geometry prologue / epilogue that surround the rasterizer call in
 * the reference's render() (gaussian_renderer/__init__.py:36-214), of the single-view normal-consistency
 * term of the training loss, of the fused Adam step and of simple-knn's distCUDA2.
 *
 * Conventions as in hidegs_raster.h: device pointers (fp32 unless stated), sizes, scalars, a cudaStream_t
 * passed as void*; int status return (hg_status); no host synchronisation inside unless stated.
 *
 * Reference functions replaced (paths relative to the reference tree):
 *   hg_geometry_all_map            gaussian_renderer/__init__.py:161-169 (input_all_map) with
 *                                  GaussianModel.get_normal / get_smallest_axis / get_rotation_matrix
 *                                  (scene/gaussian_model.py:150-166; pytorch3d quaternion_to_matrix)
 *   hg_geometry_all_map_backward   the autograd backward of the above (~10 PyTorch ops)
 *   hg_depth_normal                render_normal (gaussian_renderer/__init__.py:21-33) ->
 *                                  normal_from_depth_image / depth2point_world / depth2point_cam / ndc_2_cam /
 *                                  depth_pcd2normal (utils/graphics_utils.py:17-23,108-166), offset=None,
 *                                  scale=1, times rendered_alpha.detach() (gaussian_renderer/__init__.py:201)
 *   hg_depth_normal_backward       its autograd backward w.r.t. the plane depth
 *   hg_normal_consistency_loss     single-view term  w * mean(image_weight * sum_c |depth_normal_c - normal_c|)
 *                                  (weights arguments/__init__.py:118-119; composed from render()'s
 *                                  "depth_normal" / "rendered_normal" outputs and get_img_grad_weight,
 *                                  utils/loss_utils.py:66-78; see DESIGN.md for the definition)
 *   hg_activate_params(+_backward) scene/gaussian_model.py:60-75,118-137 (exp / sigmoid / normalize activations and their
 *                                  autograd backward, fused with the gradient accumulation of a multi-view step)
 *   hg_adam_step                   scene/OurAdam.py:106-337 (Adam update of the parameter groups; dense and
 *                                  visibility-masked "sparse" variant)
 *   hg_expand_to_size, hg_interpolation_weights   gaussian_hierarchy._C.expand_to_size / get_interpolation_weights
 *                                  (submodules/gaussianhierarchy/runtime_switching.cu:402-527, torch/torch_interface.cpp:77-119)
 *   hg_dist2_knn3                  simple_knn: distCUDA2 -> SimpleKNN::knn (submodules/simple-knn/spatial.cu:15-26,
 *                                  simple_knn.cu:186-222): mean squared distance to the 3 nearest neighbours
 */
#ifndef HIDEGS_GEOMETRY_H
#define HIDEGS_GEOMETRY_H

#include <stddef.h>
#include <stdint.h>
#include "hidegs_raster.h"

#ifdef __cplusplus
extern "C" {
#endif

/* all_map[n] = [ R_view^T normal_n (3), 1, |<normal_view, p_view>| ] with normal_n = the column of
 * quaternion_to_matrix(rotation_n) that belongs to the smallest scaling axis, flipped to face campos.
 * xyz [N,3], scaling [N,3] (activated), rotation [N,4] (real-first; need not be normalised),
 * viewmatrix [16] (row-vector convention, cameras.py:127), campos [3]; out [N,5]. */
HG_API int hg_geometry_all_map(const float *xyz, const float *scaling, const float *rotation,
                               const float *viewmatrix, const float *campos, int64_t N, float *out_all_map,
                               void *stream);

/* dL/dxyz [N,3] and dL/drotation [N,4] from dL/dall_map [N,5]; both outputs are fully WRITTEN (not
 * accumulated).  No gradient reaches the scaling (argmin) or the camera. */
HG_API int hg_geometry_all_map_backward(const float *xyz, const float *scaling, const float *rotation,
                                        const float *viewmatrix, const float *campos, int64_t N,
                                        const float *dL_dall_map, float *dL_dxyz, float *dL_drotation,
                                        void *stream);

/* Parameter activations of GaussianModel (scene/gaussian_model.py:60-75,118-137): scaling = exp(raw), opacity =
 * sigmoid(raw), rotation = raw / max(|raw|, 1e-12) (torch.nn.functional.normalize).  Forward writes the three
 * activated arrays; backward chains the gradients w.r.t. the activated arrays (and the pass-through gradients of xyz
 * [N,3] and features [N,F]) back to the raw parameters and stores them into the five destination arrays
 *   dst = beta * dst + chain(grad),  beta = 0 (overwrite) or 1 (accumulate across the views of a step).
 * Any gradient pointer may be NULL (= zero gradient). */
HG_API int hg_activate_params(const float *raw_scaling, const float *raw_rotation, const float *raw_opacity,
                              int64_t N, float *scaling, float *rotation, float *opacity, void *stream);
HG_API int hg_activate_params_backward(const float *raw_scaling, const float *raw_rotation, const float *raw_opacity,
                                       int64_t N, int32_t F, const float *g_xyz, const float *g_features,
                                       const float *g_opacity, const float *g_scaling, const float *g_rotation,
                                       float beta, float *d_xyz, float *d_features, float *d_opacity,
                                       float *d_scaling, float *d_rotation, void *stream);

/* The executor's fused prologue backward of a training view: all_map backward (gaussian_renderer/__init__.py:161-169
 * and its autograd) + the gradient of the scale regulariser (g_scaling_extra * *extra_scale, a DEVICE scalar; both may
 * be NULL) + hg_activate_params_backward, in one pass over the rows the view rendered.  `radii` (int32 [N], the
 * rasterizer's output; may be NULL = every row): rows with radii <= 0 are zero-filled (beta = 0) or left alone
 * (beta = 1) WITHOUT reading their gradient rows, so the rasterizer's backward may leave them unwritten
 * (HG_BWD_SKIP_CULLED_ROWS of hg_raster_backward_chunked).  g_* are the rasterizer's gradients w.r.t. the ACTIVATED
 * parameters, g_all_map its dL/dall_map [N,5]; xyz / viewmatrix / campos as in hg_geometry_all_map. */
HG_API int hg_prologue_backward(const float *raw_scaling, const float *raw_rotation, const float *raw_opacity,
                                const float *xyz, int64_t N, int32_t F, const int32_t *radii, const float *viewmatrix,
                                const float *campos, const float *g_xyz, const float *g_features,
                                const float *g_opacity, const float *g_scaling, const float *g_rotation,
                                const float *g_all_map, const float *g_scaling_extra, const float *extra_scale,
                                float beta, float *d_xyz, float *d_features, float *d_opacity, float *d_scaling,
                                float *d_rotation, void *stream);

/* Camera intrinsics as Camera.get_calib_matrix_nerf builds them (scene/cameras.py:93-96,135-138). */
typedef struct hg_intrinsics {
  float fx, fy, cx, cy;
} hg_intrinsics;

/* depth_normal [3,H,W] = pad(normalize(cross(P(y,x+1)-P(y,x-1), P(y-1,x)-P(y+1,x)))) * alpha, P = the
 * unprojected plane depth; alpha [H,W] may be NULL (plain render_normal). */
HG_API int hg_depth_normal(const float *plane_depth, const float *alpha, int32_t H, int32_t W, hg_intrinsics K,
                           float *out_normal, void *stream);

/* dL/dplane_depth [H,W] (fully written) from dL/ddepth_normal [3,H,W]; alpha is treated as a constant
 * (the reference detaches it). */
HG_API int hg_depth_normal_backward(const float *plane_depth, const float *alpha, const float *dL_dnormal,
                                    int32_t H, int32_t W, hg_intrinsics K, float *dL_dplane_depth, void *stream);

/* Fused forward + backward of the single-view normal-consistency term:
 *   loss = weight * mean_{H,W}( image_weight * sum_c | depth_normal_c - all_map_c | ),  c = 0..2,
 * depth_normal as in hg_depth_normal with alpha = all_map[3] (detached).  image_weight [H,W] may be NULL (= 1).
 * Writes out_loss[0]; if dL_dplane_depth / dL_dall_map are non-NULL they receive the gradient for a unit
 * upstream gradient ([H,W] and [5,H,W]; channels 3, 4 of the latter are zero).  workspace:
 * hg_normal_consistency_workspace_bytes(H, W) bytes. */
HG_API size_t hg_normal_consistency_workspace_bytes(int32_t H, int32_t W);
HG_API int hg_normal_consistency_loss(const float *plane_depth, const float *all_map, const float *image_weight,
                                      int32_t H, int32_t W, hg_intrinsics K, float weight, float *out_loss,
                                      float *dL_dplane_depth, float *dL_dall_map, void *workspace, void *stream);

/* One Adam step over a flat fp32 parameter block of n_rows rows of row_width floats (torch.optim.Adam
 * semantics as used by OurAdam.py: no weight decay, no amsgrad):
 *   m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps).
 * Row selection (the reference's `relevant`, OurAdam.py:249-337; rows not selected keep parameter AND state):
 *   visible_mask (u8 [n_rows]) or visible_idx (int64 [n_idx], unique entries) or neither (every row, the
 *   reference's _single_tensor_adam2 path for an empty `relevant`).  `step` is the 1-based step count of the
 *   parameter; grad_scale multiplies g on the fly (e.g. 1/views after a SUM all-reduce).  lr / betas / eps are
 *   The first `head_cols` columns of every row step with `head_lr` instead of `lr` (the SH block [N,16,3] holds the DC
 *   term, learning rate feature_lr, in its first 3 columns and the rest at feature_lr / 20, as the two parameter groups
 *   of GaussianModel.training_setup do; head_cols = 0 for a uniform rate).  lr / betas / eps are
 *   doubles, as Python hands them to torch (`1 - beta2` is formed in double before it is narrowed to fp32). */
HG_API int hg_adam_step(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, int64_t n_rows,
                        int32_t row_width, const uint8_t *visible_mask, const int64_t *visible_idx, int64_t n_idx,
                        double lr, double beta1, double beta2, double eps, int32_t step, float grad_scale,
                        int32_t head_cols, double head_lr, void *stream);

/* GaussianModel.add_densification_stats (scene/gaussian_model.py:763-765) for update_filter = (radii > 0), fused with the
 * training loop's max_radii2D update:  accum[n] = max(|grad_means2D[n, :2]|, accum[n]); denom[n] += 1;
 * max_radii2D[n] = max(max_radii2D[n], radii[n]) (max_radii2D may be NULL).  grad_means2D [N,3], radii [N] i32. */
HG_API int hg_densification_stats(const float *grad_means2D, const int32_t *radii, int64_t N,
                                  float *xyz_gradient_accum, float *denom, float *max_radii2D, void *stream);

/* Adaptive density control over the training arenas (DESIGN.md §3 "Densify and prune"): graphdeco 3DGS
 * densify_and_clone + densify_and_split + prune, in three steps.  An arena holds the five groups of N rows
 * xyz 3 | features 48 | opacity 1 (logit) | scaling 3 (log) | rotation 4, each starting at group_offsets[g] (host
 * int64 [5], in floats, multiples of 4; GaussianParams' layout), 16-byte aligned.
 *   hg_densify_plan: g = accum (NaN -> 0), smax = max exp(scaling); clone C = |g| >= max_grad && smax <= (float)(
 *     percent_dense * extent); split S = g >= max_grad && smax > that; a row of the output is pruned when
 *     sigmoid(opacity) < min_opacity or (max_screen_size > 0, 0 = None) smax > (float)(0.1 * extent).  Writes the
 *     decisions into `workspace` (hg_densify_workspace_bytes(N) bytes) and returns through host out-params the kept
 *     original rows, |C|, |S| and N'.  Synchronises the stream once (N' sizes the new arenas).  A model with
 *     skybox_points != 0 is rejected.
 *   hg_densify_apply: from the same workspace, writes the N' rows [kept rows | clones | first children | second
 *     children] (each in source order, pruned rows left out) into the new parameter arena and both new Adam moment
 *     arenas (kept rows keep their moments, new rows start at zero; pad floats are zeroed).  Children: xyz = R(q) s + xyz
 *     with s = exp(scaling) * z, z ~ N(0, I) from Philox4x32-10 (key = seed, counter = (source row, child)), or
 *     s = samples [2|S|, 3] (rows: first children, then second children, in source order) when non-NULL;
 *     scaling = log(exp(scaling) / 1.6); features, opacity, rotation copied.
 *   hg_reset_opacity: opacity = inverse_sigmoid(min(sigmoid(opacity), 0.01)) over N floats, and that group's two
 *     moment blocks zeroed. */
HG_API size_t hg_densify_workspace_bytes(int64_t N);
HG_API int hg_densify_plan(const float *param, const int64_t *group_offsets, int64_t N, const float *accum,
                           int32_t skybox_points, double max_grad, double min_opacity, double extent,
                           double max_screen_size, double percent_dense, void *workspace, int64_t *out_kept,
                           int64_t *out_cloned, int64_t *out_split, int64_t *out_new_n, void *stream);
HG_API int hg_densify_apply(const float *old_param, const float *old_exp_avg, const float *old_exp_avg_sq,
                            const int64_t *old_offsets, int64_t N, float *new_param, float *new_exp_avg,
                            float *new_exp_avg_sq, const int64_t *new_offsets, int64_t new_n, const float *samples,
                            uint64_t seed, const void *workspace, void *stream);
HG_API int hg_reset_opacity(float *opacity, float *exp_avg, float *exp_avg_sq, int64_t N, void *stream);

/* Hierarchy LOD cut (SURVEY.md §8(f) f1).  nodes [N,7] i32 (types.h:47-56: depth, parent, start, count_leafs,
 * count_merged, start_children, count_children), boxes [N,2,4] f32 (min xyz + extent, max xyz + pad), viewpoint [3] on
 * the device.  hg_expand_to_size = Switching::expandToSize (runtime_switching.cu:496-527): for every node whose
 * projected size is >= target (or whose parent's is), its Gaussians go to render_indices (with the parent node's first
 * Gaussian in parent_indices and the node id in nodes_for_render_indices; both nullable; node_markers nullable), in
 * node order.  *out_count (host) receives the number of indices; the index buffers hold `capacity` entries (the reference
 * writes without a bound).  Synchronises the stream once, as the reference's blocking cudaMemcpy does.
 * hg_interpolation_weights = Switching::getTsIndexed (:433-494): ts[i], kids[i] for node indices[i]. */
HG_API size_t hg_expand_to_size_workspace_bytes(int32_t N);
HG_API int hg_expand_to_size(const int32_t *nodes, const float *boxes, int32_t N, float target_size,
                             const float *viewpoint, int32_t capacity, int32_t *render_indices,
                             int32_t *parent_indices, int32_t *nodes_for_render_indices, int32_t *node_markers,
                             void *workspace, int32_t *out_count, void *stream);
HG_API int hg_interpolation_weights(const int32_t *indices, int32_t n, float target_size, const int32_t *nodes,
                                    const float *boxes, float vx, float vy, float vz, float *ts, int32_t *kids,
                                    void *stream);

/* Parent interpolation of a hierarchy cut — the `interp_python` branch of render_post
 * (gaussian_renderer/__init__.py:278-318): for e < E, out[e] = ts[e] * x[render_indices[e]] + (1 - ts[e]) *
 * x[parent_indices[e]] for means3D [N,3], scales [N,3], rotations [N,4] (the parent's quaternion negated when its dot
 * product with the child's is negative), opacity [N,1] and shs [N,M,3]; rows E..E+S-1 are the model's last S rows
 * (skybox).  Negative indices wrap like torch indexing.  Outputs hold E+S rows.  The backward ACCUMULATES (atomics)
 * into d_* [N,...], which the caller zero-fills; any g_x / d_x pair may be NULL. */
HG_API int hg_hier_interpolate(const float *means3D, const float *scales, const float *rotations, const float *opacity,
                               const float *shs, int64_t N, int32_t M, const int32_t *render_indices,
                               const int32_t *parent_indices, const float *ts, int64_t E, int64_t S,
                               float *out_means3D, float *out_scales, float *out_rotations, float *out_opacity,
                               float *out_shs, void *stream);
HG_API int hg_hier_interpolate_backward(const float *rotations, int64_t N, int32_t M, const int32_t *render_indices,
                                        const int32_t *parent_indices, const float *ts, int64_t E, int64_t S,
                                        const float *g_means3D, const float *g_scales, const float *g_rotations,
                                        const float *g_opacity, const float *g_shs, float *d_means3D, float *d_scales,
                                        float *d_rotations, float *d_opacity, float *d_shs, void *stream);

/* Mean squared distance of every point to its 3 nearest neighbours (exact).  points [N,3] -> out [N].
 * workspace: hg_dist2_knn3_workspace_bytes(N) bytes.  No host synchronisation. */
HG_API size_t hg_dist2_knn3_workspace_bytes(int64_t N);
HG_API int hg_dist2_knn3(const float *points, int64_t N, float *out_mean_dist2, void *workspace, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HIDEGS_GEOMETRY_H */
