/*
 * qed_splat.h — C-ABI of the B200-native (sm_100a) depth-supervised splat render/train hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference,
 * leggedrobotics/qed-splatter, reaches this path through ONE Python call,
 *     gsplat.rendering.rasterization(...)            qed_splatter/model.py:267-288
 * (import at qed_splatter/model.py:6-9) and through torch autograd for the backward
 * (loss at qed_splatter/model.py:73-118).  gsplat 1.4.0 implements that call as a chain
 * of torch custom ops over its CUDA extension `gsplat_cuda`
 * (gsplat/cuda/_wrapper.py: fully_fused_projection, spherical_harmonics, isect_tiles,
 * isect_offset_encode, rasterize_to_pixels).  Every entry point below names the gsplat op
 * (and hence the stage of the model.py:267-288 call) it replaces.
 *
 * Conventions
 *   - plain C: raw device pointers + extents; contiguous row-major tensors; no torch types.
 *   - every function returns int: 0 = ok, < 0 = QED_ERR_* argument error, > 0 = cudaError_t.
 *   - never throws, never exits, never synchronises the device, holds no mutable state shared
 *     between threads (the qed_debug_* test hooks, which are not declared here, are thread-local);
 *     all work is enqueued on the `stream` argument (a cudaStream_t).
 *   - caller owns every buffer.  Outputs are fully overwritten unless stated "accumulates".
 *   - float = IEEE binary32.  "flat index" = c*N + n into the [C,N,...] arrays.
 */
#ifndef QED_SPLAT_H_
#define QED_SPLAT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* qed_stream_t; /* cudaStream_t */

#define QED_OK 0
#define QED_ERR_BAD_ARG (-1)
#define QED_ERR_UNSUPPORTED (-2)
#define QED_ERR_WORKSPACE (-3)

#define QED_ABI_VERSION 3

/* Library / ABI version (QED_ABI_VERSION the .so was built with). */
int qed_abi_version(void);
/* Static string for a return code of any function here (cudaGetErrorString for > 0). */
const char* qed_error_string(int code);

/* `activations` bits of qed_project_fwd / qed_project_bwd */
#define QED_ACT_LOG_SCALES 1
#define QED_ACT_LOGIT_OPACITIES 2

/* ------------------------------------------------------------------------------------------------
 * (a) fused projection + EWA 2-D covariance + SH colour + tile count
 * replaces: gsplat fully_fused_projection (fwd) + spherical_harmonics (fwd) + the
 *           `clamp_min(colors + 0.5, 0)`, depth-channel concat and opacity*compensation glue of
 *           gsplat.rendering.rasterization, + the counting pass of isect_tiles.
 *           Reached from qed_splatter/model.py:267-288 (args means, quats, scales, opacities,
 *           colors, viewmats, Ks, width, height, near_plane, far_plane, sh_degree, rasterize_mode).
 *
 *  means[N,3] quats[N,4](wxyz) scales[N,3] opacities[N]
 *  activations: 0 = scales / opacities are the activated values gsplat takes; QED_ACT_LOG_SCALES and/or
 *             QED_ACT_LOGIT_OPACITIES = they are the stored parameters and exp / sigmoid
 *             (qed_splatter/model.py:269-271) are applied inside the kernel; qed_project_bwd then returns the
 *             gradients with respect to the stored parameters (chain rule folded in).
 *  colors_in: sh_degree >= 0 : SH coefficients [N,K,3], uses the first (sh_degree+1)^2 of K
 *             sh_degree <  0 : colours [N,3] (colors_per_camera=0) or [C,N,3] (=1); ignored when n_color==0
 *  viewmats[C,4,4] world->camera, Ks[C,3,3]
 *  n_color in {0,3}: colour channels produced; append_depth in {0,1}: depth appended as last channel.
 *      D = n_color + append_depth must be 1, 3 or 4   (render_mode D/ED -> 0+1, RGB -> 3+0, RGB+D/ED -> 3+1)
 *  outputs (all [C,N,...]):
 *      radii i32, means2d[.,2], depths, conics[.,3], compensations (NULL unless calc_compensations),
 *      colors_out[.,D], opacities_out (opacity * compensation), tiles_per_gauss i32,
 *      tiles_exact i32 (NULL to skip): how many of those tiles the Gaussian can reach with alpha >= 1/255 at a pixel centre
 *      (one interval of tile columns per tile row of the bounding box; conservative) -- the count EXACT tile lists are
 *      built from: pass it to qed_isect_prepare instead of tiles_per_gauss and geom to qed_isect_fill.
 *      geom[.,8] packed {mx,my,opacity,depth | conic a,b,c, 0} = the record the compositor gathers.
 *  Culled entries (radii == 0) get zeros everywhere.
 */
int qed_project_fwd(int C, int N, const float* means, const float* quats, const float* scales,
                    const float* opacities, int activations, const float* colors_in, int K, int sh_degree,
                    int colors_per_camera, const float* viewmats, const float* Ks, int width, int height,
                    float eps2d, float near_plane, float far_plane, float radius_clip,
                    int calc_compensations, int tile_size, int n_color, int append_depth,
                    int32_t* radii, float* means2d, float* depths, float* conics, float* compensations,
                    float* colors_out, float* opacities_out, int32_t* tiles_per_gauss, int32_t* tiles_exact, float* geom,
                    qed_stream_t stream);

/* Backward of qed_project_fwd.
 * replaces: gsplat fully_fused_projection (bwd) + spherical_harmonics (bwd) + the glue above.
 *  v_means2d[C,N,2] v_depths[C,N] v_conics[C,N,3] v_colors[C,N,D] v_opacities_cn[C,N]
 *      (any may be NULL = zero).  When `packed_grads` != NULL it is the [C*N,12] record written by
 *      qed_raster_bwd {v_mx,v_my,abs_x,abs_y | v_ca,v_cb,v_cc,v_opacity | v_colour[0..3]} and is
 *      ADDED to the separate arrays (fused path: pass only packed_grads).
 *  outputs (overwritten): v_means[N,3] v_quats[N,4] v_scales[N,3] v_opacities[N]
 *      v_colors_in: same shape as colors_in ([N,K,3], all K rows written, unused ones zero).
 *  Gradients are summed over the C cameras in a fixed order (deterministic).
 */
int qed_project_bwd(int C, int N, const float* means, const float* quats, const float* scales,
                    const float* opacities, int activations, const float* colors_in, int K, int sh_degree,
                    int colors_per_camera, const float* viewmats, const float* Ks, int width, int height,
                    float eps2d, int calc_compensations, int n_color, int append_depth,
                    const int32_t* radii, const float* conics, const float* compensations,
                    const float* v_means2d, const float* v_depths, const float* v_conics,
                    const float* v_colors, const float* v_opacities_cn, const float* packed_grads,
                    float* v_means, float* v_quats, float* v_scales, float* v_opacities,
                    float* v_colors_in, qed_stream_t stream);

/* qed_project_bwd that also returns the gradient with respect to the camera poses (gsplat's v_viewmats; splatfacto's
 * camera optimizer, whose poses enter through qed_splatter/model.py:212,246).
 *  Same arguments and outputs as qed_project_bwd, plus
 *  v_viewmats[C,4,4] (overwritten): d loss / d viewmats over every visible (view, Gaussian): the camera-space mean
 *      (p = W mu + t), the camera-space covariance (W Sigma W^T, incl. the antialiasing compensation) and, with SH colours,
 *      the view direction mu - campos with campos = -W^-1 t (general inverse).  Row 3 is zero.
 *  workspace: device memory of at least qed_project_bwd_pose_workspace_bytes(C, N) bytes, 16-byte aligned (per-warp partial
 *      sums; may be NULL when N == 0).
 *  Deterministic: no atomics; partials are summed in a fixed order in float64.  C <= 1024 as for qed_project_bwd. */
size_t qed_project_bwd_pose_workspace_bytes(int C, int N);
int qed_project_bwd_pose(int C, int N, const float* means, const float* quats, const float* scales,
                         const float* opacities, int activations, const float* colors_in, int K, int sh_degree,
                         int colors_per_camera, const float* viewmats, const float* Ks, int width, int height,
                         float eps2d, int calc_compensations, int n_color, int append_depth,
                         const int32_t* radii, const float* conics, const float* compensations,
                         const float* v_means2d, const float* v_depths, const float* v_conics,
                         const float* v_colors, const float* v_opacities_cn, const float* packed_grads,
                         float* v_means, float* v_quats, float* v_scales, float* v_opacities,
                         float* v_colors_in, float* v_viewmats, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* Pack separate arrays into the compositor's geom record (op-level entry for callers that did not
 * come through qed_project_fwd, e.g. gsplat-style rasterize_to_pixels(means2d, conics, ..)). */
int qed_pack_geom(int CN, const float* means2d, const float* conics, const float* opacities,
                  const float* depths /* may be NULL */, float* geom, qed_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (b) tile intersection: count -> scan -> emit keys -> sort -> per-tile ranges (all integer, bit-exact)
 * replaces: gsplat isect_tiles (count pass, torch cumsum, fill pass, cub::DeviceRadixSort) and
 *           isect_offset_encode.  Reached from model.py:267-288 via tile_size=16 (model.py:243,277).
 */

/* tiles_per_gauss[C*N] from means2d/radii (only needed when projection was not done by qed_project_fwd). */
int qed_isect_count(int C, int N, const float* means2d, const int32_t* radii, int tile_size, int tile_width,
                    int tile_height, int32_t* tiles_per_gauss, qed_stream_t stream);

/* Workspace (bytes) for qed_isect_scan over n elements. */
size_t qed_isect_scan_workspace_bytes(int64_t n);
/* Inclusive prefix sum cum[i] = sum_{j<=i} tiles_per_gauss[j] (int64); *n_isects_dev = cum[n-1] (int64, device).
 * Also copies the total to `n_isects_host_pinned` (int64 in pinned host memory) when non-NULL, asynchronously. */
int qed_isect_scan(int64_t n, const int32_t* tiles_per_gauss, int64_t* cum, int64_t* n_isects_dev,
                   int64_t* n_isects_host_pinned, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* Emit unsorted (key,value): key = cam << (32+tile_n_bits) | tile << 32 | bits(depth); value = flat index.
 * Emission order: ascending flat index, then tile rows, then tile columns (gsplat isect_tiles fill pass). */
int qed_isect_emit(int C, int N, const float* means2d, const int32_t* radii, const float* depths,
                   const int64_t* cum, int tile_size, int tile_width, int tile_height, int64_t* isect_ids,
                   int32_t* flatten_ids, qed_stream_t stream);

/* Stable ascending sort of (int64 key, int32 value) pairs on key bits [0, end_bit).
 * qed_sort_pairs_cub is the library baseline (what gsplat calls); qed_sort_pairs is this library's own
 * radix sort.  Both produce identical output.  keys_in/vals_in may be clobbered. */
size_t qed_sort_pairs_workspace_bytes(int64_t n);
int qed_sort_pairs(int64_t n, int64_t* keys_in, int32_t* vals_in, int64_t* keys_out, int32_t* vals_out,
                   int end_bit, void* workspace, size_t workspace_bytes, qed_stream_t stream);
size_t qed_sort_pairs_cub_workspace_bytes(int64_t n);
int qed_sort_pairs_cub(int64_t n, int64_t* keys_in, int32_t* vals_in, int64_t* keys_out, int32_t* vals_out,
                       int end_bit, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* Two-level build of the same sorted intersection list (the product path; identical output to
 * qed_isect_emit + qed_sort_pairs + qed_tile_ranges with ~5x less memory traffic):
 *   prepare: ordered compaction of the visible (camera, Gaussian) entries, stable radix sort by
 *            (camera, depth bits), scan of their tile counts in that order.
 *            counts_dev[2] (int64, device) = {n_visible, n_isects}; also copied asynchronously to
 *            counts_host_pinned[2] when non-NULL (the caller reads it after a stream sync to size outputs).
 *   fill:    warp-cooperative coalesced emission of (camera|tile, flat index) in depth order, stable radix
 *            sort on the camera|tile bits only, then isect_ids = key << 32 | bits(depth) and the per-tile
 *            ranges (isect_ids and/or isect_offsets may be NULL to skip them; the compositor needs only
 *            flatten_ids + isect_offsets).
 * `prepare_workspace` must be the buffer qed_isect_prepare filled for the same (C, N).
 *
 * geom == NULL: gsplat's lists, bit for bit (every tile of each Gaussian's 3-sigma bounding box; prepare ran on
 *   tiles_per_gauss; n_isects entries).
 * geom != NULL (the packed [C*N,8] records of qed_project_fwd; prepare ran on its tiles_exact): EXACT tile lists -- only
 *   the (Gaussian, tile) pairs that can reach alpha >= 1/255 at a pixel centre of the tile, about half of gsplat's
 *   entries, and no pixel changes.  The projection kernel counted them, this call enumerates the same spans: n_visible /
 *   n_isects are the counts of THAT prepare call.  isect_offsets must have C*tile_height*tile_width + 1 elements, the last
 *   one receiving the end of the last range (pass offsets_has_end = 1 to qed_raster_fwd).
 * n_exact_dev (optional, any mode): receives the number of entries written, on the device (int64).
 *
 * counts_dev != NULL (= the counts_dev of qed_isect_prepare): NO host synchronisation is needed between prepare and fill.
 *   n_visible / n_isects are then CAPACITIES (n_visible = C*N is always enough; n_isects = what the caller sized
 *   flatten_ids / isect_ids / the workspace for); the real counts are read on the device.  isect_offsets must have
 *   C*tile_height*tile_width + 1 elements (its last element receives the end of the last range, pass offsets_has_end = 1
 *   to qed_raster_fwd) also for gsplat's lists.  If the real entry count exceeds the capacity an EMPTY list is built
 *   (every consumer stays memory-safe) -- the caller reads counts_host_pinned once the work is queued, sees the
 *   overflow, grows its buffers and repeats the fill (pipeline.FusedSplatStep does; the device never idles on that read). */
size_t qed_isect_prepare_workspace_bytes(int64_t CN);
int qed_isect_prepare(int C, int N, const float* depths, const int32_t* tiles_per_gauss, void* workspace,
                      size_t workspace_bytes, int64_t* counts_dev, int64_t* counts_host_pinned, qed_stream_t stream);
size_t qed_isect_fill_workspace_bytes(int64_t n_isects);
int qed_isect_fill(int C, int N, int64_t n_visible, int64_t n_isects, const float* means2d, const int32_t* radii,
                   const float* depths, const float* geom, int image_width, int image_height, int tile_size, int tile_width,
                   int tile_height, const void* prepare_workspace, void* workspace, size_t workspace_bytes,
                   const int64_t* counts_dev, int64_t* isect_ids, int32_t* flatten_ids, int32_t* isect_offsets,
                   int64_t* n_exact_dev, qed_stream_t stream);

/* isect_offsets[C*tile_height*tile_width] i32: first sorted index of each (camera,tile); empty tiles get
 * the start of the next non-empty one; tiles after the last entry get n_isects. */
int qed_tile_ranges(int64_t n_isects, const int64_t* isect_ids_sorted, int C, int tile_width, int tile_height,
                    int32_t* isect_offsets, qed_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (c) per-tile front-to-back compositing of D channels (RGB + depth)
 * replaces: gsplat rasterize_to_pixels (fwd) + the ED normalisation tail of rasterization().
 *  geom[C*N,8], colors[C*N,D] gathered through flatten_ids; backgrounds[C,D] or NULL.
 *  normalize_last != 0 : last channel /= max(alpha, 1e-10) (render_mode ED / RGB+ED).
 *  outputs: render[C,H,W,D], alphas[C,H,W], last_ids[C,H,W] i32 (index in sorted list of the last
 *  composited Gaussian; 0 if none).  For normalize_last the un-normalised last channel is
 *  recoverable as render*max(alpha,1e-10) (the backward does so).
 *  offsets_has_end != 0 : isect_offsets has one more element holding the end of the last range (exact tile
 *  lists of qed_isect_fill, whose entry count lives on the device); n_isects is then only an upper bound.
 */
int qed_raster_fwd(int C, int N, int64_t n_isects, int D, const float* geom, const float* colors,
                   const float* backgrounds, int width, int height, int tile_size, int tile_width,
                   int tile_height, const int32_t* isect_offsets, int offsets_has_end, const int32_t* flatten_ids,
                   int normalize_last, float* render, float* alphas, int32_t* last_ids, qed_stream_t stream);

/* (d) compositing backward.
 * replaces: gsplat rasterize_to_pixels (bwd) incl. absgrad (model.py:284 absgrad=True).
 *  v_render[C,H,W,D], v_alphas[C,H,W] (NULL = zero): gradients w.r.t. the OUTPUTS of qed_raster_fwd
 *  (i.e. after ED normalisation when normalize_last).
 *  packed_grads[C*N,12] ACCUMULATES (caller zero-fills): {v_mx,v_my,|v_mx|,|v_my| | v_conic a,b,c,
 *  v_opacity | v_colour[0..D-1], 0..}.  Per warp and Gaussian the 12 values are summed over the lanes (transposed through
 *  shared memory) and added with vector reductions (red.global.add.v4.f32): the sums are order-dependent in the last bits.
 */
int qed_raster_bwd(int C, int N, int64_t n_isects, int D, const float* geom, const float* colors,
                   const float* backgrounds, int width, int height, int tile_size, int tile_width,
                   int tile_height, const int32_t* isect_offsets, const int32_t* flatten_ids,
                   int normalize_last, const float* render, const float* alphas, const int32_t* last_ids,
                   const float* v_render, const float* v_alphas, float* packed_grads, qed_stream_t stream);

/* Unpack packed_grads into gsplat-shaped gradient tensors (any output may be NULL). */
int qed_unpack_grads(int CN, int D, const float* packed_grads, float* v_means2d, float* v_means2d_abs,
                     float* v_conics, float* v_colors, float* v_opacities, qed_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * (d') qed-splatter loss + its gradient w.r.t. the compositor outputs, fused
 * replaces: the autograd graph of qed_splatter/model.py:295-306 (background composite, clamp, depth fill)
 *           and :87-116 (masked depth-L1 * depth_lambda) + the L1 term of splatfacto's RGB loss
 *           (model.py:83-85), i.e. SURVEY.md §8 rows a11-a13.
 *  render[C,H,W,4] (RGB + depth; depth normalised iff normalize_last), alphas[C,H,W],
 *  gt_rgb[C,H,W,3]: float32 in [0,1], or (gt_rgb_is_u8 != 0) the uint8 image cache of the data side
 *      (qed_splatter/config.py:37 cache_images_type="uint8"), converted as splatfacto's `image.float() / 255.0` does on CUDA (u8 * (1.0f / 255.0f)) at the point of use;
 *  gt_depth[C,H,W] (<=0 or non-finite = invalid): float32 metres, or (gt_depth_is_u16 != 0) the raw uint16 sensor image,
 *      converted at the point of use as nerfstudio's depth loader does with the reference's unit scale
 *      (qed_splatter/dataparser.py:15 depth_unit_scale_factor = 0.001, times the scene scale): float(double(u16) *
 *      depth_unit_scale); bg[3].
 *  mask[C,H,W] or NULL: the batch's `mask` (qed_splatter/model.py:93-97), float32 or (mask_is_u8 != 0) uint8 / bool.
 *      As in the reference, rendered and ground-truth depth are both multiplied by it BEFORE the validity test
 *      (model.py:96-97), and -- splatfacto's parent loss, model.py:83-85 -- so are the predicted and ground-truth
 *      RGB images before L1 and SSIM (means still run over all H*W pixels).  The depth fill value stays the
 *      maximum of the unmasked rendered depth (model.py:304-306 run before the loss).
 *  loss = rgb_weight * mean|m clamp(rgb + (1-a) bg) - m gt| + ssim_lambda * (1 - SSIM(m clamped rgb, m gt))
 *         + depth_lambda * mean_valid|m depth - m gt_depth|,  per camera (one camera = one reference step: its own
 *         depth fill / n_valid), then the mean over cameras.  splatfacto: rgb_weight = 1 - ssim_lambda = 0.8.
 *  SSIM = pytorch_msssim.SSIM(data_range=1, channel=3): 11x11 Gaussian window (sigma 1.5), valid convolution,
 *         mean over channels and pixels; ssim_lambda == 0 skips it (then workspace may be NULL).
 *  stats_dev[C*8] (double, per camera): {sum|rgb err|, sum|depth err|, n_valid, (scratch), max depth, sum SSIM map, (scratch), 0};
 *  loss_dev[3] float: {total, rgb term (L1 + SSIM), depth term}.  grad_scale multiplies every gradient
 *  (local_views / total_views for a view-sharded batch).  v_render / v_alphas are overwritten.
 */
size_t qed_loss_workspace_bytes(int C, int width, int height, float ssim_lambda);
int qed_loss_fwd_bwd(int C, int width, int height, const float* render, const float* alphas,
                     const void* gt_rgb, int gt_rgb_is_u8, const void* gt_depth, int gt_depth_is_u16, double depth_unit_scale,
                     const void* mask, int mask_is_u8, const float* bg, float rgb_weight,
                     float depth_lambda, float ssim_lambda, float grad_scale, double* stats_dev, float* loss_dev,
                     float* v_render, float* v_alphas, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* The same loss with splatfacto's bilateral grid (nerfstudio lib_bilagrid, per-image colour correction) applied to the
 * clamped composite of every view before the mask, L1 and SSIM.  The depth term is unchanged.
 *  grids[num_grids,12,L,Y,X] float32: per training image a 3x4 affine colour matrix A[i][j] = grid channel 4i+j.
 *  grid_ids[C] int32 in [0, num_grids): the grid of each view (the caller validates; an id outside the range gives NaN).
 *  Slice of pixel (row h, column w) with clamped colour c: x = w/(W-1), y = h/(H-1) (0 for an extent of 1),
 *  gray = 0.299 c0 + 0.587 c1 + 0.114 c2; lattice coordinates gx = x (X-1), gy = y (Y-1), gz = gray (L-1), each clamped
 *  to its axis, as grid_sample(mode="bilinear", align_corners=True, padding_mode="border") on [12, L, Y, X]; A = trilinear
 *  interpolation of the 8 neighbouring cells; out_i = sum_j A[i][j] c_j + A[i][3], not clamped.
 *  The gradient to render / alphas runs through out -> c, including the guidance term through gz (zero where gz is clamped).
 *  v_grid_rows[C,12,L,Y,X] (overwritten): d loss / d grid of each VIEW, i.e. before views sharing a grid are summed
 *  (qed_bilagrid_accumulate does that).  Deterministic: no atomics, the same inputs give the same bits.
 *  Supported: 2 <= X, Y <= 1024, 2 <= L <= 16 (QED_ERR_UNSUPPORTED otherwise).  workspace_bytes >=
 *  qed_loss_bilagrid_workspace_bytes (32 B/pixel of per-pixel records, plus the SSIM buffers when ssim_lambda > 0). */
size_t qed_loss_bilagrid_workspace_bytes(int C, int width, int height, float ssim_lambda);
int qed_loss_fwd_bwd_bilagrid(int C, int width, int height, const float* render, const float* alphas,
                              const void* gt_rgb, int gt_rgb_is_u8, const void* gt_depth, int gt_depth_is_u16, double depth_unit_scale,
                              const void* mask, int mask_is_u8, const float* bg, float rgb_weight,
                              float depth_lambda, float ssim_lambda, float grad_scale, double* stats_dev, float* loss_dev,
                              float* v_render, float* v_alphas, const float* grids, const int32_t* grid_ids, int num_grids,
                              int grid_X, int grid_Y, int grid_L, float* v_grid_rows, void* workspace, size_t workspace_bytes,
                              qed_stream_t stream);

/* Ground truth of a step rendered at 1/factor resolution (splatfacto's resolution schedule: `_downscale_if_required`, a
 * factor x factor box filter = conv2d with weights 1/factor^2 and stride factor, on the image, the depth and the mask).
 *  In: gt_rgb[C,height,width,3] float32 or (rgb_is_u8) uint8; gt_depth[C,height,width] float32 or (depth_is_u16) raw uint16;
 *  mask[C,height,width] float32 or (mask_is_u8) uint8 / bool, or NULL.  Values are converted as qed_loss_fwd_bwd converts
 *  them (u8 * (1.0f / 255.0f); float(double(u16) * depth_unit_scale); bool -> 0 / 1) BEFORE the filter.
 *  Out (float32, overwritten): out_rgb[C,h,w,3], out_depth[C,h,w] (metres), out_mask[C,h,w] (fractional; only when mask is
 *  not NULL), h = height / factor, w = width / factor rounded down (trailing rows / columns that fill no block are dropped).
 *  Each output = sum over its block, in row-major order starting from 0, of (1/factor^2) * x, individually rounded (no
 *  FMA).  NaN / inf propagate; zero (invalid) depth is averaged in, as the reference does.
 *  QED_ERR_BAD_ARG: C, width or height < 1, factor < 1, h or w == 0, a NULL input / output (out_mask when mask != NULL). */
int qed_downscale_ground_truth(int C, int width, int height, int factor, const void* gt_rgb, int rgb_is_u8, const void* gt_depth,
                               int depth_is_u16, double depth_unit_scale, const void* mask, int mask_is_u8, float* out_rgb,
                               float* out_depth, float* out_mask, qed_stream_t stream);

/* Held-out evaluation metrics of C rendered views (nerfstudio's eval: torchmetrics PSNR / SSIM, and qed-splatter's
 * DepthMetrics, metrics.py:115-156), forward only.
 *  render[C,height,width,4] (RGB + depth), alphas[C,height,width], gt_rgb / gt_depth / depth_unit_scale as for
 *  qed_loss_fwd_bwd (u8 * (1.0f / 255.0f); float(double(u16) * depth_unit_scale)), bg[3].
 *  Per view, with the prediction formed as qed_loss_fwd_bwd forms it: rgb = clamp(render.rgb + (1 - alpha) bg, 0, 1);
 *  depth = the depth channel where alpha > 0, else the view's maximum rendered depth.  metrics_dev[c * QED_EVAL_METRICS + k]
 *  (overwritten) holds, in this order:
 *    psnr = 10 log10(1 / rgb_mse) (+inf for a perfect image); ssim = the loss's SSIM (11x11 Gaussian window, sigma 1.5,
 *    valid windows, C1 = 1e-4, C2 = 9e-4, mean over channels and pixels, no mask); rgb_mse = mean over H*W*3 of
 *    (rgb - gt)^2; then, over the pixels whose ground-truth depth g is finite and > depth_tolerance, with d the predicted
 *    depth: abs_rel = mean |g - d| / g, sq_rel = mean (g - d)^2 / g, rmse = sqrt(mean (g - d)^2),
 *    rmse_log = sqrt(mean (log g - log d)^2), a1 / a2 / a3 = mean [max(g / d, d / g) < 1.25^k], and n_depth = their
 *    number.  With n_depth = 0 the seven depth values are NaN; non-finite values (d = 0) propagate.
 *  Sums in float64, per-block partials summed in a fixed order: the same inputs give the same bits, and a view's row does
 *  not depend on the other views.  workspace_bytes >= qed_eval_metrics_workspace_bytes (16-byte aligned).
 *  QED_ERR_UNSUPPORTED when width or height <= 10 (no valid SSIM window) or C > 21845. */
#define QED_EVAL_METRICS 11 /* psnr, ssim, rgb_mse, abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n_depth */
size_t qed_eval_metrics_workspace_bytes(int C, int width, int height);
int qed_eval_metrics(int C, int width, int height, const float* render, const float* alphas, const void* gt_rgb, int gt_rgb_is_u8,
                     const void* gt_depth, int gt_depth_is_u16, double depth_unit_scale, const float* bg, float depth_tolerance,
                     double* metrics_dev, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* Total-variation regulariser of the bilateral grids (splatfacto get_loss_dict while training):
 *  loss_out[1] = weight / G * sum_{axes d in L, Y, X} sum (x[.., i+1, ..] - x[.., i, ..])^2 / (elements of one grid's
 *  difference along d, i.e. 12 L Y X (n_d - 1) / n_d).  v_grids[G,12,L,Y,X] is OVERWRITTEN with its gradient;
 *  tv_per_grid[G] (double, overwritten) = each grid's unweighted sum of the per-axis means.  Fixed-order sums, no atomics.
 *  Shapes as for qed_loss_fwd_bwd_bilagrid. */
int qed_bilagrid_tv(int num_grids, int grid_X, int grid_Y, int grid_L, const float* grids, float weight, float* v_grids,
                    double* tv_per_grid, float* loss_out, qed_stream_t stream);
/* v_grids[grid_ids[r]] += v_grid_rows[r] for r = 0 .. n_rows-1 in row order, so rows sharing an id are summed
 * deterministically.  Rows whose id is outside [0, num_grids) are skipped. */
int qed_bilagrid_accumulate(int n_rows, const int32_t* grid_ids, const float* v_grid_rows, int num_grids, int grid_X, int grid_Y,
                            int grid_L, float* v_grids, qed_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * trainer-side kernels (SURVEY.md §8 rows a14, a16)
 */
/* Fused Adam (torch.optim.Adam semantics, no weight decay / amsgrad) over a flat arena: param/grad/m/v [n].
 * The arena is G <= 16 contiguous groups with end offsets group_ends[G] (device, int64); element i of group g
 * uses lr_by_group[g], or lr_alt_by_group[g] when group_period[g] > 0 and (i - start_g) % group_period[g] >=
 * group_split[g] (the SH block [N,16,3]: period 48, split 3 -> features_dc vs features_rest learning rates).
 * lr_alt_by_group / group_period / group_split may be NULL.  Bias corrections use `step` (1-based).
 * replaces: the six torch Adam groups of qed_splatter/config.py:44-68 with one launch. */
int qed_adam_arena(int64_t n, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int G,
                   const int64_t* group_ends, const float* lr_by_group, const float* lr_alt_by_group,
                   const int32_t* group_period, const int32_t* group_split, double beta1, double beta2, double eps,
                   int step, qed_stream_t stream);

/* gsplat DefaultStrategy._update_state on the `info` of model.py:267,289-292: for radii>0:
 *   grad2d[n] += ||g[c,n] * (W/2 * n_cameras, H/2 * n_cameras)||, count[n] += 1,
 *   radii_max[n] = max(radii_max[n], radii[c,n] / max(W,H)),   g = absgrad (or grad) slots of packed_grads.
 * n_cameras = size of the view batch the loss was averaged over (<= 0: C).  Accumulates. */
int qed_strategy_update(int C, int N, const float* packed_grads, int use_absgrad, const int32_t* radii,
                        int width, int height, int n_cameras, float* grad2d, float* count, float* radii_max,
                        qed_stream_t stream);

/* gsplat DefaultStrategy._grow_gs / _prune_gs data movement (ops.duplicate / ops.split / ops.remove + the optimizer-
 * state surgery) as ONE gather over the flat arenas (SURVEY.md section 8 row a15 / f3).  The caller decides, per
 * Gaussian of the NEW set, where it comes from; this builds the new parameter / exp_avg / exp_avg_sq arenas:
 *   src[j]        row of the old set that output j copies,
 *   fresh[j] != 0 its Adam moments start at zero (duplicates and split children), else they are copied,
 *   child_row[j]  >= 0: output j is a split child whose mean / log-scale come from child_means / child_scales[row]
 *                 (NULL or -1: copied from src like everything else).
 * Arena layout (old and new, for their own N): group-major  means 3N | quats 4N | log-scales 3N | logit-opacities N |
 * SH 48N, every group starting on a 16-byte boundary; old_group_starts / new_group_starts = the 5 group starts in
 * floats (HOST arrays).  The SH group start must be a multiple of 4 floats.  Padding floats are left untouched. */
int qed_arena_gather(int64_t n_new, const int32_t* src, const uint8_t* fresh, const int32_t* child_row,
                     const float* child_means, const float* child_scales, const float* old_param,
                     const float* old_exp_avg, const float* old_exp_avg_sq, const int64_t* old_group_starts,
                     float* new_param, float* new_exp_avg, float* new_exp_avg_sq, const int64_t* new_group_starts,
                     qed_stream_t stream);

/* Splatfacto's MCMC strategy (nerfstudio strategy="mcmc" -> gsplat MCMCStrategy) on the flat arenas above (group_starts:
 * HOST int64[5], the quats and SH starts multiples of 4 floats, param 16-byte aligned).  o = sigmoid(logit-opacity).
 * Random numbers: Philox4x32-10 (curand_Philox4x32_10) with key = seed and counter = (index, step, stream_id, 0).
 *
 * qed_mcmc_census: dead rows (o <= min_opacity, float32) -> dead_idx[0 .. n_dead) ascending, *n_dead_dev (device int64).
 * qed_mcmc_sample: weights w_i = floor(o_i * 2^24) (o in float64; 0 for dead rows when zero_dead), their exact int64
 *   inclusive scan, *total_dev = sum w.  Draw j (< n_draws, with replacement) = first row i with scan[i] > u_j, u_j =
 *   (64-bit Philox word (x << 32 | y) of counter (j, step, stream_id, 0) * total) >> 64; counts[N] = bincount(draws)
 *   (overwritten).  total == 0: draws untouched, counts zero.
 *   Both take workspace_bytes >= qed_mcmc_workspace_bytes(N) (16-byte aligned).
 * qed_mcmc_relocate: every row i with counts[i] > 0 gets gsplat compute_relocation at ratio min(counts[i] + 1, 51):
 *   o' = 1 - (1 - o)^(1/ratio) (then clamped to [min_opacity, 1 - FLT_EPSILON]), scale' = o / D(o', ratio) * scale with
 *   D(x, n) = sum_{j=1..n} C(n, j) (-1)^(j-1) x^j / sqrt(j) in float64; with zero_moments its exp_avg / exp_avg_sq rows
 *   are zeroed.  Then, after that, parameter row src[j] is copied to row dst[j] for j < n_copies (src and dst disjoint;
 *   the moments of dst are kept).  exp_avg / exp_avg_sq may be NULL without zero_moments.
 * qed_mcmc_noise: means += R diag(s)^2 R^T (n * sigmoid(100 ((1 - o) - 0.995)) * scaler) with n = three Box-Muller normals
 *   of counter (i, step, 0, 0), s = exp(log-scales), R of the normalised quaternion.
 * qed_mcmc_reg: loss[0] = opacity_reg * mean_N o, loss[1] = scale_reg * mean_3N exp(log-scale) (device floats); their
 *   gradients opacity_reg / N * o (1 - o) and scale_reg / (3 N) * exp(log-scale) are ADDED to grad (same layout).
 *   workspace_bytes >= qed_mcmc_reg_workspace_bytes(), zeroed before the first call (every call leaves it zeroed).
 *   Deterministic: fixed-order float64 sums. */
size_t qed_mcmc_workspace_bytes(int64_t N);
int qed_mcmc_census(int64_t N, const float* logit_opacities, float min_opacity, int32_t* dead_idx, int64_t* n_dead_dev, void* workspace,
                    size_t workspace_bytes, qed_stream_t stream);
int qed_mcmc_sample(int64_t N, const float* logit_opacities, float min_opacity, int zero_dead, int64_t n_draws, uint64_t seed, uint32_t step,
                    uint32_t stream_id, int32_t* draws, int32_t* counts, int64_t* total_dev, void* workspace, size_t workspace_bytes,
                    qed_stream_t stream);
int qed_mcmc_relocate(int64_t N, const int32_t* counts, float min_opacity, int zero_moments, int64_t n_copies, const int32_t* src,
                      const int32_t* dst, float* param, float* exp_avg, float* exp_avg_sq, const int64_t* group_starts, qed_stream_t stream);
int qed_mcmc_noise(int64_t N, float* param, const int64_t* group_starts, float scaler, uint64_t seed, uint32_t step, qed_stream_t stream);
size_t qed_mcmc_reg_workspace_bytes(void);
int qed_mcmc_reg(int64_t N, const float* param, const int64_t* group_starts, float opacity_reg, float scale_reg, float* grad, float* loss,
                 void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * camera + data side (SURVEY.md section 8 rows a1 and f4)
 */
/* qed_splatter/model.py:22-38 `get_viewmat`: nerfstudio camera-to-world [C, rows, 4] (rows = 3 or 4; OpenGL camera axes)
 * -> gsplat world-to-camera viewmats [C,4,4]: flip the y and z columns of R, analytic rigid inverse [R^T | -R^T T].
 * Called once per step by the model (model.py:246) on the optimised camera pose. */
int qed_viewmat_from_c2w(int C, int rows, const float* camera_to_worlds, float* viewmats, qed_stream_t stream);
/* Backward of qed_viewmat_from_c2w: v_viewmats [C,4,4] -> v_camera_to_worlds [C, rows, 4] (overwritten; row 3 of a 4-row
 * input gets zero, row 3 of v_viewmats is ignored).  With Rf = c2w[:3,:3] diag(1,-1,-1), T = c2w[:3,3]:
 * v_Rf = v_rot^T - T v_trans^T, v_T = -Rf v_trans, v_c2w[:3,:3] = v_Rf diag(1,-1,-1), v_c2w[:3,3] = v_T. */
int qed_viewmat_from_c2w_bwd(int C, int rows, const float* camera_to_worlds, const float* v_viewmats, float* v_camera_to_worlds,
                             qed_stream_t stream);

/* Splatfacto's camera optimizer in mode SO3xR3 (nerfstudio CameraOptimizer, applied at model.py:212/246).
 *  pose_adjustment[num_cameras,6] float32: per training camera {translation t (3), rotation log omega (3)}.
 *  camera_ids[C] int32 in [0, num_cameras): the table row of each view (the caller validates; an id outside the range
 *  gives a NaN viewmat and no gradient).  camera_to_worlds [C, rows, 4] as for qed_viewmat_from_c2w.
 *  theta^2 = max(|omega|^2, 1e-4), R = I + (sin theta / theta) [omega]x + ((1 - cos theta) / theta^2) [omega]x^2 (float64),
 *  c2w' = c2w[:3,:4] @ [[R, t], [0, 1]]  (R' = Rc R, t' = Rc t + tc; t is not rotated), viewmat = get_viewmat(c2w').
 * qed_camera_opt_apply: viewmats[C,4,4].  A view whose table row is zero gets exactly the bits of qed_viewmat_from_c2w.
 * qed_camera_opt_bwd: v_pose_adjustment[num_cameras,6] (overwritten; rows of no view get zero) = d loss / d table from
 *  v_viewmats[C,4,4], float64 inside; views sharing a camera id are summed in view order (no atomics, deterministic).
 * qed_camera_opt_reg: the regulariser of CameraOptimizer.get_loss_dict over all rows,
 *  reg_loss[1] (device) = trans_weight * mean_rows |t| + rot_weight * mean_rows |omega|; its gradient (zero at a zero
 *  norm) is ADDED to v_pose_adjustment.  One block, fixed-order float64 sums. */
int qed_camera_opt_apply(int C, int rows, int num_cameras, const int32_t* camera_ids, const float* camera_to_worlds,
                         const float* pose_adjustment, float* viewmats, qed_stream_t stream);
int qed_camera_opt_bwd(int C, int rows, int num_cameras, const int32_t* camera_ids, const float* camera_to_worlds,
                       const float* pose_adjustment, const float* v_viewmats, float* v_pose_adjustment, qed_stream_t stream);
int qed_camera_opt_reg(int num_cameras, const float* pose_adjustment, float trans_weight, float rot_weight, float* v_pose_adjustment,
                       float* reg_loss, qed_stream_t stream);

/* qed_splatter/create_init_pointcloud.py:148-196 `backproject_frame` (Open3D PointCloud.create_from_depth_image, :176-185):
 * depth [height,width] float32 or raw uint16 (depth_is_u16), metres = value * depth_unit_scale (float32 product, :165);
 * every `stride`-th pixel (u, v) with 0 < d < depth_max gives the world point inverse(extrinsic) * ((u-cx) d/fx, (v-cy) d/fy, d).
 * intrinsic_host [3,3] and extrinsic_host [4,4] (OpenCV world-to-camera, :59-70) are HOST arrays.  points [ceil(W/stride) *
 * ceil(H/stride), 3] receives the survivors compacted in pixel order, *n_points_dev (device) their count. */
size_t qed_backproject_workspace_bytes(int width, int height, int stride);
int qed_backproject_depth(int width, int height, const void* depth, int depth_is_u16, double depth_unit_scale, float depth_max,
                          int stride, const float* intrinsic_host, const float* extrinsic_host, float* points,
                          int64_t* n_points_dev, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* Open3D PointCloud.voxel_down_sample (create_init_pointcloud.py:89, :194, :260): points [n,3] binned by
 * floor(p / voxel_size); every occupied voxel yields the mean of its points.  Output sorted by voxel key (x, then y, then z
 * index), *n_out_dev (device) = number of voxels; points_out needs room for n rows.  n_dev (optional, device): only the
 * first min(*n_dev, n) points are real (the count qed_backproject_depth left on the device -- no host sync in between). */
size_t qed_voxel_downsample_workspace_bytes(int64_t n);
int qed_voxel_downsample(int64_t n, const int64_t* n_dev, const float* points, float voxel_size, float* points_out,
                         int64_t* n_out_dev, void* workspace, size_t workspace_bytes, qed_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * multi-GPU: sum of the gradient arena over the ranks of the view-sharded step (SURVEY.md section 8e; the reference has
 * no collective -- it renders one camera per step on one GPU, qed_splatter/model.py:211)
 *
 * The arena must live in SYMMETRIC memory: the same allocation on every rank, mapped into every peer process
 * (`peer_bases[r]` = address of rank r's arena in THIS process) and, when the box has NVSwitch multicast, into one
 * multicast address range (`multicast_base`, NULL = use the peer path).  `peer_flags[r]` = address of rank r's flag
 * block (qed_comm_flag_words() uint32, zero-initialised once, symmetric as well).  peer_bases / peer_flags are HOST
 * arrays of `world` device pointers.
 *
 * qed_comm_allreduce_f32: elements [begin, end) (multiples of 4) of every rank's arena are replaced by their sum over
 *   the ranks, in ONE kernel on `stream`: rank r sums the r-th part of the range -- inside the switch
 *   (multimem.ld_reduce) or from peer loads -- and broadcasts it (multimem.st / peer stores); epoch flags (release /
 *   acquire, system scope) order it against the other ranks' kernels, so no host synchronisation and no NCCL call is
 *   involved.  Every rank must call it with the same (begin, end, epoch) in the same order; `epoch` must grow by 2
 *   from call to call (it uses epoch and epoch + 1), starting at 1.  All replicas receive identical bits.
 *
 * View-colour exchange (what makes the per-step traffic small).  81 % of the arena is the SH coefficient gradient
 * [N,16,3], and d colour / d coeff[k,ch] = basis_k(direction): v_sh[n] = sum over views of basis(dir(n,view)) (x)
 * v_colour(n,view) -- rank-1 per view.  So instead of all-reducing 192 B per Gaussian:
 *   qed_project_bwd_exchange = qed_project_bwd (fused path: packed_grads in, v_means / v_quats / v_scales / v_opacities
 *     out, SH colours) that does NOT build the coefficient gradient; it stores the gated colour gradient
 *     {v_r, v_g, v_b, tag} of every VISIBLE (view, Gaussian) into slot (first_slot + c) * N + n of the exchange buffer of
 *     EVERY rank (one multimem.st through the switch, or peer stores), and its views' camera positions {x, y, z, tag}
 *     behind the slots (element total_slots * N + slot).  Exchange buffer = (total_slots * N + total_slots) float4,
 *     symmetric, zero-initialised once; `tag` must differ from step to step (records of Gaussians not visible this
 *     step stay stale and are recognised by their tag).  Callers alternate between two exchange buffers from step to
 *     step, so that a rank one step ahead never overwrites records a slower rank is still reading.
 *   qed_comm_allreduce_f32 over the 11 floats per Gaussian that are left (means, quats, scales, opacity), then
 *   qed_sh_grad_from_view_colors: every rank rebuilds v_sh[N,K,3] from ITS copy of the exchange buffer -- all views, in
 *     slot order, same bits everywhere -- after the all-reduce (whose entry barrier also orders the exchange).
 * Per GPU and step 16 B x visible (view, Gaussian) pairs + 44 B x N x (1 + 1/G) cross NVLink instead of 236 B x N x (1 + 1/G).
 */
int qed_project_bwd_exchange(int C, int N, const float* means, const float* quats, const float* scales,
                             const float* opacities, int activations, const float* sh_coeffs, int K, int sh_degree,
                             const float* viewmats, const float* Ks, int width, int height, float eps2d,
                             int calc_compensations, int append_depth, const int32_t* radii, const float* conics,
                             const float* compensations, const float* packed_grads, float* v_means, float* v_quats,
                             float* v_scales, float* v_opacities, float* exchange_multicast, float* const* exchange_peers,
                             int world, int first_slot, int total_slots, float tag, qed_stream_t stream);
/* qed_project_bwd_exchange that also returns the gradient with respect to this rank's C view poses, as qed_project_bwd_pose
 * does: v_viewmats[C,4,4] (overwritten, the rank's own views, not summed over ranks) and pose_ws / ws_bytes >=
 * qed_project_bwd_pose_workspace_bytes(C, N) (16-byte aligned; may be NULL when N == 0).  Deterministic. */
int qed_project_bwd_exchange_pose(int C, int N, const float* means, const float* quats, const float* scales,
                                  const float* opacities, int activations, const float* sh_coeffs, int K, int sh_degree,
                                  const float* viewmats, const float* Ks, int width, int height, float eps2d,
                                  int calc_compensations, int append_depth, const int32_t* radii, const float* conics,
                                  const float* compensations, const float* packed_grads, float* v_means, float* v_quats,
                                  float* v_scales, float* v_opacities, float* exchange_multicast, float* const* exchange_peers,
                                  int world, int first_slot, int total_slots, float tag, float* v_viewmats, void* pose_ws,
                                  size_t ws_bytes, qed_stream_t stream);
int qed_sh_grad_from_view_colors(int total_slots, int N, int K, int sh_degree, const float* means, const float* exchange_local,
                                 float tag, float* v_sh, qed_stream_t stream);
int qed_comm_flag_words(void);
/* All ranks' work enqueued before this call on their streams is complete and visible to every rank afterwards (one tiny
 * kernel, epoch flags as above; uses `epoch` only -- the caller's epoch counter grows by 1). */
int qed_comm_barrier(uint32_t* const* peer_flags, int rank, int world, uint32_t epoch, qed_stream_t stream);
int qed_comm_allreduce_f32(float* multicast_base, float* const* peer_bases, uint32_t* const* peer_flags, int rank, int world,
                           int64_t begin, int64_t end, uint32_t epoch, int blocks, qed_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* QED_SPLAT_H_ */
