/*
 * grendel_gs_b200.h -- C ABI of the B200-native (sm_100a) Gaussian rasterizer hot path.
 *
 * This is the drop-in boundary for the ONE path nyu-systems/Grendel-GS reaches through its
 * `diff_gaussian_rasterization` extension (SURVEY.md section 8b).  Every entry point names the
 * reference call site it replaces.  The reference binds these operators from Python, so the
 * reference-side stub is a ctypes binding: INTEGRATION.md shows it, and
 * grendel-gs_b200/diff_gaussian_rasterization/ is that binding, exporting the reference's own
 * names (GaussianRasterizationSettings, GaussianRasterizer, _C.get_local2j_ids_bool, ...).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless its name ends in _host;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing is
 *    synchronised unless stated;
 *  - tensors are dense row-major fp32 / int32 / uint8 exactly as the reference passes them;
 *  - return value 0 = success, otherwise a negative GS_E* code; gs_last_error() gives text;
 *  - the library owns no persistent device memory: callers pass every workspace (sizes from the
 *    gs_*_bytes queries), which keeps the operator re-entrant across the B rasterizer instances
 *    that coexist in one training step (gaussian_renderer/__init__.py:919-963).
 *  - gradient conventions (see oracle/gs_oracle.c:gso_preprocess_backward): dL_dmeans2D is per
 *    NDC unit (pixel gradient * (W/2, H/2)), which is what densification.py:24 reads from
 *    means2D.grad; dL_dconic_opacity holds true partials (dA, dB, dC, dOpacity).
 */
#ifndef GRENDEL_GS_B200_H
#define GRENDEL_GS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GS_OK 0
#define GS_EINVAL (-1)  /* bad argument */
#define GS_ECUDA (-2)   /* CUDA runtime error; see gs_last_error() */
#define GS_ENOMEM (-3)  /* workspace too small */

#define GS_BLOCK_X 16
#define GS_BLOCK_Y 16
#define GS_ONE_DIM_BLOCK_SIZE 256
#define GS_REC_FLOATS 12 /* packed per-splat record: 3 x float4 */

#if defined(__GNUC__)
#define GS_API __attribute__((visibility("default")))
#else
#define GS_API
#endif

/* Text of the last error raised on the calling thread. */
GS_API const char *gs_last_error(void);

/* Library / build identification, e.g. "grendel-gs_b200 sm_100a r1". */
GS_API const char *gs_version(void);

/* _C.get_block_XY()  -- /root/reference/arguments/__init__.py:254-257 */
GS_API int gs_get_block_xy(int *block_x, int *block_y, int *one_dim_block_size);

/* GaussianRasterizer.preprocess_gaussians forward (CUDA stage "10 preprocess")
 * -- /root/reference/gaussian_renderer/__init__.py:949-956.
 * means3D (P,3) scales (P,3, activated) rotations (P,4, normalised wxyz) opacities (P,1, activated)
 * shs (P,16,3); viewmatrix/projmatrix (4,4) in the reference's transposed storage
 * (scene/cameras.py:84-99); campos (3).
 * out: means2D (P,2) pixels, depths (P), radii (P) int32 (0 = culled), conic_opacity (P,4),
 * rgb (P,3), clamped (P) uint8 bit c = channel c clamped at 0.  All outputs are written for every
 * splat (zeros when culled); no pre-initialisation needed. */
GS_API int gs_preprocess_forward(int P, int sh_degree, const float *means3D, const float *scales, float scale_modifier,
                          const float *rotations, const float *opacities, const float *shs, const float *viewmatrix,
                          const float *projmatrix, const float *campos, int image_width, int image_height,
                          float tanfovx, float tanfovy, float *means2D, float *depths, int32_t *radii,
                          float *conic_opacity, float *rgb, uint8_t *clamped, void *stream);

/* autograd backward of preprocess_gaussians (CUDA stage "b20 preprocess")
 * -- /root/reference/train_internal.py:195 reaching gaussian_renderer/__init__.py:949-958.
 * All five gradient outputs are written for every splat (zeros when culled). */
GS_API int gs_preprocess_backward(int P, int sh_degree, const float *means3D, const float *scales, float scale_modifier,
                           const float *rotations, const float *shs, const float *viewmatrix, const float *projmatrix,
                           const float *campos, int image_width, int image_height, float tanfovx, float tanfovy,
                           const int32_t *radii, const uint8_t *clamped, const float *dL_dmeans2D,
                           const float *dL_dconic_opacity, const float *dL_drgb, float *dL_dmeans3D, float *dL_dscales,
                           float *dL_drotations, float *dL_dopacities, float *dL_dshs, void *stream);

/* Fused-activation variants (SURVEY.md 8f "next" #3): take the six RAW GaussianModel parameters
 * (/root/reference/scene/gaussian_model.py:219-228: _xyz (P,3), _features_dc (P,1,3), _features_rest (P,15,3),
 * _scaling (P,3) log, _rotation (P,4) unnormalised, _opacity (P,1) logit), apply the activations of
 * gaussian_model.py:109-129 (exp, normalize, sigmoid, cat) in registers, and return gradients for the raw
 * tensors.  They replace the five torch activation kernels + torch.cat of
 * gaussian_renderer/__init__.py:902-906 and their autograd backward. */
GS_API int gs_preprocess_forward_raw(int P, int sh_degree, const float *xyz, const float *features_dc,
                                     const float *features_rest, const float *scaling, float scale_modifier,
                                     const float *rotation, const float *opacity, const float *viewmatrix,
                                     const float *projmatrix, const float *campos, int image_width, int image_height,
                                     float tanfovx, float tanfovy, float *means2D, float *depths, int32_t *radii,
                                     float *conic_opacity, float *rgb, uint8_t *clamped, void *stream);
GS_API int gs_preprocess_backward_raw(int P, int sh_degree, const float *xyz, const float *features_dc,
                                      const float *features_rest, const float *scaling, float scale_modifier,
                                      const float *rotation, const float *opacity, const float *viewmatrix,
                                      const float *projmatrix, const float *campos, int image_width, int image_height,
                                      float tanfovx, float tanfovy, const int32_t *radii, const uint8_t *clamped,
                                      const float *dL_dmeans2D, const float *dL_dconic_opacity, const float *dL_drgb,
                                      float *dL_dxyz, float *dL_dfeatures_dc, float *dL_dfeatures_rest,
                                      float *dL_dscaling, float *dL_drotation, float *dL_dopacity, void *stream);

/* Batched fused-activation variants: ALL B cameras of a step (gaussian_renderer/__init__.py:919-963 loops over them
 * in Python) in one launch; each Gaussian's parameters are read once and projected into every camera, and the
 * backward accumulates the B cameras' contributions before writing each parameter gradient once.
 * cams: (B,40) floats per camera = viewmatrix[16], projmatrix[16], campos[3], tanfovx, tanfovy, 3 pad; all cameras
 * share image_width/height.  Outputs are (B,P,...) with camera k's slice identical to the single-camera result. */
GS_API int gs_preprocess_forward_batched(int B, int P, int sh_degree, const float *xyz, const float *features_dc,
                                         const float *features_rest, const float *scaling, float scale_modifier,
                                         const float *rotation, const float *opacity, const float *cams,
                                         int image_width, int image_height, float *means2D, float *depths,
                                         int32_t *radii, float *conic_opacity, float *rgb, uint8_t *clamped,
                                         void *stream);
GS_API int gs_preprocess_backward_batched(int B, int P, int sh_degree, const float *xyz, const float *features_dc,
                                          const float *features_rest, const float *scaling, float scale_modifier,
                                          const float *rotation, const float *opacity, const float *cams,
                                          int image_width, int image_height, const int32_t *radii,
                                          const uint8_t *clamped, const float *dL_dmeans2D,
                                          const float *dL_dconic_opacity, const float *dL_drgb, float *dL_dxyz,
                                          float *dL_dfeatures_dc, float *dL_dfeatures_rest, float *dL_dscaling,
                                          float *dL_drotation, float *dL_dopacity, void *stream);

/* _C.get_local2j_ids_bool -- /root/reference/gaussian_renderer/workload_division.py:721-744.
 * strategy: (world_size+1) int32 ascending flattened tile ids; out: (P, world_size) uint8/bool. */
GS_API int gs_get_local2j_ids_bool(int P, int image_height, int image_width, int world_size, const float *means2D,
                            const int32_t *radii, const int32_t *strategy, uint8_t *out, void *stream);

/* _C.get_local2j_ids_bool_adjust_mode6 -- workload_division.py:471-484 (legacy).
 * rects: (world_size,4) int32 tile rectangles (y_l, y_r, x_l, x_r). */
GS_API int gs_get_local2j_ids_bool_rects(int P, int image_height, int image_width, int world_size, const float *means2D,
                                  const int32_t *radii, const int32_t *rects, uint8_t *out, void *stream);

/* ---- GaussianRasterizer.render_gaussians -- gaussian_renderer/__init__.py:1271-1282 -------------
 * Three calls because the number R of (splat, local tile) instances is data dependent:
 *   gs_render_count   stages 21-24 + 30: per-splat LOCAL tile count, depth order of the splats, inclusive scan,
 *                     packed records
 *   gs_render_forward stages 40,50,60,70,81-83: duplicate-with-keys, radix sort, tile ranges, blend
 *   gs_render_backward stage b10
 * The sorted instance list is the one the published 64-bit sort (key = tile << 32 | fp32 depth bits, stable)
 * produces; it is obtained as a stable 32-bit depth sort of the P splats followed by a stable sort of the R
 * instances on their tile bits only (see csrc/binning.cu).
 */

/* Bytes of scratch gs_render_count needs for P splats. */
GS_API size_t gs_render_count_temp_bytes(int P);

/* compute_locally: (TILE_Y*TILE_X) uint8/bool mask (workload_division.py:773-787).
 * order: (P) uint32 splat indices in ascending depth (splats without a local tile last).
 * offsets: (P) uint32 inclusive prefix sum of local tiles touched, IN THAT ORDER.
 * rec: (P, GS_REC_FLOATS) packed per-splat records consumed by the blend kernels.
 * R_host: HOST pointer; receives the instance count.  This call synchronises `stream`. */
GS_API int gs_render_count(int P, int image_height, int image_width, const float *means2D, const float *conic_opacity,
                           const float *rgb, const float *depths, const int32_t *radii, const uint8_t *compute_locally,
                           uint32_t *order, uint32_t *offsets, float *rec, void *temp, size_t temp_bytes,
                           int64_t *R_host, void *stream);

/* Bytes of radix-sort scratch for R instances. */
GS_API size_t gs_render_sort_temp_bytes(int64_t R);

/* Bytes of the segment workspace that links a forward to its backward (R instances, num_tiles = tiles of all views):
 * the forward leaves a per-pixel checkpoint every 64 entries of a tile list plus the list of (tile, segment) units,
 * which lets gs_render_backward walk every segment independently (csrc/blend.cu, k_blend_bwd_seg).  No reference
 * counterpart: the published backward re-walks each tile list as a whole (cuda_rasterizer/backward.cu). */
GS_API size_t gs_render_seg_bytes(int64_t R, int num_tiles);

/* tiles_unsorted/tiles_sorted: (R) uint32 tile ids; ids_unsorted/ids_sorted: (R) uint32 splat ids.
 * ranges: (T,2) uint32 [start,end) per tile.  bg: (3).  image: (3,H,W) -- written in full: non-local
 * tiles are exactly 0 (loss_distribution.py:1875).  final_T (H,W) f32 and n_contrib (H,W) uint32 are
 * kept for the backward.  stats: optional (3) int64 sums of n_render / n_consider / n_contrib, or NULL.
 * seg_ws: gs_render_seg_bytes(R, T) bytes, 256-byte aligned, kept for the backward; NULL for a forward-only render
 * (mode "test", gaussian_renderer/__init__.py:524: no checkpoints are written; the image is bit-identical). */
GS_API int gs_render_forward(int P, int64_t R, int image_height, int image_width, const float *means2D,
                             const int32_t *radii, const uint8_t *compute_locally, const uint32_t *order,
                             const uint32_t *offsets, const float *rec, const float *bg, uint32_t *tiles_unsorted,
                             uint32_t *ids_unsorted, uint32_t *tiles_sorted, uint32_t *ids_sorted, void *sort_temp,
                             size_t sort_temp_bytes, uint32_t *ranges, float *image, float *final_T,
                             uint32_t *n_contrib, int64_t *stats, void *seg_ws, size_t seg_ws_bytes, void *stream);

/* dL_dimage: (3,H,W).  The three gradient outputs (P,2) (P,4) (P,3) are zero-filled and
 * accumulated by this call.  seg_ws: the workspace the forward filled (segment-parallel kernel), or NULL (tile-parallel
 * kernel of round 1: one CTA per tile; same results up to summation order). */
GS_API int gs_render_backward(int P, int64_t R, int image_height, int image_width, const float *rec, const float *bg,
                       const uint8_t *compute_locally, const uint32_t *ranges, const uint32_t *ids_sorted,
                       const float *final_T, const uint32_t *n_contrib, const float *dL_dimage, const void *seg_ws,
                       size_t seg_ws_bytes, float *dL_dmeans2D, float *dL_dconic_opacity, float *dL_drgb, void *stream);

/* ---- the same three calls for ALL cameras of a training batch at once --------------------------------------
 * The reference loops over the B cameras of a batch and calls render_gaussians once per camera
 * (render_final, gaussian_renderer/__init__.py:1217-1288, called at train_internal.py:178); with the pixels of every camera cut into
 * W strips each of those calls works on 1/W of an image, so at W = 8 a rank issues 8 x ~12 small launches and waits
 * 8 times for an instance count.  These entry points bin and blend the strips of all B cameras in ONE pass:
 *   - the splats of the B cameras are concatenated: camera v owns rows [view_start[v], view_start[v+1]) of
 *     means2D / conic_opacity / rgb / depths / radii (view_start: HOST int32[num_views+1], view_start[0] = 0);
 *   - compute_locally is (B, TILE_Y*TILE_X), ranges (B*T, 2), the sort key is v*T + tile;
 *   - image (B,3,H,W), final_T (B,H,W), n_contrib (B,H,W), stats (B,3) or NULL, dL_dimage (B,3,H,W);
 *   - order / offsets / rec / ids index the concatenated splat rows, the gradients are (P,2) (P,4) (P,3) with
 *     P = view_start[num_views].
 * Per camera the result is bit-identical to the single-camera call (same instance order within every tile).
 * num_views <= GS_MAX_VIEWS; scratch sizes are those of the single-camera calls with P and R totals. */
#define GS_MAX_VIEWS 64
GS_API int gs_render_count_batched(int num_views, const int32_t *view_start_host, int image_height, int image_width,
                                   const float *means2D, const float *conic_opacity, const float *rgb,
                                   const float *depths, const int32_t *radii, const uint8_t *compute_locally,
                                   uint32_t *order, uint32_t *offsets, float *rec, void *temp, size_t temp_bytes,
                                   int64_t *R_host, void *stream);
/* The count in two halves.  gs_render_count_launch enqueues stages 21-24 + 30 (view_start_host = NULL, P = number of splats:
 * the single-camera form; otherwise P is ignored and the total is view_start_host[num_views]) and hands back a ticket;
 * gs_render_count_read blocks until the instance total -- complete after the FIRST kernel -- has reached the host and
 * returns it, while the depth sort and the scan are still running: the caller sizes its buffers and enqueues
 * gs_render_forward behind them, so the stream does not run dry behind the operator's one host sync
 * (the reference syncs on num_rendered the same way; gaussian_renderer/__init__.py:1271-1282).  At most 64 tickets may be
 * outstanding.  gs_render_count / gs_render_count_batched = launch + read. */
GS_API int gs_render_count_launch(int num_views, const int32_t *view_start_host, int P, int image_height, int image_width,
                                  const float *means2D, const float *conic_opacity, const float *rgb, const float *depths,
                                  const int32_t *radii, const uint8_t *compute_locally, uint32_t *order, uint32_t *offsets,
                                  float *rec, void *temp, size_t temp_bytes, void **ticket, void *stream);
GS_API int gs_render_count_read(void *ticket, int64_t *R_host, void *stream);
GS_API int gs_render_forward_batched(int num_views, const int32_t *view_start_host, int64_t R, int image_height,
                                     int image_width, const float *means2D, const int32_t *radii,
                                     const uint8_t *compute_locally, const uint32_t *order, const uint32_t *offsets,
                                     const float *rec, const float *bg, uint32_t *tiles_unsorted, uint32_t *ids_unsorted,
                                     uint32_t *tiles_sorted, uint32_t *ids_sorted, void *sort_temp,
                                     size_t sort_temp_bytes, uint32_t *ranges, float *image, float *final_T,
                                     uint32_t *n_contrib, int64_t *stats, void *seg_ws, size_t seg_ws_bytes,
                                     void *stream);
GS_API int gs_render_backward_batched(int num_views, int P, int64_t R, int image_height, int image_width,
                                      const float *rec, const float *bg, const uint8_t *compute_locally,
                                      const uint32_t *ranges, const uint32_t *ids_sorted, const float *final_T,
                                      const uint32_t *n_contrib, const float *dL_dimage, const void *seg_ws,
                                      size_t seg_ws_bytes, float *dL_dmeans2D, float *dL_dconic_opacity, float *dL_drgb,
                                      void *stream);

/* ---- per-kernel device timing ------------------------------------------------------------------
 * The reference's fork logs per-stage GPU times under --zhx_time ("10 preprocess time: 0.29 ms", ...;
 * /root/reference/analyze_statistic.py:1972-1991).  When enabled, every launch site brackets its
 * kernel(s) with CUDA events on the launching stream; gs_profile_read synchronises those events and
 * returns the accumulated milliseconds and launch count of one stage, then resets it. */
enum {
    GS_STAGE_PREPROCESS_FWD = 0, /* "10 preprocess" */
    GS_STAGE_COUNT_TILES,        /* "21-24 updateDistributedStatLocally" */
    GS_STAGE_SCAN,               /* "30 InclusiveSum" */
    GS_STAGE_DUPLICATE,          /* "40 duplicateWithKeys" */
    GS_STAGE_SORT,               /* "50 SortPairs" */
    GS_STAGE_RANGES,             /* "60 identifyTileRanges" */
    GS_STAGE_BLEND_FWD,          /* "70 render" */
    GS_STAGE_BLEND_BWD,          /* "b10 render" */
    GS_STAGE_PREPROCESS_BWD,     /* "b20 preprocess" */
    GS_STAGE_LOSS_FWD,
    GS_STAGE_LOSS_BWD,
    GS_STAGE_LOCAL2J,
    GS_STAGE_PACK,
    GS_STAGE_UNPACK,
    GS_STAGE_NUM
};
GS_API int gs_profile_enable(int on);
GS_API int gs_profile_read(int stage, double *total_ms, int64_t *launches);
GS_API const char *gs_profile_stage_name(int stage);

/* ---- test-only switches (no reference counterpart) ------------------------------------------------
 * The blend kernels skip 4x4 / 8x4 pixel blocks a splat cannot reach with alpha >= 1/255, using per-splat
 * extents computed in gs_render_count.  That cull must be CONSERVATIVE: it may never drop a contribution the
 * reference (which tests alpha per pixel, cuda_rasterizer/forward.cu:513-519) would have blended.
 * GS_DEBUG_NO_BLOCK_CULL makes gs_render_count write infinite extents, so tests can check that the culled and
 * unculled kernels produce the same image and n_contrib.  Returns the previous flags. */
enum {
    GS_DEBUG_NO_BLOCK_CULL = 1,
    /* gs_render_backward: use the tile-parallel kernel of round 1 (one CTA per tile, k_blend_bwd) even when a segment
     * workspace is passed -- A/B timing and cross-checking of the two backward kernels. */
    GS_DEBUG_BWD_TILE = 2,
    /* gs_render_forward: the half-warp-per-4x4-block blend kernel of round 1 (k_blend_fwd) instead of the packed
     * two-pixels-per-lane kernel (k_blend_fwd2); the images are bit-identical. */
    GS_DEBUG_FWD_HALFWARP = 4,
    /* direct exchange: pack with a CTA-level compaction per destination (one row per thread, 200-400-byte NVLink spans)
     * instead of per-warp stores; same rows, same bytes (A/B switch until it is measured at 8 ranks) */
    GS_DEBUG_XR_PACK_CTA = 8,
    /* gs_render_backward with a segment workspace: round 2's segment-parallel kernel (k_blend_bwd_seg, one reduction and
     * RED set per splat) instead of round 3's (k_blend_bwd_seg3: compacted passes, packed sums, reduction tail shared by
     * two splats); the same sums, reduced in a different order.  GS_DEBUG_BWD_TILE takes precedence. */
    GS_DEBUG_BWD_SEG_R2 = 16
};
GS_API int gs_debug_set(int flags);

/* ---- per-strip loss -- gaussian_renderer/loss_distribution.py:2536-2585 + utils/loss_utils.py:88-132 ----
 * image: (3,H,W) full-size render of which rows [row0,row1) are this rank's strip;
 * gt_u8: (3,row1-row0,W) uint8 ground-truth strip (camera.original_image of loss_distribution.py:2561).
 * out_l1_ssim: (2) float = { sum|x-y| , sum ssim_map } / (3*H*W)  -- the Ll1 and ssim_loss of :2571,2576.
 * temp (gs_loss_temp_bytes) keeps three derivative maps for the backward.
 * backward: dL_dimage (3,H,W) = grad_l1[0]*dLl1/dimage + grad_ssim[0]*dssim/dimage, with grad_* DEVICE
 * scalars (the autograd upstream gradients; no host sync); rows outside the strip are written 0.
 * [count_row0,count_row1) within [row0,row1) are the rows whose pixels are SUMMED; the other rows of the window only
 * feed the 11x11 SSIM windows of their neighbours -- the live path passes count = window (zero padding at strip edges),
 * the border-pixel exchange of loss_distribution.py:601-972 passes a window widened by the 5 halo rows received from the
 * neighbouring strips, which makes the sum of the strip losses equal the full-image loss. */
GS_API size_t gs_loss_temp_bytes(int rows, int image_width);
GS_API int gs_loss_forward(int image_height, int image_width, int row0, int row1, int count_row0, int count_row1,
                           const float *image, const uint8_t *gt_u8, float *out_l1_ssim, void *temp, size_t temp_bytes,
                           void *stream);
GS_API int gs_loss_backward(int image_height, int image_width, int row0, int row1, int count_row0, int count_row1,
                            const float *image, const uint8_t *gt_u8, const void *temp, const float *grad_l1,
                            const float *grad_ssim, float *dL_dimage, void *stream);

/* The strip losses of all B cameras of a batch in one launch (the reference loops batched_loss over the cameras,
 * loss_distribution.py:2588-2640).  rows4_host: HOST int32 (B,4) = row0, row1, count_row0, count_row1 per camera
 * (row1 == row0: this rank renders no strip of that camera; its outputs are 0).  image / dL_dimage: (B,3,H,W);
 * gt_u8_ptrs_host: HOST array of B device pointers to the (3,rows,W) uint8 strips; out_l1_ssim: (B,2);
 * grad_l1 / grad_ssim: DEVICE (B).  Per camera the numbers are those of the single-camera calls. */
GS_API size_t gs_loss_temp_bytes_batched(int num_views, const int32_t *rows4_host, int image_width);
GS_API int gs_loss_forward_batched(int num_views, int image_height, int image_width, const int32_t *rows4_host,
                                   const float *image, const void *const *gt_u8_ptrs_host, float *out_l1_ssim,
                                   void *temp, size_t temp_bytes, void *stream);
GS_API int gs_loss_backward_batched(int num_views, int image_height, int image_width, const int32_t *rows4_host,
                                    const float *image, const void *const *gt_u8_ptrs_host, const void *temp,
                                    const float *grad_l1, const float *grad_ssim, float *dL_dimage, void *stream);

/* ---- held-out evaluation -- train_internal.py:466-479, render.py:120-138 -> metrics.py:26-36 ----------------
 * Forward-only image metrics of B views in one launch: the loss forward's 11x11 window without derivative maps.  Per
 * view v and channel c, over the counted rows [count_row0, count_row1) of the window [row0, row1) (rows4_host as in
 * gs_loss_forward_batched; row1 == row0: the view's sums are 0), out_sums (B,3,3) fp64 is OVERWRITTEN with
 *   out_sums[v][0][c] = sum |x - y|,  out_sums[v][1][c] = sum (x - y)^2,  out_sums[v][2][c] = sum ssim_map(x, y)
 * where y = gt_u8 / 255 and x = clamp(image, 0, 1) (saved_mode 0: training_report, utils/image_utils.py:19-21) or,
 * saved_mode 1, that value after torchvision.utils.save_image's 8-bit quantisation and to_tensor's read-back,
 * uint8(min(255, x * 255 + 0.5)) / 255 with the multiply and add rounded separately (render.py:127-138).
 * images: (B,3,H,W); gt_u8_host_array: HOST array of B device pointers to the (3, row1-row0, W) uint8 windows.
 * Every per-pixel term is added in fp64: a view split into strips with 5-row halos sums to its whole-image value. */
GS_API int gs_metrics_batched(int num_views, int image_height, int image_width, const int32_t *rows4_host,
                              const float *images, const uint8_t *const *gt_u8_host_array, int saved_mode,
                              double *out_sums, void *stream);

/* ---- all-to-all staging -- gaussian_renderer/__init__.py:590-607,651-658 --------------------------
 * Replaces the per-(destination, camera) nonzero() + index_select + torch.cat glue around the sparse
 * all-to-all: rows of 11 floats forward (means2D 2, rgb 3, conic_opacity 4, radius as float, depth), 9 floats
 * backward.  gs_route_scan is the building block: exclusive ranks of the flagged entries of a (P, ncols) byte mask
 * taken in column-major order (gpos, ncols*P) and the per-column starts (colstart, ncols+1); ncols <= 16. */
GS_API size_t gs_route_scan_temp_bytes(int P, int ncols);
GS_API int gs_route_scan(int P, int ncols, const uint8_t *mask, int32_t *gpos, int32_t *colstart, void *temp,
                         size_t temp_bytes, void *stream);

/* Exchange of ALL B cameras of a step, one launch per stage (B, W <= 16; B*W <= 128 non-empty (source, camera) segments).
 * Flags / scan positions are laid out [destination rank j][camera k][splat i] -- the all_to_all_single send layout --
 * so gpos IS the row index in the send buffer.  *_ptrs_host are HOST arrays of B device pointers (one per camera);
 * row_lo/row_hi_host are HOST (B*W) tile-row ranges [lo,hi) of camera k owned by global rank j (row strips of
 * workload_division.py:852-941).  counts: (W*B) int32 device, [j][k]. */
GS_API size_t gs_xchg_temp_bytes(int B, int P, int W);
GS_API int gs_xchg_route(int B, int P, int W, int image_height, int image_width, const void *const *means2D_ptrs_host,
                         const void *const *radii_ptrs_host, const int32_t *row_lo_host, const int32_t *row_hi_host,
                         uint8_t *flags, int32_t *gpos, int32_t *counts, void *temp, size_t temp_bytes, void *stream);
GS_API int gs_xchg_pack(int B, int P, int W, const uint8_t *flags, const int32_t *gpos,
                        const void *const *means2D_ptrs_host, const void *const *rgb_ptrs_host,
                        const void *const *conic_opacity_ptrs_host, const void *const *radii_ptrs_host,
                        const void *const *depths_ptrs_host, float *send_rows, void *stream);
GS_API int gs_xchg_unpack(int nseg, const int32_t *seg_recv_start_host, const int32_t *seg_len_host,
                          const int32_t *seg_cam_host, const int32_t *seg_dst_start_host, int total_rows,
                          const float *recv_rows, int B, void *const *means2D_ptrs_host, void *const *rgb_ptrs_host,
                          void *const *conic_opacity_ptrs_host, void *const *radii_ptrs_host,
                          void *const *depths_ptrs_host, void *stream);
GS_API int gs_xchg_pack_grad(int nseg, const int32_t *seg_recv_start_host, const int32_t *seg_len_host,
                             const int32_t *seg_cam_host, const int32_t *seg_dst_start_host, int total_rows, int B,
                             const void *const *d_means2D_ptrs_host, const void *const *d_rgb_ptrs_host,
                             const void *const *d_conic_opacity_ptrs_host, float *grad_rows, void *stream);
GS_API int gs_xchg_scatter_grad(int B, int P, int W, const uint8_t *flags, const int32_t *gpos, const float *grad_rows,
                                void *const *d_means2D_ptrs_host, void *const *d_rgb_ptrs_host,
                                void *const *d_conic_opacity_ptrs_host, void *stream);

/* ---- the same exchange over NVLink peer memory: pack + transfer fused in one kernel -----------------------------
 * Replaces torch.distributed.all_to_all_single (gaussian_renderer/__init__.py:609-628 forward, its autograd mirror
 * backward) for ranks of one NVLink/NVSwitch node.  Each rank owns one receive buffer (11-float rows) and one
 * gradient buffer (9-float rows), allocated by gs_peer_alloc and exported as a 64-byte CUDA IPC handle; peers map
 * them with gs_peer_open.  gs_xchg_pack_p2p stores every row directly into its final row of the destination's
 * receive buffer (the row all_to_all_single would have delivered it to), gs_xchg_pack_grad_p2p stores every gradient
 * row directly into the row of the source's gradient buffer that gs_xchg_scatter_grad reads.  The caller orders
 * producers and consumers across ranks (a 4-byte all-reduce enqueued after the kernel; see csrc/distribute.cu). */
GS_API int gs_peer_alloc(size_t bytes, void **dev_ptr, void *ipc_handle_64);
GS_API int gs_peer_open(const void *ipc_handle_64, void **peer_ptr);
GS_API int gs_peer_close(void *peer_ptr);
GS_API int gs_peer_free(void *dev_ptr);
/* dst_rows_ptrs_host: HOST array of W pointers, rank j's receive buffer as mapped in this process (own buffer for
 * j == me); row_delta_host: HOST (W) = recv_base_j[me] - send_base_me[j]. */
GS_API int gs_xchg_pack_p2p(int B, int P, int W, const uint8_t *flags, const int32_t *gpos,
                            const void *const *means2D_ptrs_host, const void *const *rgb_ptrs_host,
                            const void *const *conic_opacity_ptrs_host, const void *const *radii_ptrs_host,
                            const void *const *depths_ptrs_host, void *const *dst_rows_ptrs_host,
                            const int32_t *row_delta_host, void *stream);
/* seg_dst_ptrs_host: HOST array of nseg pointers, the first gradient row of segment q inside the SOURCE rank's
 * gradient buffer (as mapped in this process). */
GS_API int gs_xchg_pack_grad_p2p(int nseg, const int32_t *seg_recv_start_host, const int32_t *seg_len_host,
                                 const int32_t *seg_cam_host, const int32_t *seg_dst_start_host, int total_rows, int B,
                                 const void *const *d_means2D_ptrs_host, const void *const *d_rgb_ptrs_host,
                                 const void *const *d_conic_opacity_ptrs_host, void *const *seg_dst_ptrs_host,
                                 void *stream);

/* gs_xr_pack with the destination rows computed on the device from the all-gathered counts (counts_all_dev: W*B*W int32,
 * [source][camera][destination]; row0_dev: W*B + 1 int32 scratch = rows + over-capacity flag): enqueued right behind the
 * all-gather of gaussian_renderer/__init__.py:609-628's sizes, before the host has read them -- the stream does not run
 * dry at the exchange's host sync.  Over capacity nothing is written and every rank takes the all_to_all_single path. */
GS_API int gs_xr_pack_dev(int B, int P, int W, int image_height, int image_width, const void *const *means2D_ptrs_host,
                          const void *const *rgb_ptrs_host, const void *const *conic_opacity_ptrs_host,
                          const void *const *radii_ptrs_host, const void *const *depths_ptrs_host,
                          const int32_t *row_lo_host, const int32_t *row_hi_host, const int32_t *blkbase,
                          void *const *peer_recv_ptrs_host, const int32_t *counts_all_dev, int me, int32_t *row0_dev,
                          long long cap_rows, void *stream);
/* ---- direct-placement exchange (csrc/distribute.cu, "xr"): same collective, same row order, but nothing is staged --
 * gs_xr_count: per (destination rank j, camera k, block of 256 splats) hit counts + their exclusive scan + the (j,k)
 * totals (the counts every rank all-gathers, gaussian_renderer/__init__.py:574-588).
 * gs_xr_pack: every splat is stored field by field into its FINAL row of the destination rank's structure-of-arrays
 * receive region (means2D | rgb | conic_opacity | radii | depths, cap_rows rows each; gs_peer_alloc'ed, 11*cap floats),
 * i.e. straight into the tensors that rank's render reads -- no send rows, no unpack (replaces :590-607 and :631-658).
 * gs_xr_pull_grad: the mirrored backward; the owner of a splat loads its gradient rows from the gradient regions
 * (d means2D (2) | d rgb padded to 4 floats per row | d conic_opacity (4): 10*cap floats) of the ranks it sent the
 * splat to and sums them.
 * row_lo/row_hi: (B*W) HOST ints as in gs_xchg_route; dst_row0_host[j*B+k]: first row of the calling rank's block inside
 * camera k of rank j's arrays (from the all-gathered counts).  The caller orders pack -> consumers and the gradient
 * writers -> pull across ranks (a stream-ordered barrier). */
GS_API size_t gs_xr_temp_bytes(int B, int P, int W);
GS_API int gs_xr_count(int B, int P, int W, int image_height, int image_width, const void *const *means2D_ptrs_host,
                       const void *const *radii_ptrs_host, const int32_t *row_lo_host, const int32_t *row_hi_host,
                       int32_t *blkcnt, int32_t *blkbase, int32_t *counts, void *temp, size_t temp_bytes, void *stream);
GS_API int gs_xr_pack(int B, int P, int W, int image_height, int image_width, const void *const *means2D_ptrs_host,
                      const void *const *rgb_ptrs_host, const void *const *conic_opacity_ptrs_host,
                      const void *const *radii_ptrs_host, const void *const *depths_ptrs_host,
                      const int32_t *row_lo_host, const int32_t *row_hi_host, const int32_t *blkbase,
                      void *const *peer_recv_ptrs_host, const int32_t *dst_row0_host, long long cap_rows, void *stream);
GS_API int gs_xr_pull_grad(int B, int P, int W, int image_height, int image_width, const void *const *means2D_ptrs_host,
                           const void *const *radii_ptrs_host, const int32_t *row_lo_host, const int32_t *row_hi_host,
                           const int32_t *blkbase, void *const *peer_grad_ptrs_host, const int32_t *dst_row0_host,
                           long long cap_rows, void *const *d_means2D_ptrs_host, void *const *d_rgb_ptrs_host,
                           void *const *d_conic_opacity_ptrs_host, void *stream);

/* ---- sparse per-Gaussian gradient all-reduce staging (replicated Gaussians) ----------------------------------
 * /root/reference/scene/gaussian_model.py:1332-1391 (get_sparse_ids, sync_gradients_sparsely) and the
 * "fused_sparse" mode it leaves NotImplemented (:1438-1439).  mask[i] = _xyz.grad row i is non-zero; after an
 * all-reduce(MAX) of the mask and gs_route_scan(ncols = 1), pack writes one 59-float row per touched Gaussian
 * (xyz 3, features_dc 3, features_rest 45, scaling 3, rotation 4, opacity 1) for ONE all-reduce(SUM); unpack
 * scatters the sums back.  grads_host: HOST array of the six device gradient pointers in that order. */
GS_API int gs_sparse_grad_mask(int P, const float *xyz_grad, uint8_t *mask, void *stream);
GS_API int gs_sparse_grad_pack(int P, const uint8_t *mask, const int32_t *pos, void *const *grads_host, float *rows,
                               void *stream);
GS_API int gs_sparse_grad_unpack(int P, const uint8_t *mask, const int32_t *pos, const float *rows,
                                 void *const *grads_host, void *stream);

/* ---- fused Adam step (SURVEY.md 8f rank 3) -- /root/reference/train_internal.py:316-329 ---------------------------
 * torch.optim.Adam(l, lr=0.0, eps=1e-15) over the six parameter groups (scene/gaussian_model.py:257-292), preceded by
 * `param.grad /= args.bsz` (train_internal.py:319-324): one launch for up to GS_ADAM_MAX_TENSORS tensors with
 * per-tensor lr / betas / eps, torch's arithmetic and operation order (no weight decay, no amsgrad).
 * All *_host are HOST arrays of num_tensors entries; pointers are fp32 contiguous device tensors of numel[k] elements
 * (NULL grad: tensor skipped, like .grad is None).  step[k] >= 1: the step counter AFTER this update.
 * grad_scale multiplies every gradient first (1/bsz).  params, exp_avg, exp_avg_sq are updated in place. */
#define GS_ADAM_MAX_TENSORS 8
GS_API int gs_adam_step(int num_tensors, const int64_t *numel_host, void *const *params_host,
                        const void *const *grads_host, void *const *exp_avg_host, void *const *exp_avg_sq_host,
                        const double *lr_host, const double *beta1_host, const double *beta2_host,
                        const double *eps_host, const int64_t *step_host, float grad_scale, void *stream);

/* ---- densification step (SURVEY.md 8f rank 4) -- /root/reference/scene/gaussian_model.py:1005-1044 ------------------
 * densify_and_prune = densify_and_clone (:973-1003) + densify_and_split (:922-971) + prune_points (:816-835) over the
 * six parameters and both Adam moments (cat_tensors_to_optimizer :837-881, _prune_optimizer :789-814), ~150 torch
 * kernels and a dozen host read-backs in the reference.  Here: gs_densify_select computes every Gaussian's decisions
 * and ONE scan that yields the output row of every survivor / clone / split child (order of the reference's end state:
 * survivors, clones, children copy 1, children copy 2; each in index order) and reads six counts back;
 * gs_densify_gather then writes every tensor once (moments of new Gaussians zero, children: position
 * R(q)(s * z) + x from caller-provided standard-normal draws z, log-scale log(s / 1.6)).
 * counts_host: HOST int32[6] = kept, clones, children copy 1, children copy 2, S (split-selected; the split reads
 * 2 S rows of noise), new number of Gaussians.  scaling_raw / opacity_raw / rotation_raw are the raw parameters
 * (log-scale, logit, unnormalised quaternion).  Written after round 1's device budget was spent: NOT yet run on a GPU. */
GS_API size_t gs_densify_temp_bytes(int P);
GS_API int gs_densify_select(int P, const float *xyz_gradient_accum, const float *denom, const float *scaling_raw,
                             const float *opacity_raw, float max_grad, float min_opacity, float extent,
                             float percent_dense, int use_screen_size, void *temp, size_t temp_bytes,
                             int32_t *counts_host, void *stream);
/* src_host / dst_host: HOST arrays of num_tensors (<= 24) device pointers to (P, width) inputs / (new_P, width) outputs of
 * 4-byte elements; kind_host: 0 copy, 1 position (width 3), 2 log-scale (width 3), 3 Adam moment. */
GS_API int gs_densify_gather(int P, int S, int new_P, int num_tensors, const void *const *src_host, void *const *dst_host,
                             const int32_t *width_host, const int32_t *kind_host, const float *scaling_raw,
                             const float *rotation_raw, const float *noise, const void *temp, void *stream);

/* ---- simple_knn._C.distCUDA2 -- /root/reference/scene/gaussian_model.py:20,163-166 ------------------------------------
 * Mean squared distance of every point to its 3 nearest OTHER points (self excluded by index, duplicates count at
 * distance 0; fewer than 3 other points: the mean of those that exist), the start-up scale initialisation.  Exact, by
 * tiled brute force (init-time only).  points (N,3) fp32 -> mean_dist2 (N) fp32.  NOT yet run on a device. */
GS_API int gs_knn3_mean_dist2(int N, const float *points, float *mean_dist2, void *stream);

/* ---- legacy tile-mask / tile-exchange helpers (SURVEY.md 8a rows L3-L4; dead code in the shipped trainer) ------
 * _C.get_touched_locally                     -- gaussian_renderer/loss_distribution.py:136-141
 * _C.get_pixels_compute_locally_and_in_rect  -- loss_distribution.py:205-213
 * load_image_tiles_by_pos / merge_image_tiles_by_pos (forward of one is the adjoint of the other)
 *                                            -- loss_distribution.py:168-175, 188-195
 * masks are uint8/bool; pos is (n,2) int64 GLOBAL tile (y,x); image_rect is (3,rect_h,rect_w) whose pixel (0,0) is
 * image pixel (rect_min_y, rect_min_x); tiles is (n,3,16,16). */
GS_API int gs_get_touched_locally(int tile_y, int tile_x, int extension_distance, const uint8_t *compute_locally,
                                  uint8_t *out, void *stream);
GS_API int gs_get_pixels_compute_locally_and_in_rect(int image_height, int image_width, const uint8_t *compute_locally,
                                                     int min_y, int max_y, int min_x, int max_x, uint8_t *out,
                                                     void *stream);
GS_API int gs_image_tiles_gather(int n, const int64_t *pos, const float *image_rect, int rect_h, int rect_w,
                                 int rect_min_y, int rect_min_x, int image_height, int image_width, float *tiles,
                                 void *stream);
GS_API int gs_image_tiles_scatter_add(int n, const int64_t *pos, const float *tiles, int rect_h, int rect_w,
                                      int rect_min_y, int rect_min_x, int image_height, int image_width,
                                      float *image_rect, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GRENDEL_GS_B200_H */
