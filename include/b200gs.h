/*
 * b200gs — C ABI of the sm_100a differentiable 3D-Gaussian rasterizer (libb200gs.so).
 *
 * This is the drop-in boundary for the hot path of yzslab/gaussian-splatting-lightning.  The reference has no
 * native code of its own: its renderers call two pip extensions through Python, and these entry points are what a
 * binding for those call sites needs (citations relative to /root/reference):
 *
 *   diff_gaussian_rasterization.GaussianRasterizer(...)(means3D, means2D, shs, colors_precomp, opacities, scales,
 *       rotations, cov3D_precomp) -> (color, radii)            internal/renderers/vanilla_renderer.py:62-77,111-120
 *   gsplat.v0_interfaces.project_gaussians(...) -> 7-tuple     internal/renderers/gsplat_renderer.py:64-79
 *   gsplat.sh.spherical_harmonics(deg, dirs, coeffs)           internal/renderers/gsplat_renderer.py:105
 *   gsplat.rasterize.rasterize_gaussians(...) -> [H,W,D](,alpha)  internal/renderers/gsplat_renderer.py:86-99
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named host_*; all floating point is fp32, contiguous.
 *   - the library never allocates or frees device memory: the caller (PyTorch's caching allocator) owns every
 *     buffer including the workspace -> no hidden cudaMalloc, no hidden synchronisation (except where stated).
 *   - all work is enqueued on the cudaStream_t passed as `stream` (a CUstream handle; pass
 *     torch.cuda.current_stream().cuda_stream).
 *   - return 0 on success, a negative B200GS_E* code on failure; b200gs_last_error() gives a thread-local message.
 *     Nothing throws across the ABI; nothing calls exit().  Re-entrant: no global mutable state.
 *   - "mode": B200GS_MODE_VANILLA = diff-gaussian-rasterization semantics (near 0.2, mean2D via the NDC projection
 *     matrix, pixel sample at integer coords, alpha clamp 0.99 straight-through, stop T<1e-4, rect max uses +15);
 *     B200GS_MODE_GSPLAT = the semantics of internal/utils/gaussian_projection.py + gsplat's rasterizer (near 0.01,
 *     K t/(z+1e-6), blur compensation, pixel centres +0.5, alpha clamp 0.999 as a true clamp, stop T<=1e-4,
 *     rect max = int((p+r)/16)+1).
 */
#ifndef B200GS_H
#define B200GS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B200GS_API __attribute__((visibility("default")))
#else
#define B200GS_API
#endif

#define B200GS_MODE_VANILLA 0
#define B200GS_MODE_GSPLAT 1

#define B200GS_OK 0
#define B200GS_EINVAL (-1)    /* bad argument (null pointer, bad size, unsupported degree/channels) */
#define B200GS_ECUDA (-2)     /* a CUDA call or launch failed; message holds cudaGetErrorString */
#define B200GS_ENOSPACE (-3)  /* workspace or pair capacity too small */

#define B200GS_TILE 16

/* One view.  Matrices are stored exactly as the reference's Camera stores them (cameras.py:147-189):
 * viewmatrix = world_to_camera, "transposed" (row-major [4][4], translation in the last ROW; p_cam = p * M[:3,:3] + M[3,:3]);
 * projmatrix = full_projection = world_to_camera @ projection (same layout; vanilla mode only). */
typedef struct B200gsView {
    int32_t width;
    int32_t height;
    int32_t mode;           /* B200GS_MODE_* */
    int32_t sh_degree;      /* active degree 0..4 */
    int32_t sh_stride;      /* coefficients stored per Gaussian (K of shs[N,K,3]); >= (sh_degree+1)^2 */
    int32_t reserved0;
    float fx, fy, cx, cy;   /* gsplat mode intrinsics (gsplat_renderer.py:70-73) */
    float tanfovx, tanfovy; /* vanilla mode (vanilla_renderer.py:59-60) */
    float scale_modifier;
    float eps2d;            /* 2D low-pass added to the cov2D diagonal: 0.3 */
    float near_plane;       /* <=0 selects the mode default (0.2 vanilla / 0.01 gsplat) */
    float reserved1;
    float viewmatrix[16];
    float projmatrix[16];
    float campos[3];
    float reserved2;
} B200gsView;

B200GS_API const char* b200gs_last_error(void);
B200GS_API int b200gs_version(void);
/* number of CUDA kernels this library has launched in this process (monotonic; every launch site increments it) */
B200GS_API int64_t b200gs_launch_count(void);

/* ---- K1: per-Gaussian projection (+ optional fused SH colour) ------------------------------------------------
 * replaces dgr preprocessCUDA / gsplat project_gaussians (+ spherical_harmonics when shs != NULL).
 * in : means[n,3] scales[n,3] quats[n,4] (wxyz, used as given); shs[n,sh_stride,3] or NULL.
 * out: xy[n,2] depth[n] radii[n] conic[n,3] tiles[n]; comp[n] (gsplat, nullable); cov3d[n,6] upper triangle (nullable);
 *      rgb[n,3] = max(SH+0.5,0) and clamped[n] (bit c set when channel c was clamped) when shs != NULL.
 *      Culled Gaussians get zeros everywhere (radii 0, tiles 0).
 * SH view direction: normalize(mean - campos).  */
B200GS_API int b200gs_project_fwd(const B200gsView* view, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, float* xy, float* depth, int32_t* radii, float* conic, float* comp,
                       int32_t* tiles, float* cov3d, float* rgb, uint8_t* clamped, void* stream);

/* ---- K8: backward of K1 ------------------------------------------------------------------------------------------
 * in : the K1 inputs, radii (visibility), clamped (when shs), and cotangents v_xy[n,2] (vanilla: dgr's NDC-scaled
 *      dL/dmean2D, i.e. pixel gradient x (0.5W, 0.5H); gsplat: pixel units), v_depth[n] (nullable), v_conic[n,3] (true
 *      partials of power = -(A dx^2 + C dy^2)/2 - B dx dy), v_comp[n] (nullable), v_rgb[n,3] (nullable unless shs).
 * out: v_means[n,3] v_scales[n,3] v_quats[n,4] and v_shs[n,sh_stride,3] (when shs) — fully written (zeros for culled).
 * vanilla mode back-propagates the SH view direction into v_means; gsplat mode does not (renderers detach it). */
B200GS_API int b200gs_project_bwd(const B200gsView* view, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, const int32_t* radii, const uint8_t* clamped, const float* v_xy,
                       const float* v_depth, const float* v_conic, const float* v_comp, const float* v_rgb,
                       float* v_means, float* v_scales, float* v_quats, float* v_shs, void* stream);

/* ---- K1 / K8 with the model's activations fused ("raw parameter" fast path) -------------------------------------------
 * Same kernels, reading the RAW parameter tensors of VanillaGaussianModel (internal/models/vanilla_gaussian.py:66,345-358;
 * internal/models/gaussian.py:250-254) instead of its getters: scales = exp(log_scales), quats = normalize(raw_quats),
 * opacity = sigmoid(opacity_logits) (all evaluated inside the kernel, the geometry part in fp64), SH = shs_dc[n,1,3] |
 * shs_rest[n,sh_stride-1,3] read in place (no torch.cat).  Removes 5 elementwise kernels + the 192 B/Gaussian
 * concatenation and their autograd backward from every training step.
 * fwd extra out: opacity_out[n] = the opacity the blend kernels consume (x compensation in gsplat mode when
 *     anti_aliased != 0; gsplat_renderer.py:81-83).
 * The matching K8 is b200gs_project_bwd_rows (below): gradients w.r.t. the RAW tensors, cotangents from gradient rows. */
B200GS_API int b200gs_project_fwd_raw(const B200gsView* view, int64_t n, const float* means, const float* log_scales,
                           const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                           int32_t anti_aliased, float* xy, float* depth, int32_t* radii, float* conic, float* comp,
                           int32_t* tiles, float* rgb, uint8_t* clamped, float* opacity_out, void* stream);

/* ---- per-Gaussian passes next to the renderer in a training step (SURVEY §8f rank 4) ---------------------------------------
 * b200gs_selective_adam: visibility-masked Adam step of one [rows, width] parameter tensor (gsplat.optimizers.SelectiveAdam /
 *     diff-accel SparseGaussianAdam, internal/optimizers.py:26-90): for the rows with visible[row] != 0
 *     m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= lr m / (sqrt(v) + eps)   (no bias correction, like those kernels);
 *     rows that did not take part in the view keep parameter and moments untouched.
 * b200gs_densify_stats: VanillaDensityControllerImpl.update_states (vanilla_density_controller.py:101-123) in one pass: on the
 *     visible rows (visible[n] bytes, or radii > 0 when NULL) max_radii2d = max(max_radii2d, radii), grad_accum += |grad[:, :2] *
 *     (scale_x, scale_y)|, denom += 1.  grad has grad_stride floats per row (2 for gsplat xys, 3 for dgr's screenspace points). */
B200GS_API int b200gs_selective_adam(int64_t rows, int32_t width, float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                                     const uint8_t* visible, float lr, float beta1, float beta2, float eps, void* stream);
B200GS_API int b200gs_densify_stats(int64_t n, const int32_t* radii, const uint8_t* visible, const float* grad, int32_t grad_stride,
                                    float scale_x, float scale_y, float* max_radii2d, float* grad_accum, float* denom, void* stream);

/* b200gs_knn_mean_dist2: simple_knn's distCUDA2 (vanilla_gaussian.py:122-125, the scale initialiser): mean_dist2[i] = mean of the squared
 *     distances from points[i] (float[n,3]) to its 3 nearest neighbours (exact).  Synchronises the stream once (the hash grid is sized
 *     on the host from the bounding box); init-time only. */
B200GS_API size_t b200gs_knn_workspace_bytes(int64_t n);
B200GS_API int b200gs_knn_mean_dist2(int64_t n, const float* points, float* mean_dist2, void* workspace, size_t workspace_bytes, void* stream);

/* ---- standalone SH (gsplat.sh.spherical_harmonics; gsplat_renderer.py:105) -------------------------------------------
 * dirs[n,3] need not be unit (normalised inside, as gsplat does).  out rgb[n,3] = SH (no +0.5, no clamp).
 * bwd: v_coeffs[n,sh_stride,3] fully written; v_dirs[n,3] nullable. */
B200GS_API int b200gs_sh_fwd(int32_t degree, int32_t sh_stride, int64_t n, const float* dirs, const float* coeffs, float* rgb, void* stream);
B200GS_API int b200gs_sh_bwd(int32_t degree, int32_t sh_stride, int64_t n, const float* dirs, const float* coeffs, const float* v_rgb,
                  float* v_coeffs, float* v_dirs, void* stream);

/* ---- K2-K5: tile binning ------------------------------------------------------------------------------------------
 * replaces dgr InclusiveSum + duplicateWithKeys + SortPairs + identifyTileRanges / gsplat isect_tiles + isect_offset_encode.
 * Result order is exactly that of a stable sort of (tile_id << 32 | float_bits(depth)) keys emitted Gaussian-major:
 * implemented as a stable depth sort of the visible Gaussians, a stable partition of (coarse cell, Gaussian) pairs (a
 * cell = 8x8 tiles) and an order-preserving multi-split of every cell's list into its 64 tiles that writes each id
 * once.  Both sorts are hand-written onesweep-style radix passes (decoupled look-back); no library sort is involved.
 *
 * Counters: d_counts = device int64[4], host_counts = host int64[4] (pinned or pageable; nullable):
 *     [0] number of (tile, Gaussian) pairs of the 3-sigma bounding rects — the reference's pair count, an upper bound
 *         of [2] and equal to it without culling                                              (written by phase A)
 *     [1] number of (coarse cell, Gaussian) pairs                                              (written by phase A)
 *     [2] number of pairs actually listed in sorted_ids / tile_ranges                          (written by phase B)
 *     [3] number of visible Gaussians (non-empty tile rect)                                    (written by phase A)
 *   Each phase ends by delivering d_counts to host_counts (when != NULL) in stream order — pinned/mapped host memory is
 *   written by a tiny kernel with system-scope stores (a D2H copy would queue on a copy engine behind the application's
 *   bulk transfers), pageable memory by cudaMemcpyAsync — and, when sync_host != 0, SYNCHRONISES the stream.
 *   Sync-free use: size max_coarse from the previous view's counts[1] and max_pairs from its counts[0] (the bound is known
 *   after phase A already), pass sync_host = 0, record an event after phase A and check
 *   counts[1] <= max_coarse && counts[0] <= max_pairs once the rest of the forward has been enqueued.
 * cull_conic[n,3] / cull_opacity[n] (both NULL, or both given): exact tile culling.  A (tile, Gaussian) pair is dropped
 *     when no pixel sample of the tile can reach alpha >= 1/255 for that Gaussian (minimum of the conic's quadratic
 *     over the tile box > ln(255*opacity)); the blend loop would have skipped it at every pixel, so images and
 *     gradients do not change while the pair list shrinks ~2x.  With NULL the pair list is exactly the reference's
 *     (every tile of the 3-sigma bounding rect).
 * b200gs_bin_count_workspace_bytes / b200gs_bin_sort_workspace_bytes: bytes of scratch for phase A (n Gaussians) and
 *     phase B (up to max_coarse coarse pairs).  Two buffers because counts[1] is only known after phase A.
 * b200gs_bin_count: phase A.  Compaction of the visible Gaussians, depth keys, stable depth sort; counts[0], [1], [3].  Everything
 *     phase B needs to know about a Gaussian (xy, radius, cull_conic, cull_opacity) is packed into workspace_a, which
 *     must stay untouched until phase B has been enqueued.
 * b200gs_bin_sort: phase B (reads workspace_a only; cull = whether phase A was given the cull arrays).  Writes sorted_ids (Gaussian ids, front to back inside each tile; capacity max_pairs),
 *     tile_ranges[n_tiles,2] (int32 [start,end), clamped to max_pairs) and counts[2].  Coarse pairs beyond max_coarse
 *     and ids beyond max_pairs are DROPPED (never written out of bounds): the caller compares the counters with the
 *     capacities and redoes the phase with larger buffers if either overflowed.  max_pairs = counts[0] and
 *     max_coarse = counts[1] can never overflow. */
B200GS_API size_t b200gs_bin_count_workspace_bytes(int64_t n);
B200GS_API size_t b200gs_bin_sort_workspace_bytes(int64_t n, int64_t max_coarse, int32_t width, int32_t height);
B200GS_API int b200gs_bin_count(int32_t mode, int32_t width, int32_t height, int64_t n, const float* xy, const float* depth,
                     const int32_t* radii, const float* cull_conic, const float* cull_opacity, void* workspace_a, size_t workspace_a_bytes,
                     int64_t* d_counts, int64_t* host_counts, int32_t sync_host, void* stream);
B200GS_API int b200gs_bin_sort(int32_t mode, int32_t width, int32_t height, int64_t n, int32_t cull, int64_t max_coarse, int64_t max_pairs,
                    int64_t* d_counts, const void* workspace_a, void* workspace_b, size_t workspace_b_bytes, int32_t* sorted_ids,
                    int32_t* tile_ranges, int64_t* host_counts, int32_t sync_host, void* stream);

/* b200gs_publish_i64: deliver n device int64 counters to host memory in stream order, the way the binning phases do
 *     (kernel with system-scope stores for pinned/mapped memory, cudaMemcpyAsync for pageable): for callers that run their
 *     own sync-free capacity protocol (the sharded renderer's row exchange). */
B200GS_API int b200gs_publish_i64(const int64_t* d_values, int64_t* host_values, int32_t n, void* stream);

/* ---- K6: blend forward ---------------------------------------------------------------------------------------------
 * replaces dgr renderCUDA fwd / gsplat rasterize_to_pixels fwd.  channels in {1,2,3,4}.
 * in : xy[n,2] conic[n,3] opacity[n] colors[n,channels]; bg[channels] or NULL.
 * out: image, addressed as image[pixel*pix_stride + channel*ch_stride] (vanilla [C,H,W]: pix_stride 1, ch_stride H*W;
 *      gsplat [H,W,C]: pix_stride C, ch_stride 1); final_T[H*W]; n_contrib[H*W] (1-based position in the tile's list of
 *      the last contributing splat); alpha[H*W] = 1 - final_T (nullable). */
B200GS_API int b200gs_blend_fwd(int32_t mode, int32_t width, int32_t height, int32_t channels, const int32_t* tile_ranges,
                     const int32_t* sorted_ids, const float* xy, const float* conic, const float* opacity,
                     const float* colors, const float* bg, float* image, int64_t pix_stride, int64_t ch_stride,
                     float* final_T, int32_t* n_contrib, float* alpha, void* stream);
/* b200gs_blend_fwd_hits: the same, and hit_any[g] = 1 for every splat g that contributed to at least one pixel (caller zero-fills
 *     hit_any[n]): gsplat's `means2d.has_hit_any_pixels` (optimizers.py:39 SelectiveAdam; gsplat_v1_renderer.py:287 acc_vis). */
B200GS_API int b200gs_blend_fwd_hits(int32_t mode, int32_t width, int32_t height, int32_t channels, const int32_t* tile_ranges,
                     const int32_t* sorted_ids, const float* xy, const float* conic, const float* opacity,
                     const float* colors, const float* bg, float* image, int64_t pix_stride, int64_t ch_stride,
                     float* final_T, int32_t* n_contrib, float* alpha, uint8_t* hit_any, void* stream);

/* ---- K7: blend backward --------------------------------------------------------------------------------------------
 * replaces dgr renderCUDA bwd / gsplat rasterize_to_pixels bwd.
 * in : forward inputs + final_T, n_contrib + v_image (same addressing as image) + v_alpha[H*W] (nullable).
 * out (ACCUMULATED with atomics — caller zero-fills): v_xy[n,2] (pixel units x (xy_scale_x, xy_scale_y)),
 *      v_conic[n,3], v_opacity[n], v_colors[n,channels]; v_xy_abs[n,2] (nullable; sum of |pixel grad|, gsplat absgrad). */
B200GS_API int b200gs_blend_bwd(int32_t mode, int32_t width, int32_t height, int32_t channels, const int32_t* tile_ranges,
                     const int32_t* sorted_ids, const float* xy, const float* conic, const float* opacity,
                     const float* colors, const float* bg, const float* final_T, const int32_t* n_contrib,
                     const float* v_image, int64_t pix_stride, int64_t ch_stride, const float* v_alpha,
                     float xy_scale_x, float xy_scale_y, float* v_xy, float* v_conic, float* v_opacity,
                     float* v_colors, float* v_xy_abs, void* stream);

/* ---- fused L1 + SSIM training loss on the rendered image (validated on B200: tests/test_gpu_loss.py) -------------------------
 * replaces  loss = (1-lambda) * l1_loss(image, gt) + lambda * (1 - ssim(image, gt))   (internal/metrics/vanilla_metrics.py:57-74,
 * internal/utils/ssim.py:17-63: 11-tap Gaussian window sigma 1.5, zero padding, C1 = 0.01^2, C2 = 0.03^2).  image/target [C,H,W].
 * b200gs_loss_fwd: partials[b200gs_loss_blocks(...)][2] <- per-CTA sums of |image-target| and of the SSIM map (the caller sums them
 *     and divides by C*H*W); dmaps[3][C][H][W] <- partial derivatives of the SSIM map, kept for the backward.
 * b200gs_loss_bwd: v_image[C,H,W] <- (*v_loss or 1) * dloss/dimage. */
B200GS_API int64_t b200gs_loss_blocks(int32_t channels, int32_t width, int32_t height);
B200GS_API int b200gs_loss_fwd(int32_t channels, int32_t width, int32_t height, const float* image, const float* target, float* dmaps,
                               float* partials, void* stream);
B200GS_API int b200gs_loss_bwd(int32_t channels, int32_t width, int32_t height, const float* image, const float* target, const float* dmaps,
                               float lambda_dssim, const float* v_loss, float* v_image, void* stream);

/* ---- [n,12] splat rows: the exchange format of the Gaussian-sharded multi-GPU renderer ------------------------------
 * replaces the packing / splitting around the reference's all-to-all of projected splats
 * (internal/renderers/gsplat_distributed_renderer.py:127-217): one fp32 row per VISIBLE Gaussian,
 *   col 0-1 xy | 2 depth | 3-5 conic | 6 compensation | 7 opacity | 8-10 rgb | 11 radius (int32 bit pattern).
 * b200gs_pack_rows: compacts the visible (radii > 0) entries of K1's outputs into rows, in index order; row_index[n] (int32)
 *     = the row of entry i, kept for the backward.  segment_cap == 0: one dense block, d_count[0] <- number of rows.
 *     segment_cap > 0: entries [j*segment_len, (j+1)*segment_len) (one camera = one destination rank) fill the fixed-size
 *     block rows[j*segment_cap, (j+1)*segment_cap) — the all-to-all then needs no size exchange (no host sync); unused
 *     rows are zero (radius 0: ignored by the binning that reads them in place); entries that do not fit are DROPPED
 *     (row_index -1) and d_count[j] <- visible entries of segment j, for the caller to compare with segment_cap.
 * b200gs_bin_count_rows (then b200gs_bin_sort) / blend_fwd_rows / blend_bwd_rows: K2-K7 reading the rows IN PLACE (strided
 *     access, no split copies); blend_bwd_rows accumulates into a zero-filled [n,12] gradient row buffer that goes
 *     straight back through the all-to-all.  3 colour channels; cull != 0 enables exact tile culling. */
#define B200GS_MAX_VIEWS 8      /* cameras per multi-view launch (one NVSwitch box) */
#define B200GS_ROW_FLOATS 12
#define B200GS_ROW_XY 0
#define B200GS_ROW_DEPTH 2
#define B200GS_ROW_CONIC 3
#define B200GS_ROW_COMP 6
#define B200GS_ROW_OPACITY 7
#define B200GS_ROW_RGB 8
#define B200GS_ROW_RADIUS 11
/* b200gs_project_fwd_rows: K1 (fused activations, either constant set) writing ONE [n,12] row per Gaussian instead of the separate
 *     arrays — the single-GPU renderers' fast path: K2-K7 read the rows in place (b200gs_bin_count_rows, b200gs_blend_fwd_rows,
 *     b200gs_blend_bwd_rows), K8 reads the gradient rows (b200gs_project_bwd_rows with row_offsets = NULL).  Rows of culled
 *     Gaussians have radius 0, zeros in columns 0..3 and 8..10 (columns 4..7 unspecified).  radii[n], clamped[n] (what K8 needs) are written too; tiles may be NULL. */
B200GS_API int b200gs_project_fwd_rows(const B200gsView* view, int64_t n, const float* means, const float* log_scales,
                                       const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                       int32_t anti_aliased, float* rows, int32_t* radii, uint8_t* clamped, int32_t* tiles, void* stream);
/* b200gs_project_bwd_rows: K8 (fused activations) taking its cotangents straight from compacted [V,12] gradient rows
 *     (v_rows[row_offsets[i]] for visible i; row_offsets = NULL: v_rows[i]) and, when accumulate != 0, ADDING to the gradient buffers — the sharded
 *     renderer calls it once per camera of the step without unpack copies or separate sum kernels.
 *     v_mean2d (optional, may be NULL): [n, v_mean2d_cols] (2 or 3 columns) <- dL/dmean2D of every Gaussian (columns 0..1 of its gradient row; zeros
 *     for culled Gaussians and in column 2): the `.grad` of the renderer contract's `viewspace_points` (vanilla_renderer.py:55-56,
 *     vanilla_density_controller.py:101-123), written here instead of by a fill + strided copy after the kernel. */
B200GS_API int b200gs_project_bwd_rows(const B200gsView* view, int64_t n, const float* means, const float* log_scales,
                                       const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                       int32_t anti_aliased, const int32_t* radii, const uint8_t* clamped, const int32_t* row_offsets,
                                       const float* v_rows, int32_t accumulate, float* v_means, float* v_log_scales, float* v_raw_quats,
                                       float* v_opacity_logits, float* v_shs_dc, float* v_shs_rest, float* v_mean2d, int32_t v_mean2d_cols,
                                       void* stream);
/* b200gs_project_fwd_raw_multi / b200gs_project_bwd_rows_multi: K1 / K8 of one shard for ALL n_views (<= B200GS_MAX_VIEWS) cameras of a
 *     step in one launch each (gsplat constants, raw parameters; sh_degree / sh_stride / scale_modifier of views[0] apply to all).
 *     fwd: camera-major outputs, view j at elements [j*n, (j+1)*n); parameters and SH blocks are read once per Gaussian.
 *     bwd: every thread accumulates its Gaussian's gradients over the cameras in registers and writes them once; cotangents are
 *     [.,12] gradient rows, entry (j, i) reads row row_index[j*n+i] of v_rows[j] — a HOST array of n_views device pointers, each
 *     of which may address a peer GPU's buffer (the camera owner's gradient rows are pulled over NVLink, no return all-to-all). */
B200GS_API int b200gs_project_fwd_raw_multi(const B200gsView* views, int32_t n_views, int64_t n, const float* means, const float* log_scales,
                                            const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                            int32_t anti_aliased, float* xy, float* depth, int32_t* radii, float* conic, float* rgb,
                                            uint8_t* clamped, float* opacity_out, void* stream);
/* b200gs_project_pack_multi: K1 of one shard for all n_views cameras FUSED with the packing of the exchange.  The visible splats of
 *     camera j leave the kernel as [.,12] rows, in Gaussian-index order, stored straight into dst_rows[j] (a HOST array of n_views device
 *     pointers: block of block_rows rows in the receive buffer of the rank that owns camera j — peer memory over NVLink — or in a local
 *     send buffer); rows past block_rows are dropped.  d_count[j] = visible splats of camera j (compare with block_rows).  Kept locally
 *     for K8 and the renderer contract, camera-major ([j*n + i]): xy (mean2D), radii, clamped, row_index (j*block_rows + k, -1 = dropped).
 *     Replaces b200gs_project_fwd_raw_multi + b200gs_pack_rows (gsplat_distributed_renderer.py:127-217: project, then all-to-all). */
B200GS_API size_t b200gs_project_pack_workspace_bytes(int32_t n_views, int64_t n);
B200GS_API int b200gs_project_pack_multi(const B200gsView* views, int32_t n_views, int64_t n, const float* means, const float* log_scales,
                                         const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                         int32_t anti_aliased, float* xy, int32_t* radii, uint8_t* clamped, int32_t* row_index,
                                         void* const* dst_rows, int64_t block_rows, void* workspace, size_t workspace_bytes,
                                         int64_t* d_count, void* stream);
B200GS_API int b200gs_project_bwd_rows_multi(const B200gsView* views, int32_t n_views, int64_t n, const float* means, const float* log_scales,
                                             const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                             int32_t anti_aliased, const int32_t* radii, const uint8_t* clamped, const int32_t* row_index,
                                             const float* const* v_rows, float* v_means, float* v_log_scales, float* v_raw_quats,
                                             float* v_opacity_logits, float* v_shs_dc, float* v_shs_rest, void* stream);
/* b200gs_ipc_alloc / _handle / _open / _close / _free: device buffers that peer processes of the same box can map (cudaMalloc +
 *     CUDA IPC): the exchange buffers of the sharded renderer.  handle = 64 bytes to pass to the peers by any host channel. */
B200GS_API int b200gs_ipc_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64);
B200GS_API int b200gs_ipc_open(const unsigned char* handle64, void** dev_ptr);
B200GS_API int b200gs_ipc_close(void* dev_ptr);
B200GS_API int b200gs_ipc_free(void* dev_ptr);
B200GS_API size_t b200gs_pack_rows_workspace_bytes(int64_t n);
B200GS_API int b200gs_pack_rows(int64_t n, int64_t segment_len, int64_t segment_cap, const float* xy, const float* depth,
                                const float* conic, const float* comp, const float* opacity, const float* rgb, const int32_t* radii,
                                void* workspace, size_t workspace_bytes, int32_t* row_index, float* rows, int64_t* d_count, void* stream);
/* block_counts / block_rows (optional; NULL / 0 = every row counts): the rows arrive in blocks of block_rows rows of which only the first
 *     block_counts[b] are valid (the fixed-capacity exchange of the sharded renderer) — the rest reads as culled, so the receive buffer
 *     needs no padding pass. */
B200GS_API int b200gs_bin_count_rows(int32_t mode, int32_t width, int32_t height, int64_t n, const float* rows, int32_t cull,
                                     void* workspace_a, size_t workspace_a_bytes, int64_t* d_counts, int64_t* host_counts,
                                     int32_t sync_host, void* stream, const int64_t* block_counts, int64_t block_rows);
B200GS_API int b200gs_blend_fwd_rows(int32_t mode, int32_t width, int32_t height, const int32_t* tile_ranges, const int32_t* sorted_ids,
                                     const float* rows, const float* bg, float* image, int64_t pix_stride, int64_t ch_stride,
                                     float* final_T, int32_t* n_contrib, float* alpha, void* stream);
/* grad_scale_x / _y: factor on the mean2D columns of the gradient rows (vanilla renderers: 0.5 W, 0.5 H — the vanilla rasterizer's
 *     NDC-unit convention; gsplat renderers: 1, 1).  v_rows must be zero-filled: the kernel accumulates with 128-bit reductions. */
B200GS_API int b200gs_blend_bwd_rows(int32_t mode, int32_t width, int32_t height, const int32_t* tile_ranges, const int32_t* sorted_ids,
                                     const float* rows, const float* bg, const float* final_T, const int32_t* n_contrib,
                                     const float* v_image, int64_t pix_stride, int64_t ch_stride, const float* v_alpha,
                                     float grad_scale_x, float grad_scale_y, float* v_rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200GS_H */
