// Shared device/host helpers for libb200gs (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b200gs.h"

namespace b200gs {

void set_error(const char* fmt, ...);
void count_launch();   // every kernel launch of the library is counted (b200gs_launch_count): B200GS_LAUNCH_CHECK follows each <<<>>>

#define B200GS_CHECK_ARG(cond, msg)                                  \
    do {                                                              \
        if (!(cond)) {                                                \
            b200gs::set_error("%s: %s", __func__, msg);              \
            return B200GS_EINVAL;                                     \
        }                                                             \
    } while (0)

#define B200GS_CUDA(call)                                                                     \
    do {                                                                                       \
        cudaError_t _e = (call);                                                               \
        if (_e != cudaSuccess) {                                                               \
            b200gs::set_error("%s: %s failed: %s", __func__, #call, cudaGetErrorString(_e));  \
            return B200GS_ECUDA;                                                               \
        }                                                                                      \
    } while (0)

#define B200GS_LAUNCH_CHECK()                                                                  \
    do {                                                                                       \
        b200gs::count_launch();                                                                \
        cudaError_t _e = cudaGetLastError();                                                   \
        if (_e != cudaSuccess) {                                                               \
            b200gs::set_error("%s: kernel launch failed: %s", __func__, cudaGetErrorString(_e)); \
            return B200GS_ECUDA;                                                               \
        }                                                                                      \
    } while (0)

constexpr int TILE = B200GS_TILE;

__host__ __device__ inline int div_up(int a, int b) { return (a + b - 1) / b; }
inline int64_t div_up64(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Tile rectangle touched by a splat: the two rules of SURVEY §8c.
//   vanilla (dgr getRect):   min = clamp(int((p - r)/16)),  max = clamp(int((p + r + 15)/16))
//   gsplat  (gaussian_projection.py:118-123): min = clamp(int((p - r)/16)),  max = clamp(int((p + r)/16) + 1)
// (int) truncates toward zero exactly like torch's .int(); clamp to [0, grid].
template <bool GSPLAT>
__device__ __forceinline__ void tile_rect(float x, float y, float r, int grid_x, int grid_y, int& x0, int& y0, int& x1, int& y1) {
    const float inv = 1.0f / float(TILE);  // exact power of two: same result as dividing
    x0 = min(grid_x, max(0, (int)((x - r) * inv)));
    y0 = min(grid_y, max(0, (int)((y - r) * inv)));
    if (GSPLAT) {
        x1 = min(grid_x, max(0, (int)((x + r) * inv) + 1));
        y1 = min(grid_y, max(0, (int)((y + r) * inv) + 1));
    } else {
        x1 = min(grid_x, max(0, (int)((x + r + float(TILE - 1)) * inv)));
        y1 = min(grid_y, max(0, (int)((y + r + float(TILE - 1)) * inv)));
    }
}

__device__ __forceinline__ float warp_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

// launchers (one per translation unit)
int launch_project_fwd(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, float* xy, float* depth, int32_t* radii, float* conic, float* comp,
                       int32_t* tiles, float* cov3d, float* rgb, uint8_t* clamped, cudaStream_t s);
int launch_project_bwd(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, const int32_t* radii, const uint8_t* clamped, const float* v_xy,
                       const float* v_depth, const float* v_conic, const float* v_comp, const float* v_rgb,
                       float* v_means, float* v_scales, float* v_quats, float* v_shs, cudaStream_t s);
int launch_project_fwd_raw(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                           const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, float* xy,
                           float* depth, int32_t* radii, float* conic, float* comp, int32_t* tiles, float* cov3d, float* rgb,
                           uint8_t* clamped, float* opac_out, cudaStream_t s, float* rows = nullptr);
int launch_project_bwd_raw(const B200gsView& v, int64_t n, const float* means, const float* scales, const float* quats,
                           const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased,
                           const int32_t* radii, const uint8_t* clamped, const float* v_xy, const float* v_depth,
                           const float* v_conic, const float* v_comp, const float* v_rgb, const float* v_opac, float* v_means,
                           float* v_scales, float* v_quats, float* v_opac_logit, float* v_shs_dc, float* v_shs_rest,
                           cudaStream_t s, const float* v_rows = nullptr, const int32_t* row_offsets = nullptr, int accumulate = 0,
                           float* v_mean2d = nullptr, int v_mean2d_cols = 0);
int launch_project_fwd_multi(const B200gsView* views, int n_views, int64_t n, const float* means, const float* scales, const float* quats,
                             const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, float* xy, float* depth,
                             int32_t* radii, float* conic, float* rgb, uint8_t* clamped, float* opac_out, cudaStream_t s);
size_t project_pack_workspace_bytes(int n_views, int64_t n);
int launch_project_pack_multi(const B200gsView* views, int n_views, int64_t n, const float* means, const float* scales, const float* quats,
                              const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, float* xy, int32_t* radii,
                              uint8_t* clamped, int32_t* row_index, float* const* dst_rows, int64_t cap, void* workspace, size_t workspace_bytes,
                              int64_t* d_count, cudaStream_t s);
int launch_project_bwd_multi(const B200gsView* views, int n_views, int64_t n, const float* means, const float* scales, const float* quats,
                             const float* opac_logits, const float* shs_dc, const float* shs_rest, int anti_aliased, const int32_t* radii,
                             const uint8_t* clamped, const int32_t* row_index, const float* const* v_rows, float* v_means, float* v_scales,
                             float* v_quats, float* v_opac_logit, float* v_shs_dc, float* v_shs_rest, cudaStream_t s);
int launch_sh_fwd(int degree, int stride, int64_t n, const float* dirs, const float* coeffs, float* rgb, cudaStream_t s);
int launch_sh_bwd(int degree, int stride, int64_t n, const float* dirs, const float* coeffs, const float* v_rgb,
                  float* v_coeffs, float* v_dirs, cudaStream_t s);

size_t bin_count_workspace_bytes(int64_t n);
size_t bin_sort_workspace_bytes(int64_t n, int64_t max_coarse, int width, int height);
int bin_count(int mode, int width, int height, int64_t n, int row_stride, const float* xy, const float* depth, const int32_t* radii,
              const float* conic, const float* opacity, void* ws, size_t ws_bytes, int64_t* d_counts, int64_t* host_counts,
              int sync_host, cudaStream_t s, const int64_t* block_counts = nullptr, int64_t block_rows = 0);
int publish_i64(const int64_t* d_values, int64_t* host_values, int n, cudaStream_t s);
size_t pack_rows_workspace_bytes(int64_t n);
int pack_rows(int64_t n, int64_t seg_len, int64_t seg_cap, const float* xy, const float* depth, const float* conic, const float* comp,
              const float* opacity, const float* rgb, const int32_t* radii, void* ws, size_t ws_bytes, int32_t* row_index, float* rows,
              int64_t* d_count, cudaStream_t s);
int bin_sort(int mode, int width, int height, int64_t n, int cull, int64_t max_coarse, int64_t max_pairs, int64_t* d_counts,
             const void* ws_a, void* ws_b, size_t ws_b_bytes, int32_t* sorted_ids, int32_t* tile_ranges, int64_t* host_counts,
             int sync_host, cudaStream_t s);

int launch_selective_adam(int64_t rows, int width, float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const uint8_t* visible,
                          float lr, float b1, float b2, float eps, cudaStream_t s);
int launch_densify_stats(int64_t n, const int32_t* radii, const uint8_t* visible, const float* grad, int grad_stride, float sx, float sy,
                         float* max_radii2d, float* grad_accum, float* denom, cudaStream_t s);

size_t knn_workspace_bytes(int64_t n);
int launch_knn_mean_dist2(int64_t n, const float* points, float* out, void* ws, size_t ws_bytes, cudaStream_t s);

int64_t loss_blocks(int channels, int width, int height);
int launch_loss_fwd(int channels, int width, int height, const float* img, const float* gt, float* dmaps, float* partials, cudaStream_t s);
int launch_loss_bwd(int channels, int width, int height, const float* img, const float* gt, const float* dmaps, float lambda_dssim,
                    const float* v_loss, float* v_img, cudaStream_t s);

int launch_blend_fwd(int mode, int width, int height, int channels, const int32_t* ranges, const int32_t* ids,
                     int row_stride, const float* xy, const float* conic, const float* opacity, const float* colors, const float* bg,
                     float* image, int64_t pix_stride, int64_t ch_stride, float* final_T, int32_t* n_contrib,
                     float* alpha, cudaStream_t s, uint8_t* hit_any = nullptr);
int launch_blend_bwd(int mode, int width, int height, int channels, const int32_t* ranges, const int32_t* ids,
                     int row_stride, const float* xy, const float* conic, const float* opacity, const float* colors, const float* bg,
                     const float* final_T, const int32_t* n_contrib, const float* v_image, int64_t pix_stride,
                     int64_t ch_stride, const float* v_alpha, float sx, float sy, float* v_xy, float* v_conic,
                     float* v_opacity, float* v_colors, float* v_xy_abs, cudaStream_t s);

}  // namespace b200gs
