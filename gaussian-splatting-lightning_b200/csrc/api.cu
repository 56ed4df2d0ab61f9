// C ABI of libb200gs.so — see include/b200gs.h for the contract of every entry point.
#include <stdarg.h>
#include <string.h>

#include <atomic>

#include "common.cuh"

namespace b200gs {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static int check_view(const B200gsView* v, bool needs_sh) {
    if (v == nullptr) { set_error("view is NULL"); return B200GS_EINVAL; }
    if (v->width <= 0 || v->height <= 0) { set_error("bad image size %dx%d", v->width, v->height); return B200GS_EINVAL; }
    if (v->mode != B200GS_MODE_VANILLA && v->mode != B200GS_MODE_GSPLAT) { set_error("bad mode %d", v->mode); return B200GS_EINVAL; }
    if (needs_sh) {
        if (v->sh_degree < 0 || v->sh_degree > 4) { set_error("sh_degree %d unsupported (0..4)", v->sh_degree); return B200GS_EINVAL; }
        if (v->sh_stride < (v->sh_degree + 1) * (v->sh_degree + 1)) {
            set_error("sh_stride %d < (sh_degree+1)^2", v->sh_stride);
            return B200GS_EINVAL;
        }
    }
    return B200GS_OK;
}

}  // namespace b200gs

using namespace b200gs;

extern "C" {

const char* b200gs_last_error(void) { return g_error; }
int b200gs_version(void) { return 230; }
int64_t b200gs_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

int b200gs_project_fwd(const B200gsView* view, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, float* xy, float* depth, int32_t* radii, float* conic, float* comp,
                       int32_t* tiles, float* cov3d, float* rgb, uint8_t* clamped, void* stream) {
    int rc = check_view(view, shs != nullptr);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    if (n > 0) {
        B200GS_CHECK_ARG(means && scales && quats, "means/scales/quats must not be NULL");
        B200GS_CHECK_ARG(xy && depth && radii && conic && tiles, "xy/depth/radii/conic/tiles must not be NULL");
        B200GS_CHECK_ARG(shs == nullptr || (rgb && clamped), "rgb/clamped required when shs is given");
    }
    return launch_project_fwd(*view, n, means, scales, quats, shs, xy, depth, radii, conic, comp, tiles, cov3d, rgb, clamped,
                              (cudaStream_t)stream);
}

int b200gs_project_bwd(const B200gsView* view, int64_t n, const float* means, const float* scales, const float* quats,
                       const float* shs, const int32_t* radii, const uint8_t* clamped, const float* v_xy,
                       const float* v_depth, const float* v_conic, const float* v_comp, const float* v_rgb,
                       float* v_means, float* v_scales, float* v_quats, float* v_shs, void* stream) {
    int rc = check_view(view, shs != nullptr);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    if (n > 0) {
        B200GS_CHECK_ARG(means && scales && quats && radii, "means/scales/quats/radii must not be NULL");
        B200GS_CHECK_ARG(v_xy && v_conic, "v_xy/v_conic must not be NULL");
        B200GS_CHECK_ARG(v_means && v_scales && v_quats, "v_means/v_scales/v_quats must not be NULL");
        B200GS_CHECK_ARG((shs == nullptr) == (v_shs == nullptr), "shs and v_shs must be given together");
        B200GS_CHECK_ARG(shs == nullptr || (clamped && v_rgb), "clamped/v_rgb required when shs is given");
    }
    return launch_project_bwd(*view, n, means, scales, quats, shs, radii, clamped, v_xy, v_depth, v_conic, v_comp, v_rgb,
                              v_means, v_scales, v_quats, v_shs, (cudaStream_t)stream);
}

int b200gs_project_fwd_raw(const B200gsView* view, int64_t n, const float* means, const float* log_scales, const float* raw_quats,
                           const float* opacity_logits, const float* shs_dc, const float* shs_rest, int32_t anti_aliased,
                           float* xy, float* depth, int32_t* radii, float* conic, float* comp, int32_t* tiles, float* rgb,
                           uint8_t* clamped, float* opacity_out, void* stream) {
    int rc = check_view(view, true);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    if (n > 0) {
        B200GS_CHECK_ARG(means && log_scales && raw_quats && opacity_logits && shs_dc, "NULL input pointer");
        B200GS_CHECK_ARG(view->sh_stride == 1 || shs_rest, "shs_rest required when sh_stride > 1");
        B200GS_CHECK_ARG(xy && depth && radii && conic && tiles && rgb && clamped && opacity_out, "NULL output pointer");
    }
    return launch_project_fwd_raw(*view, n, means, log_scales, raw_quats, opacity_logits, shs_dc, shs_rest, anti_aliased, xy, depth,
                                  radii, conic, comp, tiles, nullptr, rgb, clamped, opacity_out, (cudaStream_t)stream);
}

int b200gs_project_fwd_rows(const B200gsView* view, int64_t n, const float* means, const float* log_scales, const float* raw_quats,
                            const float* opacity_logits, const float* shs_dc, const float* shs_rest, int32_t anti_aliased, float* rows,
                            int32_t* radii, uint8_t* clamped, int32_t* tiles, void* stream) {
    int rc = check_view(view, true);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    if (n > 0) {
        B200GS_CHECK_ARG(means && log_scales && raw_quats && opacity_logits && shs_dc, "NULL input pointer");
        B200GS_CHECK_ARG(view->sh_stride == 1 || shs_rest, "shs_rest required when sh_stride > 1");
        B200GS_CHECK_ARG(rows && radii && clamped, "NULL output pointer");
        B200GS_CHECK_ARG((reinterpret_cast<uintptr_t>(rows) & 15u) == 0, "rows must be 16-byte aligned");
    }
    return launch_project_fwd_raw(*view, n, means, log_scales, raw_quats, opacity_logits, shs_dc, shs_rest, anti_aliased, nullptr, nullptr,
                                  radii, nullptr, nullptr, tiles, nullptr, nullptr, clamped, nullptr, (cudaStream_t)stream, rows);
}

int b200gs_project_bwd_rows(const B200gsView* view, int64_t n, const float* means, const float* log_scales, const float* raw_quats,
                            const float* opacity_logits, const float* shs_dc, const float* shs_rest, int32_t anti_aliased,
                            const int32_t* radii, const uint8_t* clamped, const int32_t* row_offsets, const float* v_rows,
                            int32_t accumulate, float* v_means, float* v_log_scales, float* v_raw_quats, float* v_opacity_logits,
                            float* v_shs_dc, float* v_shs_rest, float* v_mean2d, int32_t v_mean2d_cols, void* stream) {
    int rc = check_view(view, true);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    B200GS_CHECK_ARG(v_mean2d == nullptr || v_mean2d_cols == 2 || v_mean2d_cols == 3, "v_mean2d_cols must be 2 or 3");
    if (n > 0) {
        B200GS_CHECK_ARG(means && log_scales && raw_quats && opacity_logits && shs_dc && radii && clamped, "NULL input pointer");
        B200GS_CHECK_ARG(view->sh_stride == 1 || (shs_rest && v_shs_rest), "shs_rest / v_shs_rest required when sh_stride > 1");
        B200GS_CHECK_ARG(v_means && v_log_scales && v_raw_quats && v_opacity_logits && v_shs_dc, "NULL output pointer");
    }
    static const float dummy = 0.f;   // v_rows may be NULL when no Gaussian of the shard is visible: never dereferenced then
    return launch_project_bwd_raw(*view, n, means, log_scales, raw_quats, opacity_logits, shs_dc, shs_rest, anti_aliased, radii,
                                  clamped, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, v_means, v_log_scales, v_raw_quats,
                                  v_opacity_logits, v_shs_dc, v_shs_rest, (cudaStream_t)stream, v_rows ? v_rows : &dummy, row_offsets,
                                  accumulate, v_mean2d, v_mean2d_cols);
}

static int check_views(const B200gsView* views, int32_t n_views) {
    if (views == nullptr) { set_error("views is NULL"); return B200GS_EINVAL; }
    if (n_views < 1 || n_views > B200GS_MAX_VIEWS) { set_error("n_views %d out of range (1..%d)", n_views, B200GS_MAX_VIEWS); return B200GS_EINVAL; }
    for (int j = 0; j < n_views; ++j) {
        int rc = check_view(views + j, true);
        if (rc) return rc;
        if (views[j].mode != B200GS_MODE_GSPLAT) { set_error("multi-view projection supports gsplat constants only"); return B200GS_EINVAL; }
        if (views[j].sh_degree != views[0].sh_degree || views[j].sh_stride != views[0].sh_stride) {
            set_error("all views of a multi-view launch must share sh_degree / sh_stride");
            return B200GS_EINVAL;
        }
    }
    return B200GS_OK;
}

int b200gs_project_fwd_raw_multi(const B200gsView* views, int32_t n_views, int64_t n, const float* means, const float* log_scales,
                                 const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                 int32_t anti_aliased, float* xy, float* depth, int32_t* radii, float* conic, float* rgb, uint8_t* clamped,
                                 float* opacity_out, void* stream) {
    int rc = check_views(views, n_views);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    if (n > 0) {
        B200GS_CHECK_ARG(means && log_scales && raw_quats && opacity_logits && shs_dc, "NULL input pointer");
        B200GS_CHECK_ARG(views[0].sh_stride == 1 || shs_rest, "shs_rest required when sh_stride > 1");
        B200GS_CHECK_ARG(xy && depth && radii && conic && rgb && clamped && opacity_out, "NULL output pointer");
    }
    return launch_project_fwd_multi(views, n_views, n, means, log_scales, raw_quats, opacity_logits, shs_dc, shs_rest, anti_aliased, xy, depth,
                                    radii, conic, rgb, clamped, opacity_out, (cudaStream_t)stream);
}

size_t b200gs_project_pack_workspace_bytes(int32_t n_views, int64_t n) { return project_pack_workspace_bytes(n_views, n); }

int b200gs_project_pack_multi(const B200gsView* views, int32_t n_views, int64_t n, const float* means, const float* log_scales,
                              const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                              int32_t anti_aliased, float* xy, int32_t* radii, uint8_t* clamped, int32_t* row_index, void* const* dst_rows,
                              int64_t block_rows, void* workspace, size_t workspace_bytes, int64_t* d_count, void* stream) {
    B200GS_CHECK_ARG(views && n_views >= 1 && n_views <= B200GS_MAX_VIEWS, "n_views must be 1..B200GS_MAX_VIEWS");
    B200GS_CHECK_ARG(n >= 0 && n < (int64_t(1) << 30) && block_rows > 0 && block_rows < (int64_t(1) << 30), "bad size");
    for (int j = 0; j < n_views; ++j) {
        int rc = check_view(views + j, true);
        if (rc) return rc;
        B200GS_CHECK_ARG(views[j].mode == B200GS_MODE_GSPLAT, "multi-view launches use the gsplat constant set");
        B200GS_CHECK_ARG(dst_rows && dst_rows[j] && (reinterpret_cast<uintptr_t>(dst_rows[j]) & 15u) == 0, "dst_rows: NULL or misaligned");
    }
    if (n > 0) {
        B200GS_CHECK_ARG(means && log_scales && raw_quats && opacity_logits && shs_dc, "NULL input pointer");
        B200GS_CHECK_ARG(views[0].sh_stride == 1 || shs_rest, "shs_rest required when sh_stride > 1");
        B200GS_CHECK_ARG(xy && radii && clamped && row_index && workspace, "NULL output pointer");
    }
    B200GS_CHECK_ARG(d_count, "NULL d_count");
    return launch_project_pack_multi(views, n_views, n, means, log_scales, raw_quats, opacity_logits, shs_dc, shs_rest, anti_aliased, xy, radii,
                                     clamped, row_index, (float* const*)dst_rows, block_rows, workspace, workspace_bytes, d_count,
                                     (cudaStream_t)stream);
}

int b200gs_project_bwd_rows_multi(const B200gsView* views, int32_t n_views, int64_t n, const float* means, const float* log_scales,
                                  const float* raw_quats, const float* opacity_logits, const float* shs_dc, const float* shs_rest,
                                  int32_t anti_aliased, const int32_t* radii, const uint8_t* clamped, const int32_t* row_index,
                                  const float* const* v_rows, float* v_means, float* v_log_scales, float* v_raw_quats,
                                  float* v_opacity_logits, float* v_shs_dc, float* v_shs_rest, void* stream) {
    int rc = check_views(views, n_views);
    if (rc) return rc;
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    if (n > 0) {
        B200GS_CHECK_ARG(means && log_scales && raw_quats && opacity_logits && shs_dc && radii && clamped && row_index && v_rows, "NULL input pointer");
        B200GS_CHECK_ARG(views[0].sh_stride == 1 || (shs_rest && v_shs_rest), "shs_rest / v_shs_rest required when sh_stride > 1");
        B200GS_CHECK_ARG(v_means && v_log_scales && v_raw_quats && v_opacity_logits && v_shs_dc, "NULL output pointer");
    }
    return launch_project_bwd_multi(views, n_views, n, means, log_scales, raw_quats, opacity_logits, shs_dc, shs_rest, anti_aliased, radii, clamped,
                                    row_index, v_rows, v_means, v_log_scales, v_raw_quats, v_opacity_logits, v_shs_dc, v_shs_rest,
                                    (cudaStream_t)stream);
}

int b200gs_ipc_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64) {
    B200GS_CHECK_ARG(dev_ptr != nullptr && handle64 != nullptr && bytes > 0, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    void* p = nullptr;
    B200GS_CUDA(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        set_error("b200gs_ipc_alloc: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
        return B200GS_ECUDA;
    }
    memcpy(handle64, &h, 64);
    *dev_ptr = p;
    return B200GS_OK;
}

int b200gs_ipc_open(const unsigned char* handle64, void** dev_ptr) {
    B200GS_CHECK_ARG(dev_ptr != nullptr && handle64 != nullptr, "bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    B200GS_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return B200GS_OK;
}

int b200gs_ipc_close(void* dev_ptr) {
    if (dev_ptr) B200GS_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return B200GS_OK;
}

int b200gs_ipc_free(void* dev_ptr) {
    if (dev_ptr) B200GS_CUDA(cudaFree(dev_ptr));
    return B200GS_OK;
}

int b200gs_selective_adam(int64_t rows, int32_t width, float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                          const uint8_t* visible, float lr, float beta1, float beta2, float eps, void* stream) {
    B200GS_CHECK_ARG(rows >= 0 && width > 0, "bad sizes");
    B200GS_CHECK_ARG(rows == 0 || (param && grad && exp_avg && exp_avg_sq && visible), "NULL pointer");
    return launch_selective_adam(rows, width, param, grad, exp_avg, exp_avg_sq, visible, lr, beta1, beta2, eps, (cudaStream_t)stream);
}

int b200gs_densify_stats(int64_t n, const int32_t* radii, const uint8_t* visible, const float* grad, int32_t grad_stride, float scale_x,
                         float scale_y, float* max_radii2d, float* grad_accum, float* denom, void* stream) {
    B200GS_CHECK_ARG(n >= 0 && grad_stride >= 2, "bad sizes");
    B200GS_CHECK_ARG(n == 0 || (radii && grad && max_radii2d && grad_accum && denom), "NULL pointer");
    return launch_densify_stats(n, radii, visible, grad, grad_stride, scale_x, scale_y, max_radii2d, grad_accum, denom, (cudaStream_t)stream);
}

size_t b200gs_knn_workspace_bytes(int64_t n) { return n < 0 ? 0 : knn_workspace_bytes(n); }

int b200gs_knn_mean_dist2(int64_t n, const float* points, float* mean_dist2, void* workspace, size_t workspace_bytes, void* stream) {
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    B200GS_CHECK_ARG(n == 0 || (points && mean_dist2 && workspace), "NULL pointer");
    return launch_knn_mean_dist2(n, points, mean_dist2, workspace, workspace_bytes, (cudaStream_t)stream);
}

int b200gs_sh_fwd(int32_t degree, int32_t sh_stride, int64_t n, const float* dirs, const float* coeffs, float* rgb, void* stream) {
    B200GS_CHECK_ARG(degree >= 0 && degree <= 4, "degree must be 0..4");
    B200GS_CHECK_ARG(sh_stride >= (degree + 1) * (degree + 1), "sh_stride < (degree+1)^2");
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    B200GS_CHECK_ARG(n == 0 || (dirs && coeffs && rgb), "NULL pointer");
    return launch_sh_fwd(degree, sh_stride, n, dirs, coeffs, rgb, (cudaStream_t)stream);
}

int b200gs_sh_bwd(int32_t degree, int32_t sh_stride, int64_t n, const float* dirs, const float* coeffs, const float* v_rgb,
                  float* v_coeffs, float* v_dirs, void* stream) {
    B200GS_CHECK_ARG(degree >= 0 && degree <= 4, "degree must be 0..4");
    B200GS_CHECK_ARG(sh_stride >= (degree + 1) * (degree + 1), "sh_stride < (degree+1)^2");
    B200GS_CHECK_ARG(n >= 0, "n < 0");
    B200GS_CHECK_ARG(n == 0 || (dirs && coeffs && v_rgb && v_coeffs), "NULL pointer");
    return launch_sh_bwd(degree, sh_stride, n, dirs, coeffs, v_rgb, v_coeffs, v_dirs, (cudaStream_t)stream);
}

size_t b200gs_bin_count_workspace_bytes(int64_t n) { return n < 0 ? 0 : bin_count_workspace_bytes(n); }

size_t b200gs_bin_sort_workspace_bytes(int64_t n, int64_t max_coarse, int32_t width, int32_t height) {
    if (n < 0 || max_coarse < 0 || width <= 0 || height <= 0) return 0;
    return bin_sort_workspace_bytes(n, max_coarse, width, height);
}

int b200gs_bin_count(int32_t mode, int32_t width, int32_t height, int64_t n, const float* xy, const float* depth,
                     const int32_t* radii, const float* cull_conic, const float* cull_opacity, void* workspace, size_t workspace_bytes,
                     int64_t* d_counts, int64_t* host_counts, int32_t sync_host, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0 && n >= 0, "bad size");
    B200GS_CHECK_ARG(workspace && d_counts, "workspace/d_counts must not be NULL");
    B200GS_CHECK_ARG(n == 0 || (xy && depth && radii), "NULL pointer");
    B200GS_CHECK_ARG(n < (int64_t(1) << 31), "n >= 2^31");
    B200GS_CHECK_ARG((cull_conic == nullptr) == (cull_opacity == nullptr), "cull_conic and cull_opacity go together");
    return bin_count(mode, width, height, n, 0, xy, depth, radii, cull_conic, cull_opacity, workspace, workspace_bytes, d_counts,
                     host_counts, sync_host, (cudaStream_t)stream);
}

int b200gs_bin_sort(int32_t mode, int32_t width, int32_t height, int64_t n, int32_t cull, int64_t max_coarse, int64_t max_pairs,
                    int64_t* d_counts, const void* workspace_a, void* workspace_b, size_t workspace_b_bytes, int32_t* sorted_ids,
                    int32_t* tile_ranges, int64_t* host_counts, int32_t sync_host, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0 && n >= 0 && max_pairs >= 0 && max_coarse >= 0, "bad size");
    B200GS_CHECK_ARG(d_counts != nullptr, "d_counts must not be NULL");
    B200GS_CHECK_ARG(workspace_a && workspace_b && tile_ranges, "workspace/tile_ranges must not be NULL");
    B200GS_CHECK_ARG(n == 0 || max_coarse == 0 || sorted_ids, "NULL pointer");
    return bin_sort(mode, width, height, n, cull, max_coarse, max_pairs, d_counts, workspace_a, workspace_b, workspace_b_bytes,
                    sorted_ids, tile_ranges, host_counts, sync_host, (cudaStream_t)stream);
}

int b200gs_blend_fwd(int32_t mode, int32_t width, int32_t height, int32_t channels, const int32_t* tile_ranges,
                     const int32_t* sorted_ids, const float* xy, const float* conic, const float* opacity,
                     const float* colors, const float* bg, float* image, int64_t pix_stride, int64_t ch_stride,
                     float* final_T, int32_t* n_contrib, float* alpha, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0, "bad size");
    B200GS_CHECK_ARG(tile_ranges && image && final_T && n_contrib, "NULL output/range pointer");
    return launch_blend_fwd(mode, width, height, channels, tile_ranges, sorted_ids, 0, xy, conic, opacity, colors, bg, image,
                            pix_stride, ch_stride, final_T, n_contrib, alpha, (cudaStream_t)stream);
}

int b200gs_blend_fwd_hits(int32_t mode, int32_t width, int32_t height, int32_t channels, const int32_t* tile_ranges,
                          const int32_t* sorted_ids, const float* xy, const float* conic, const float* opacity,
                          const float* colors, const float* bg, float* image, int64_t pix_stride, int64_t ch_stride,
                          float* final_T, int32_t* n_contrib, float* alpha, uint8_t* hit_any, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0, "bad size");
    B200GS_CHECK_ARG(tile_ranges && image && final_T && n_contrib && hit_any, "NULL output/range pointer");
    return launch_blend_fwd(mode, width, height, channels, tile_ranges, sorted_ids, 0, xy, conic, opacity, colors, bg, image,
                            pix_stride, ch_stride, final_T, n_contrib, alpha, (cudaStream_t)stream, hit_any);
}

int b200gs_blend_bwd(int32_t mode, int32_t width, int32_t height, int32_t channels, const int32_t* tile_ranges,
                     const int32_t* sorted_ids, const float* xy, const float* conic, const float* opacity,
                     const float* colors, const float* bg, const float* final_T, const int32_t* n_contrib,
                     const float* v_image, int64_t pix_stride, int64_t ch_stride, const float* v_alpha,
                     float xy_scale_x, float xy_scale_y, float* v_xy, float* v_conic, float* v_opacity,
                     float* v_colors, float* v_xy_abs, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0, "bad size");
    B200GS_CHECK_ARG(tile_ranges && final_T && n_contrib && v_image, "NULL input pointer");
    B200GS_CHECK_ARG(v_xy && v_conic && v_opacity && v_colors, "NULL output pointer");
    return launch_blend_bwd(mode, width, height, channels, tile_ranges, sorted_ids, 0, xy, conic, opacity, colors, bg, final_T,
                            n_contrib, v_image, pix_stride, ch_stride, v_alpha, xy_scale_x, xy_scale_y, v_xy, v_conic,
                            v_opacity, v_colors, v_xy_abs, (cudaStream_t)stream);
}

int b200gs_publish_i64(const int64_t* d_values, int64_t* host_values, int32_t n, void* stream) {
    B200GS_CHECK_ARG(d_values && host_values && n > 0, "bad argument");
    return publish_i64(d_values, host_values, n, (cudaStream_t)stream);
}

// ---- fused L1 + SSIM loss (experimental) ----------------------------------------------------------------------------------
int64_t b200gs_loss_blocks(int32_t channels, int32_t width, int32_t height) {
    if (channels <= 0 || width <= 0 || height <= 0) return 0;
    return loss_blocks(channels, width, height);
}

int b200gs_loss_fwd(int32_t channels, int32_t width, int32_t height, const float* image, const float* target, float* dmaps,
                    float* partials, void* stream) {
    B200GS_CHECK_ARG(channels > 0 && width > 0 && height > 0, "bad size");
    B200GS_CHECK_ARG(image && target && dmaps && partials, "NULL pointer");
    return launch_loss_fwd(channels, width, height, image, target, dmaps, partials, (cudaStream_t)stream);
}

int b200gs_loss_bwd(int32_t channels, int32_t width, int32_t height, const float* image, const float* target, const float* dmaps,
                    float lambda_dssim, const float* v_loss, float* v_image, void* stream) {
    B200GS_CHECK_ARG(channels > 0 && width > 0 && height > 0, "bad size");
    B200GS_CHECK_ARG(image && target && dmaps && v_image, "NULL pointer");
    return launch_loss_bwd(channels, width, height, image, target, dmaps, lambda_dssim, v_loss, v_image, (cudaStream_t)stream);
}

// ---- [n,12] row layout (the exchange format of the Gaussian-sharded renderer) -------------------------------------------
size_t b200gs_pack_rows_workspace_bytes(int64_t n) { return n < 0 ? 0 : pack_rows_workspace_bytes(n); }

int b200gs_pack_rows(int64_t n, int64_t segment_len, int64_t segment_cap, const float* xy, const float* depth, const float* conic,
                     const float* comp, const float* opacity, const float* rgb, const int32_t* radii, void* workspace,
                     size_t workspace_bytes, int32_t* row_index, float* rows, int64_t* d_count, void* stream) {
    B200GS_CHECK_ARG(n >= 0 && n < (int64_t(1) << 31), "bad n");
    B200GS_CHECK_ARG(segment_cap >= 0 && (segment_cap == 0 || segment_len > 0), "bad segment_len / segment_cap");
    B200GS_CHECK_ARG(segment_cap == 0 || (n + segment_len - 1) / segment_len * segment_cap < (int64_t(1) << 31), "segments * segment_cap >= 2^31");
    B200GS_CHECK_ARG(d_count != nullptr, "d_count must not be NULL");
    B200GS_CHECK_ARG(n == 0 || (xy && depth && conic && opacity && rgb && radii && workspace && row_index && rows), "NULL pointer");
    B200GS_CHECK_ARG(n == 0 || workspace_bytes >= pack_rows_workspace_bytes(n), "workspace too small");
    return pack_rows(n, segment_len, segment_cap, xy, depth, conic, comp, opacity, rgb, radii, workspace, workspace_bytes, row_index, rows,
                     d_count, (cudaStream_t)stream);
}

int b200gs_bin_count_rows(int32_t mode, int32_t width, int32_t height, int64_t n, const float* rows, int32_t cull, void* workspace,
                          size_t workspace_bytes, int64_t* d_counts, int64_t* host_counts, int32_t sync_host, void* stream,
                          const int64_t* block_counts, int64_t block_rows) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0 && n >= 0 && n < (int64_t(1) << 31), "bad size");
    B200GS_CHECK_ARG(workspace && d_counts && (n == 0 || rows), "NULL pointer");
    return bin_count(mode, width, height, n, B200GS_ROW_FLOATS, rows + B200GS_ROW_XY, rows + B200GS_ROW_DEPTH,
                     (const int32_t*)(rows + B200GS_ROW_RADIUS), cull ? rows + B200GS_ROW_CONIC : nullptr,
                     cull ? rows + B200GS_ROW_OPACITY : nullptr, workspace, workspace_bytes, d_counts, host_counts, sync_host,
                     (cudaStream_t)stream, block_counts, block_rows);
}

int b200gs_blend_fwd_rows(int32_t mode, int32_t width, int32_t height, const int32_t* tile_ranges, const int32_t* sorted_ids,
                          const float* rows, const float* bg, float* image, int64_t pix_stride, int64_t ch_stride, float* final_T,
                          int32_t* n_contrib, float* alpha, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0 && tile_ranges && image && final_T && n_contrib, "bad argument");
    return launch_blend_fwd(mode, width, height, 3, tile_ranges, sorted_ids, B200GS_ROW_FLOATS, rows + B200GS_ROW_XY,
                            rows + B200GS_ROW_CONIC, rows + B200GS_ROW_OPACITY, rows + B200GS_ROW_RGB, bg, image, pix_stride,
                            ch_stride, final_T, n_contrib, alpha, (cudaStream_t)stream);
}

int b200gs_blend_bwd_rows(int32_t mode, int32_t width, int32_t height, const int32_t* tile_ranges, const int32_t* sorted_ids,
                          const float* rows, const float* bg, const float* final_T, const int32_t* n_contrib, const float* v_image,
                          int64_t pix_stride, int64_t ch_stride, const float* v_alpha, float grad_scale_x, float grad_scale_y,
                          float* v_rows, void* stream) {
    B200GS_CHECK_ARG(mode == B200GS_MODE_VANILLA || mode == B200GS_MODE_GSPLAT, "bad mode");
    B200GS_CHECK_ARG(width > 0 && height > 0 && tile_ranges && final_T && n_contrib && v_image && v_rows, "bad argument");
    return launch_blend_bwd(mode, width, height, 3, tile_ranges, sorted_ids, B200GS_ROW_FLOATS, rows + B200GS_ROW_XY,
                            rows + B200GS_ROW_CONIC, rows + B200GS_ROW_OPACITY, rows + B200GS_ROW_RGB, bg, final_T, n_contrib, v_image,
                            pix_stride, ch_stride, v_alpha, grad_scale_x, grad_scale_y, v_rows + B200GS_ROW_XY, v_rows + B200GS_ROW_CONIC,
                            v_rows + B200GS_ROW_OPACITY, v_rows + B200GS_ROW_RGB, nullptr, (cudaStream_t)stream);
}

}  // extern "C"
