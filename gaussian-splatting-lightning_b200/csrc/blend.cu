// K6 / K7: per-tile front-to-back alpha compositing, forward and backward.
//
// Restates the published per-pixel loops of diff-gaussian-rasterization@59f5f77 renderCUDA (vanilla mode) and gsplat's
// rasterize_to_pixels (gsplat mode) — SURVEY.md §8c / Appendix B; the sources are not under /root/reference, the CPU
// restatement in oracle/gs_oracle.py::blend is the checker.
//
// One CTA per 16x16 tile, one thread per pixel; a warp owns an 8x4 pixel block.  Each round stages up to 256 splats of
// the tile's depth-sorted slab into shared memory (coalesced id read, L2-resident gathers of the 36 B splat record).
// While staging, the thread that fetched a splat also computes an 8-bit mask: which of the tile's eight 8x4 blocks
// the splat can reach with alpha >= 1/255 (exact convex minimum of the conic's quadratic over the block, same test as
// the tile culling of binning.cu).  Every warp then compacts the staged slab into its own index list with ballots, so
// its pixel loop only visits splats that can touch its block: ~half of the (warp, splat) visits of the plain loop
// disappear, and results stay bit-identical (a skipped splat would have failed the alpha test in all 32 lanes).
//
// Forward: the conic is pre-scaled by -0.5*log2(e) / -log2(e) while staging, so the per-(pixel,splat) body is
// 5 FP32 ops + one MUFU.EX2 + compare/blend; colours are fetched (one LDS.128) only by contributing lanes.
//
// Backward walks each warp's list in reverse, only up to the deepest contributor of the warp.  Each pixel evaluates RB
// consecutive list entries and keeps their 9 partial derivatives in registers; the warp then reduces them with a
// reduce-SCATTER butterfly (halving exchanges: RB -> RB/2 -> ... -> 1 value per lane) and one lane per splat issues
// the atomics: 32x fewer L2 atomics than the reference's per-pixel atomicAdd.
#include "common.cuh"

namespace b200gs {

namespace {

constexpr int BLOCK_PIX = TILE * TILE;  // 256 threads
constexpr int NWARP = BLOCK_PIX / 32;
constexpr float ALPHA_MIN = 1.0f / 255.0f;
constexpr float T_STOP = 1e-4f;
constexpr float LOG2E = 1.4426950408889634f;
constexpr unsigned FULL = 0xffffffffu;

// Element strides of the per-splat arrays: {2,3,1,CH} for separate contiguous arrays; {12,12,12,12} when all four
// pointers address columns of one [n,12] row buffer (the exchange format of the Gaussian-sharded renderer).
struct SplatStrides {
    int xs, cs, os, ks;
};

__device__ __forceinline__ void pixel_of_thread(int tid, int& lx, int& ly) {
    const int w = tid >> 5, l = tid & 31;
    lx = ((w & 1) << 3) + (l & 7);
    ly = ((w >> 1) << 2) + (l >> 3);
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Minimum of q(d) = (A dx^2 + C dy^2)/2 + B dx dy over the box [X0,X1]x[Y0,Y1] (d measured from the splat centre).
__device__ __forceinline__ float box_qmin(float A, float B, float C, float iA, float iC, float X0, float X1, float Y0, float Y1) {
    if (X0 <= 0.f && X1 >= 0.f && Y0 <= 0.f && Y1 >= 0.f) return 0.f;
    float qmin = 3.0e38f;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const float Xe = e ? X1 : X0;
        const float bx = B * Xe;
        const float ys = fminf(Y1, fmaxf(Y0, -bx * iC));
        qmin = fminf(qmin, fmaf(ys, fmaf(0.5f * C, ys, bx), 0.5f * A * Xe * Xe));
        const float Ye = e ? Y1 : Y0;
        const float by = B * Ye;
        const float xs = fminf(X1, fmaxf(X0, -by * iA));
        qmin = fminf(qmin, fmaf(xs, fmaf(0.5f * A, xs, by), 0.5f * C * Ye * Ye));
    }
    return qmin;
}

// bit w set <=> the splat can reach alpha >= 1/255 somewhere in warp w's 8x4 block of the tile at (ox, oy)
__device__ __forceinline__ unsigned block_mask(float mx, float my, float A, float B, float C, float opac, float ox, float oy) {
    const float o255 = 255.0f * opac;
    if (o255 <= 1.0f) return 0u;
    const float thresh = fmaf(__logf(o255), 1.0001f, 1e-3f);  // ln(255 o) + margin for fp32 / ex2.approx rounding
    const float iA = 1.0f / A, iC = 1.0f / C;
    unsigned m = 0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) {
        const float X0 = ox + float((w & 1) << 3) - mx, Y0 = oy + float((w >> 1) << 2) - my;
        const float q = box_qmin(A, B, C, iA, iC, X0, X0 + 7.0f, Y0, Y0 + 3.0f);
        m |= (!(q > thresh)) ? (1u << w) : 0u;  // NaN -> keep
    }
    return m;
}

// Staged splats live in shared memory as 48-byte records (3 x float4): one base address per splat, immediate offsets.
//   forward : {x, y, a', b'} {c', opacity, col0, col1} {col2, col3, -, -}     (a',b',c' = conic pre-scaled by -0.5*log2e / -log2e)
//   backward: {x, y, A, B}   {C, opacity, col0, col1}  {col2, col3, id, -}
// Record DUMMY (index 256) has opacity 0: it fails the alpha test in every lane and pads the per-warp lists to a
// multiple of the unroll factor, so the pixel loops are straight-line code.
constexpr int DUMMY = BLOCK_PIX;
constexpr int LIST_PAD = 8;

// Every warp compacts the staged slab [0,top) into the ascending list of entries whose mask has its bit set.
// my_list[LIST_PAD + k] = k-th entry; the LIST_PAD slots in front and the slots after the end hold DUMMY.
template <int FRONT = LIST_PAD>
__device__ __forceinline__ int build_list(const unsigned char* __restrict__ s_mask, unsigned short* __restrict__ my_list, int top, int warp,
                                          unsigned lane) {
    int n = 0;
    if (lane < FRONT) my_list[lane] = (unsigned short)DUMMY;
    for (int c = 0; c < top; c += 32) {
        const int j = c + (int)lane;
        const bool hit = (j < top) && ((s_mask[j] >> warp) & 1u);
        const unsigned b = __ballot_sync(FULL, hit);
        if (hit) my_list[FRONT + n + __popc(b & ((1u << lane) - 1u))] = (unsigned short)j;
        n += __popc(b);
    }
    if (lane < LIST_PAD) my_list[FRONT + n + lane] = (unsigned short)DUMMY;
    __syncwarp();
    return n;
}

template <int CH, bool GSPLAT>
__global__ void __launch_bounds__(BLOCK_PIX, 1) blend_fwd_kernel(int width, int height, int grid_x, const int2* __restrict__ ranges,
                                                              const int32_t* __restrict__ ids, const SplatStrides st, const float* __restrict__ xy,
                                                              const float* __restrict__ conic, const float* __restrict__ opacity,
                                                              const float* __restrict__ colors, const float* __restrict__ bg,
                                                              float* __restrict__ image, int64_t pix_stride, int64_t ch_stride,
                                                              float* __restrict__ final_T, int32_t* __restrict__ n_contrib,
                                                              float* __restrict__ alpha_out) {
    __shared__ float4 s_rec[(BLOCK_PIX + 1) * 3];
    __shared__ unsigned char s_mask[BLOCK_PIX];
    __shared__ unsigned short s_list[NWARP][BLOCK_PIX + 2 * LIST_PAD];

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const unsigned lane = tid & 31u;
    // 1-D grid over the tiles, row-major.  (A longest-list-first order, from a counting sort of the tile counts, was measured in round 2:
    // K6 0.286 -> 0.287 ms, K7 0.4405 -> 0.4423 ms, plus 11 us for the ordering kernel — the kernels' tails are not what limits them.)
    const int tile = (int)blockIdx.x;
    const int tile_y = tile / grid_x, tile_x = tile - tile_y * grid_x;
    int lx, ly;
    pixel_of_thread(tid, lx, ly);
    const int px = tile_x * TILE + lx, py = tile_y * TILE + ly;
    const bool inside = (px < width) && (py < height);
    const float off = GSPLAT ? 0.5f : 0.0f;
    const float pxf = float(px) + off, pyf = float(py) + off;
    const float ox = float(tile_x * TILE) + off, oy = float(tile_y * TILE) + off;
    const float amax = GSPLAT ? 0.999f : 0.99f;
    if (tid < 3) s_rec[DUMMY * 3 + tid] = make_float4(0.f, 0.f, 0.f, 0.f);

    const int2 range = ranges[tile];
    int todo = range.y - range.x;
    float T = 1.0f, Tc = inside ? 1.0f : 0.0f;     // Tc == 0: this pixel is finished (or outside the image)
    int last = 0;
    float C[4] = {0.f, 0.f, 0.f, 0.f};

    for (int base = 0; todo > 0; base += BLOCK_PIX, todo -= BLOCK_PIX) {
        if (__syncthreads_and(Tc == 0.0f)) break;
        const int cnt = min(BLOCK_PIX, todo);
        if (tid < cnt) {
            const int g = __ldg(ids + range.x + base + tid);
            const float2 m = __ldg(reinterpret_cast<const float2*>(xy + int64_t(g) * st.xs));
            const float* cq = conic + int64_t(g) * st.cs;
            const float A = __ldg(cq), B = __ldg(cq + 1), Cc = __ldg(cq + 2);
            const float o = __ldg(opacity + int64_t(g) * st.os);
            float col[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c = 0; c < CH; ++c) col[c] = __ldg(colors + int64_t(g) * st.ks + c);
            s_rec[tid * 3 + 0] = make_float4(m.x, m.y, (-0.5f * LOG2E) * A, -LOG2E * B);
            s_rec[tid * 3 + 1] = make_float4((-0.5f * LOG2E) * Cc, o, col[0], col[1]);
            if (CH > 2) s_rec[tid * 3 + 2] = make_float4(col[2], col[3], 0.f, 0.f);
            s_mask[tid] = (unsigned char)block_mask(m.x, m.y, A, B, Cc, o, ox, oy);
        }
        __syncthreads();
        if (__all_sync(FULL, Tc == 0.0f)) continue;  // warp finished: only keeps the block barriers company
        const unsigned short* my_list = s_list[warp] + LIST_PAD;
        const int nl = build_list(s_mask, s_list[warp], cnt, warp, lane);
        for (int i0 = 0; i0 < nl; i0 += 4) {
            if (__all_sync(FULL, Tc == 0.0f)) break;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = my_list[i0 + u];                 // entries past nl are DUMMY (alpha 0)
                const float4 r0 = s_rec[j * 3 + 0];
                const float4 r1 = s_rec[j * 3 + 1];
                const float dx = r0.x - pxf, dy = r0.y - pyf;
                // power * log2(e) = a' dx^2 + b' dx dy + c' dy^2
                const float p2 = fmaf(r1.x * dy, dy, fmaf(r0.w, dy, r0.z * dx) * dx);
                float a = fminf(amax, r1.y * ex2_approx(p2));
                a = (!(p2 > 0.0f) && !(a < ALPHA_MIN)) ? a : 0.f;             // a sample that fails the alpha test composites nothing
                // Tc is the transmittance used for compositing; it drops to exactly 0 when the pixel stops, so every later sample
                // weighs nothing without a `done` predicate in the arithmetic; T keeps the value in front of the stopping sample
                const float nT = fmaf(-a, Tc, Tc);
                const bool stop = GSPLAT ? (nT <= T_STOP) : (nT < T_STOP);
                const float w = stop ? 0.f : a * Tc;
                C[0] = fmaf(r1.z, w, C[0]);
                if (CH > 1) C[1] = fmaf(r1.w, w, C[1]);
                if (CH > 2) {
                    const float2 r2 = *reinterpret_cast<const float2*>(&s_rec[j * 3 + 2]);
                    C[2] = fmaf(r2.x, w, C[2]);
                    if (CH > 3) C[3] = fmaf(r2.y, w, C[3]);
                }
                last = (w > 0.f) ? base + j + 1 : last;
                T = stop ? T : nT;
                Tc = stop ? 0.f : nT;
            }
        }
    }
    if (inside) {
        const int64_t pix = int64_t(py) * width + px;
        final_T[pix] = T;
        n_contrib[pix] = last;
        if (alpha_out) alpha_out[pix] = 1.0f - T;
#pragma unroll
        for (int c = 0; c < CH; ++c) image[pix * pix_stride + c * ch_stride] = C[c] + (bg ? T * __ldg(bg + c) : 0.f);
    }
}

// ---- forward with asynchronous slab staging -----------------------------------------------------------------------------
// Same arithmetic and the same per-warp lists as blend_fwd_kernel; what changes is how a batch reaches shared memory.
// The tile's slab is an indirection (sorted ids -> records scattered over the splat arrays), so every thread copies
// "its" splat of the NEXT batch with cp.async (LDGSTS: global -> shared without a register round trip, 8 B + 7 x 4 B from the
// separate arrays, or 3 x 16 B from a [n,12] row buffer) into the second of two staging buffers while the warps blend the current
// batch; the ids are prefetched two batches ahead in a register.  When a batch starts, its copies have landed long
// ago (cp.async.wait_all + barrier), each thread post-processes its own record in place (conic pre-scaling, 8-bit block
// mask) and the warps go on to the list compaction: the two dependent L2 round trips of the synchronous version
// (id -> record) are off the critical path of the tile.
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// raw slot layout (floats): separate arrays -> {x, y, A, B | C, o, c0, c1 | c2, c3, -, -};  rows -> the 12 floats of the row
// {x, y, depth, A | B, C, comp, o | r, g, b, radius}
template <int CH, bool ROWS>
__device__ __forceinline__ void stage_async(float4* slot, int g, const SplatStrides& st, const float* __restrict__ xy,
                                            const float* __restrict__ conic, const float* __restrict__ opacity,
                                            const float* __restrict__ colors) {
    if (ROWS) {
        const float* row = xy + int64_t(g) * st.xs;     // xy points at column 0 of the row buffer
        cp_async16(slot, row);
        cp_async16(slot + 1, row + 4);
        cp_async16(slot + 2, row + 8);
    } else {
        float* f = reinterpret_cast<float*>(slot);
        cp_async8(f, xy + int64_t(g) * st.xs);
        const float* cq = conic + int64_t(g) * st.cs;
        cp_async4(f + 2, cq);
        cp_async4(f + 3, cq + 1);
        cp_async4(f + 4, cq + 2);
        cp_async4(f + 5, opacity + int64_t(g) * st.os);
#pragma unroll
        for (int c = 0; c < CH; ++c) cp_async4(f + 6 + c, colors + int64_t(g) * st.ks + c);
    }
}

// HITS: also mark every splat that contributed to at least one pixel (gsplat's `means2d.has_hit_any_pixels`, read by
// SelectiveAdam, optimizers.py:39, and exported as `acc_vis`, gsplat_v1_renderer.py:287): one byte store per (warp, contributing entry).
template <int CH, bool GSPLAT, bool ROWS, bool HITS>
__global__ void __launch_bounds__(BLOCK_PIX, 3) blend_fwd_async_kernel(int width, int height, int grid_x, const int2* __restrict__ ranges,
                                                              const int32_t* __restrict__ ids, const SplatStrides st, const float* __restrict__ xy,
                                                              const float* __restrict__ conic, const float* __restrict__ opacity,
                                                              const float* __restrict__ colors, const float* __restrict__ bg,
                                                              float* __restrict__ image, int64_t pix_stride, int64_t ch_stride,
                                                              float* __restrict__ final_T, int32_t* __restrict__ n_contrib,
                                                              float* __restrict__ alpha_out, uint8_t* __restrict__ hit_any) {
    __shared__ float4 s_buf[2][(BLOCK_PIX + 1) * 3];
    __shared__ int32_t s_gid[HITS ? BLOCK_PIX + 1 : 1];
    __shared__ unsigned char s_mask[BLOCK_PIX];
    __shared__ unsigned short s_list[NWARP][BLOCK_PIX + 2 * LIST_PAD];

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const unsigned lane = tid & 31u;
    const int tile = (int)blockIdx.x;
    const int tile_y = tile / grid_x, tile_x = tile - tile_y * grid_x;
    int lx, ly;
    pixel_of_thread(tid, lx, ly);
    const int px = tile_x * TILE + lx, py = tile_y * TILE + ly;
    const bool inside = (px < width) && (py < height);
    const float off = GSPLAT ? 0.5f : 0.0f;
    const float pxf = float(px) + off, pyf = float(py) + off;
    const float ox = float(tile_x * TILE) + off, oy = float(tile_y * TILE) + off;
    const float amax = GSPLAT ? 0.999f : 0.99f;
    if (tid < 6) s_buf[tid / 3][DUMMY * 3 + tid % 3] = make_float4(0.f, 0.f, 0.f, 0.f);

    const int2 range = ranges[tile];
    const int total = range.y - range.x;
    float T = 1.0f, Tc = inside ? 1.0f : 0.0f;
    int last = 0;
    float C[4] = {0.f, 0.f, 0.f, 0.f};

    // prologue: batch 0 in flight, ids of batch 1 in a register
    int cur_id = (tid < total) ? __ldg(ids + range.x + tid) : 0;
    if (tid < total) stage_async<CH, ROWS>(&s_buf[0][tid * 3], cur_id, st, xy, conic, opacity, colors);
    int next_id = (BLOCK_PIX + tid < total) ? __ldg(ids + range.x + BLOCK_PIX + tid) : 0;

    int buf = 0;
    for (int base = 0; base < total; base += BLOCK_PIX, buf ^= 1) {
        cp_async_wait_all();
        if (__syncthreads_and(Tc == 0.0f)) break;    // also: every thread's copies of this batch are visible
        const int cnt = min(BLOCK_PIX, total - base);
        float4* s_rec = s_buf[buf];
        if (tid < cnt) {
            const float4 q0 = s_rec[tid * 3 + 0], q1 = s_rec[tid * 3 + 1], q2 = s_rec[tid * 3 + 2];
            float mx, my, A, B, Cc, o, c0, c1, c2, c3;
            if (ROWS) { mx = q0.x; my = q0.y; A = q0.w; B = q1.x; Cc = q1.y; o = q1.w; c0 = q2.x; c1 = q2.y; c2 = q2.z; c3 = 0.f; }
            else      { mx = q0.x; my = q0.y; A = q0.z; B = q0.w; Cc = q1.x; o = q1.y; c0 = q1.z; c1 = q1.w; c2 = q2.x; c3 = q2.y; }
            s_rec[tid * 3 + 0] = make_float4(mx, my, (-0.5f * LOG2E) * A, -LOG2E * B);
            s_rec[tid * 3 + 1] = make_float4((-0.5f * LOG2E) * Cc, o, c0, CH > 1 ? c1 : 0.f);
            if (CH > 2) s_rec[tid * 3 + 2] = make_float4(c2, CH > 3 ? c3 : 0.f, 0.f, 0.f);
            s_mask[tid] = (unsigned char)block_mask(mx, my, A, B, Cc, o, ox, oy);
            if (HITS) s_gid[tid] = cur_id;
        }
        cur_id = next_id;
        // next batch: the other buffer was last read by the blend loop of the previous iteration, which every warp left
        // before the barrier above
        if (base + BLOCK_PIX + tid < total) stage_async<CH, ROWS>(&s_buf[buf ^ 1][tid * 3], next_id, st, xy, conic, opacity, colors);
        next_id = (base + 2 * BLOCK_PIX + tid < total) ? __ldg(ids + range.x + base + 2 * BLOCK_PIX + tid) : 0;
        __syncthreads();
        if (__all_sync(FULL, Tc == 0.0f)) continue;  // warp finished: only keeps the block barriers company
        const unsigned short* my_list = s_list[warp] + LIST_PAD;
        const int nl = build_list(s_mask, s_list[warp], cnt, warp, lane);
        for (int i0 = 0; i0 < nl; i0 += 4) {
            if (__all_sync(FULL, Tc == 0.0f)) break;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = my_list[i0 + u];                 // entries past nl are DUMMY (alpha 0)
                const float4 r0 = s_rec[j * 3 + 0];
                const float4 r1 = s_rec[j * 3 + 1];
                const float dx = r0.x - pxf, dy = r0.y - pyf;
                const float p2 = fmaf(r1.x * dy, dy, fmaf(r0.w, dy, r0.z * dx) * dx);
                float a = fminf(amax, r1.y * ex2_approx(p2));
                a = (!(p2 > 0.0f) && !(a < ALPHA_MIN)) ? a : 0.f;
                const float nT = fmaf(-a, Tc, Tc);             // same arithmetic as blend_fwd_kernel: see there
                const bool stop = GSPLAT ? (nT <= T_STOP) : (nT < T_STOP);
                const float w = stop ? 0.f : a * Tc;
                C[0] = fmaf(r1.z, w, C[0]);
                if (CH > 1) C[1] = fmaf(r1.w, w, C[1]);
                if (CH > 2) {
                    const float2 r2 = *reinterpret_cast<const float2*>(&s_rec[j * 3 + 2]);
                    C[2] = fmaf(r2.x, w, C[2]);
                    if (CH > 3) C[3] = fmaf(r2.y, w, C[3]);
                }
                last = (w > 0.f) ? base + j + 1 : last;
                T = stop ? T : nT;
                Tc = stop ? 0.f : nT;
                if (HITS) {
                    if (__any_sync(FULL, w > 0.f) && lane == 0) hit_any[s_gid[j]] = 1;
                }
            }
        }
    }
    cp_async_wait_all();
    if (inside) {
        const int64_t pix = int64_t(py) * width + px;
        final_T[pix] = T;
        n_contrib[pix] = last;
        if (alpha_out) alpha_out[pix] = 1.0f - T;
#pragma unroll
        for (int c = 0; c < CH; ++c) image[pix * pix_stride + c * ch_stride] = C[c] + (bg ? T * __ldg(bg + c) : 0.f);
    }
}

// ---- backward: transpose-reduce --------------------------------------------------------------------------------------------
// Round 1's kernel reduced nine partial sums per (warp, list entry) with a shuffle butterfly and a single writer lane: 63 of
// its 119 warp instructions per entry (SHFL issues at one warp instruction per clock per SM); measured 0.69 ms at 1 M / 1080p
// against 0.53 ms for this kernel with scalar atomics (profiles/round2_*).  Here each pixel lane only
// produces TWO numbers per entry —  go = dL/d(opacity-weighted Gaussian)  and  fac = alpha*T  — and stores them as one
// float2 into a per-warp shared-memory tile [GE entries][32 lanes].  After GE = 16 entries the roles flip: lane (e, h)
// owns entry e and the 16 pixels of half h of the warp's 8x4 block, reads its row with 128-bit loads (rows are padded by
// 16 B: conflict-free in both directions) and accumulates, in registers and with compile-time pixel coordinates as FFMA
// immediates, the six coordinate moments of go (the mean/conic gradients are linear in them) and the colour sums
// sum(fac * v_image[pixel]) (v_image of the warp's 32 pixels sits in shared memory, read as broadcasts).  One xor-16
// exchange combines the halves; then lane (e, 0) finishes the mean/conic algebra of entry e and issues its 5 atomics
// while lane (e, 1) issues opacity + colours: 16 entries are written by 32 lanes in parallel.  No shuffles in the
// reduction, no serial writer: ~12 instead of 63 instructions per (warp, entry) after the evaluation.
// With the absgrad side channel (gsplat's `means2d.absgrad`, vanilla_density_controller.py:112-113) each pixel stores two more
// values per entry, |dL/dmean2D.x| and |dL/dmean2D.y| of its own sample (they are summed without signs, so they cannot be
// derived from the moments): float4 rows, 3 CTAs per SM instead of 4.
constexpr int GE = 16;                          // list entries per reduction group
constexpr int BWD_LIST = BLOCK_PIX + GE + 8;    // per-warp list: GE dummies in front (reverse walk), 8 behind

template <bool ABS>
struct TrSmem {
    static constexpr int VAL_BYTES = ABS ? 16 : 8;              // per (entry, pixel): {go, fac} or {go, fac, |gx|, |gy|}
    static constexpr int VAL_ROW = 32 * VAL_BYTES + 16;         // bytes per entry row of the value tile (+ pad)
    float4 rec[(BLOCK_PIX + 1) * 3];
    float4 vo[NWARP][33];                                        // v_image of the warp's pixels; pixel p at slot p + (p >> 4): the two halves
                                                                 // of a warp read different banks in the same instruction
    unsigned char val[NWARP][GE * VAL_ROW];
    unsigned short list[NWARP][BWD_LIST];
    unsigned char mask[BLOCK_PIX];
    int wmax[NWARP];
};
static_assert(sizeof(TrSmem<false>) <= 57344, "4 CTAs per SM need <= 56 KB each");

// VROWS: the gradient outputs are the columns of one [n,12] row buffer (include/b200gs.h row layout; v_xy = its base): the nine
// sums of an entry leave as THREE 128-bit reductions (REDG.E.ADD.F32x4: {xy, -, conic0} {conic1, conic2, -, opacity} {rgb, -})
// instead of nine 32-bit ones — a third of the L2 atomic operations, which bound this kernel once the shuffles were gone.
template <int CH, bool GSPLAT, bool ABS, bool VROWS>
__global__ void __launch_bounds__(BLOCK_PIX, ABS ? 3 : 4) blend_bwd_tr_kernel(int width, int height, int grid_x, const int2* __restrict__ ranges,
                                                                    const int32_t* __restrict__ ids, const SplatStrides st, const SplatStrides so,
                                                                    const float* __restrict__ xy, const float* __restrict__ conic,
                                                                    const float* __restrict__ opacity, const float* __restrict__ colors,
                                                                    const float* __restrict__ bg, const float* __restrict__ final_T,
                                                                    const int32_t* __restrict__ n_contrib, const float* __restrict__ v_image,
                                                                    int64_t pix_stride, int64_t ch_stride, const float* __restrict__ v_alpha,
                                                                    float sx, float sy, float* __restrict__ v_xy, float* __restrict__ v_conic,
                                                                    float* __restrict__ v_opacity, float* __restrict__ v_colors,
                                                                    float* __restrict__ v_xy_abs) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef TrSmem<ABS> Smem;
    constexpr int VAL_ROW = Smem::VAL_ROW, VAL_BYTES = Smem::VAL_BYTES;
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    float4* s_rec = sm.rec;

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const unsigned lane = tid & 31u;
    const int tile = (int)blockIdx.x;
    const int tile_y = tile / grid_x, tile_x = tile - tile_y * grid_x;
    int lx, ly;
    pixel_of_thread(tid, lx, ly);
    const int px = tile_x * TILE + lx, py = tile_y * TILE + ly;
    const bool inside = (px < width) && (py < height);
    const float off = GSPLAT ? 0.5f : 0.0f;
    const float pxf = float(px) + off, pyf = float(py) + off;
    const float ox = float(tile_x * TILE) + off, oy = float(tile_y * TILE) + off;
    const float amax = GSPLAT ? 0.999f : 0.99f;
    const int64_t pix = int64_t(py) * width + px;
    if (tid < 3) s_rec[DUMMY * 3 + tid] = make_float4(0.f, 0.f, 0.f, 0.f);

    const int2 range = ranges[tile];
    const float Tf = inside ? final_T[pix] : 0.f;
    const int last = inside ? n_contrib[pix] : 0;
    float vo[4] = {0.f, 0.f, 0.f, 0.f};
    float bg_dot = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        vo[c] = inside ? __ldg(v_image + pix * pix_stride + c * ch_stride) : 0.f;
        if (bg) bg_dot += __ldg(bg + c) * vo[c];
    }
    sm.vo[warp][lane + (lane >> 4)] = make_float4(vo[0], vo[1], vo[2], vo[3]);
    const float va = (v_alpha && inside) ? __ldg(v_alpha + pix) : 0.f;
    const float tail = Tf * (va - bg_dot);  // d(out)/d(alpha_i) through everything behind the last contributor

    const int wmax = __reduce_max_sync(FULL, last);
    if (lane == 0) sm.wmax[warp] = wmax;
    __syncthreads();
    int max_last = 0;
#pragma unroll
    for (int w = 0; w < NWARP; ++w) max_last = max(max_last, sm.wmax[w]);
    if (max_last == 0) return;

    float T = Tf;
    float D = 0.f;   // <colour accumulated behind the current splat, v_image> for this pixel
    unsigned char* my_val = sm.val[warp] + lane * VAL_BYTES;      // eval phase: this pixel's value column
    const int re = lane & (GE - 1), rh = lane >> 4;               // reduce phase: entry and pixel half of this lane
    const float4* my_row = reinterpret_cast<const float4*>(sm.val[warp] + re * VAL_ROW + rh * 16 * VAL_BYTES);
    const float4* my_vo = sm.vo[warp] + rh * 17;
    // origin of the warp's 8x4 block of pixel samples; the reduce lane's pixels are rows 2 rh, 2 rh + 1 of it
    const float bx0 = ox + float((warp & 1) << 3), by0 = oy + float((warp >> 1) << 2);
    const float hh = float(2 * rh);

    for (int hi = max_last; hi > 0; hi -= BLOCK_PIX) {
        const int lo = max(0, hi - BLOCK_PIX);
        const int cnt = hi - lo;
        __syncthreads();
        if (tid < cnt) {
            const int g = __ldg(ids + range.x + lo + tid);
            const float2 m = __ldg(reinterpret_cast<const float2*>(xy + int64_t(g) * st.xs));
            const float* cq = conic + int64_t(g) * st.cs;
            const float A = __ldg(cq), B = __ldg(cq + 1), Cc = __ldg(cq + 2);
            const float o = __ldg(opacity + int64_t(g) * st.os);
            float col[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c = 0; c < CH; ++c) col[c] = __ldg(colors + int64_t(g) * st.ks + c);
            s_rec[tid * 3 + 0] = make_float4(m.x, m.y, (-0.5f * LOG2E) * A, -LOG2E * B);
            s_rec[tid * 3 + 1] = make_float4((-0.5f * LOG2E) * Cc, o, col[0], col[1]);
            s_rec[tid * 3 + 2] = make_float4(col[2], col[3], __int_as_float(g), 0.f);
            sm.mask[tid] = (unsigned char)block_mask(m.x, m.y, A, B, Cc, o, ox, oy);
        }
        __syncthreads();
        if (wmax <= lo) continue;  // this warp has no contributor in the batch
        const unsigned short* my_list = sm.list[warp] + GE;   // my_list[-GE..-1] are DUMMY
        const int nl = build_list<GE>(sm.mask, sm.list[warp], min(cnt, wmax - lo), warp, lane);
        const int rel_last = last - lo;                        // entry j of this batch is in front of the pixel's last contributor iff j < rel_last
        for (int ii = nl - 1; ii >= 0; ii -= GE) {
            unsigned vm = 0;   // bit u: this pixel has a valid sample of list entry ii-u
#pragma unroll
            for (int u = 0; u < GE; ++u) {
                const int j = my_list[ii - u];
                const float4 r0 = s_rec[j * 3 + 0];
                const float4 r1 = s_rec[j * 3 + 1];
                const float dx = r0.x - pxf, dy = r0.y - pyf;
                // same arithmetic as the forward: power * log2(e) = a' dx^2 + b' dx dy + c' dy^2
                const float p2 = fmaf(r1.x * dy, dy, fmaf(r0.w, dy, r0.z * dx) * dx);
                const float G = ex2_approx(p2);
                const float oG = r1.y * G;
                const float a = fminf(amax, oG);
                const bool valid = (j < rel_last) && !(p2 > 0.0f) && (a >= ALPHA_MIN);
                float go = 0.f, fac = 0.f, gax = 0.f, gay = 0.f;
                if (valid) {
                    const float ra = 1.0f / (1.0f - a);
                    T *= ra;
                    fac = a * T;
                    float S = r1.z * vo[0];
                    if (CH > 1) S = fmaf(r1.w, vo[1], S);
                    if (CH > 2) {
                        const float2 r2 = *reinterpret_cast<const float2*>(&s_rec[j * 3 + 2]);
                        S = fmaf(r2.x, vo[2], S);
                        if (CH > 3) S = fmaf(r2.y, vo[3], S);
                    }
                    // dL/dalpha = T <c, v> - (<colour behind, v> + T_final (bg.v - v_alpha)) / (1 - alpha);  D = <colour behind, v>
                    const float v_al = fmaf(T, S, ra * (tail - D));
                    D = fmaf(fac, S, D);
                    if (!GSPLAT || (oG <= 0.999f)) go = G * v_al;
                    vm |= 1u << u;
                    if (ABS) {   // |dL/dmean2D| of this sample: |v_sigma (A dx + B dy)|, |v_sigma (B dx + C dy)|, v_sigma = -opacity * go
                        const float vsg = r1.y * go * (2.0f / LOG2E);
                        gax = fabsf(vsg * fmaf(r0.z, dx, 0.5f * r0.w * dy));
                        gay = fabsf(vsg * fmaf(0.5f * r0.w, dx, r1.x * dy));
                    }
                }
                if (ABS) *reinterpret_cast<float4*>(my_val + u * VAL_ROW) = make_float4(go, fac, gax, gay);
                else *reinterpret_cast<float2*>(my_val + u * VAL_ROW) = make_float2(go, fac);
            }
            const unsigned present = __reduce_or_sync(FULL, vm);
            __syncwarp();   // the tile stores of all lanes are visible to the row loads below
            if (present != 0u) {
                // ---- reduce: lane (re, rh) sums entry ii-re over pixels 16 rh .. 16 rh + 15 (local x = k & 7, local row = k >> 3)
                float R0 = 0.f, R0x = 0.f, R0xx = 0.f, R1 = 0.f, R1x = 0.f, R1xx = 0.f;
                float Cs[4] = {0.f, 0.f, 0.f, 0.f};
                float Ax = 0.f, Ay = 0.f;
#pragma unroll
                for (int k2 = 0; k2 < 8; ++k2) {
                    float4 v;                             // {go, fac} of pixels 2 k2, 2 k2 + 1
                    if (ABS) {
                        const float4 va = my_row[2 * k2], vb = my_row[2 * k2 + 1];
                        v = make_float4(va.x, va.y, vb.x, vb.y);
                        Ax += va.z + vb.z;
                        Ay += va.w + vb.w;
                    } else {
                        v = my_row[k2];
                    }
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int k = 2 * k2 + e;
                        const float gk = e ? v.z : v.x, fk = e ? v.w : v.y;
                        const float x = float(k & 7);
                        if (k < 8) { R0 += gk; if (k & 7) { R0x = fmaf(gk, x, R0x); R0xx = fmaf(gk, x * x, R0xx); } }
                        else       { R1 += gk; if (k & 7) { R1x = fmaf(gk, x, R1x); R1xx = fmaf(gk, x * x, R1xx); } }
                        const float4 w = my_vo[k];
                        Cs[0] = fmaf(fk, w.x, Cs[0]);
                        if (CH > 1) Cs[1] = fmaf(fk, w.y, Cs[1]);
                        if (CH > 2) Cs[2] = fmaf(fk, w.z, Cs[2]);
                        if (CH > 3) Cs[3] = fmaf(fk, w.w, Cs[3]);
                    }
                }
                // moments in block coordinates (x = 0..7, y = 2 rh + {0, 1}), then both halves
                float S0 = R0 + R1, Sx = R0x + R1x, Sxx = R0xx + R1xx;
                float Sy = fmaf(hh, S0, R1), Sxy = fmaf(hh, Sx, R1x), Syy = fmaf(hh * hh, S0, fmaf(2.0f * hh, R1, R1));
                S0 += __shfl_xor_sync(FULL, S0, 16);
                Sx += __shfl_xor_sync(FULL, Sx, 16);
                Sy += __shfl_xor_sync(FULL, Sy, 16);
                Sxx += __shfl_xor_sync(FULL, Sxx, 16);
                Sxy += __shfl_xor_sync(FULL, Sxy, 16);
                Syy += __shfl_xor_sync(FULL, Syy, 16);
#pragma unroll
                for (int c = 0; c < CH; ++c) Cs[c] += __shfl_xor_sync(FULL, Cs[c], 16);
                if (ABS) {
                    Ax += __shfl_xor_sync(FULL, Ax, 16);
                    Ay += __shfl_xor_sync(FULL, Ay, 16);
                }
                if ((present >> re) & 1u) {
                    const int j = my_list[ii - re];
                    const int g = __float_as_int(s_rec[j * 3 + 2].z);
                    if (rh == 0) {
                        const float4 r0 = s_rec[j * 3 + 0];
                        const float4 r1 = s_rec[j * 3 + 1];
                        const float A = r0.z * (-2.0f / LOG2E), B = r0.w * (-1.0f / LOG2E), Cc = r1.x * (-2.0f / LOG2E);
                        const float ex = r0.x - bx0, ey = r0.y - by0;   // dx = ex - x, dy = ey - y
                        const float no = -r1.y;                        // dL/dsigma = -opacity * go
                        const float M1 = no * fmaf(ex, S0, -Sx), M2 = no * fmaf(ey, S0, -Sy);
                        const float M3 = no * fmaf(ex, fmaf(ex, S0, -2.0f * Sx), Sxx);
                        const float M4 = no * (fmaf(ex, fmaf(ey, S0, -Sy), Sxy) - ey * Sx);
                        const float M5 = no * fmaf(ey, fmaf(ey, S0, -2.0f * Sy), Syy);
                        const float gx = (A * M1 + B * M2) * sx, gy = (B * M1 + Cc * M2) * sy;
                        if (VROWS) {
                            float4* row = reinterpret_cast<float4*>(v_xy + int64_t(g) * B200GS_ROW_FLOATS);
                            atomicAdd(row, make_float4(gx, gy, 0.f, 0.5f * M3));
                            atomicAdd(row + 1, make_float4(M4, 0.5f * M5, 0.f, S0));
                        } else {
                            float* vx = v_xy + int64_t(g) * so.xs;
                            float* vc = v_conic + int64_t(g) * so.cs;
                            atomicAdd(vx, gx);
                            atomicAdd(vx + 1, gy);
                            atomicAdd(vc, 0.5f * M3);
                            atomicAdd(vc + 1, M4);
                            atomicAdd(vc + 2, 0.5f * M5);
                        }
                    } else {
                        if (VROWS) {
                            atomicAdd(reinterpret_cast<float4*>(v_xy + int64_t(g) * B200GS_ROW_FLOATS) + 2, make_float4(Cs[0], Cs[1], Cs[2], 0.f));
                        } else {
                            atomicAdd(v_opacity + int64_t(g) * so.os, S0);
#pragma unroll
                            for (int c = 0; c < CH; ++c) atomicAdd(v_colors + int64_t(g) * so.ks + c, Cs[c]);
                        }
                        if (ABS) {
                            atomicAdd(v_xy_abs + 2 * int64_t(g), Ax);
                            atomicAdd(v_xy_abs + 2 * int64_t(g) + 1, Ay);
                        }
                    }
                }
            }
            __syncwarp();   // the rows are read: the next group may overwrite the tile
        }
    }
}

template <int CH>
int fwd_dispatch(int mode, int width, int height, const int32_t* ranges, const int32_t* ids, int row_stride, const float* xy, const float* conic,
                 const float* opacity, const float* colors, const float* bg, float* image, int64_t ps, int64_t cs, float* final_T,
                 int32_t* n_contrib, float* alpha, uint8_t* hit_any, cudaStream_t s) {
    const int gx = div_up(width, TILE), gy = div_up(height, TILE);
    dim3 grid(gx * gy);
    const SplatStrides st = row_stride > 0 ? SplatStrides{row_stride, row_stride, row_stride, row_stride} : SplatStrides{2, 3, 1, CH};
    // Two stagings of the tile slab.  Synchronous: ids -> gathered records -> registers -> shared memory, the latency covered by the other
    // CTAs of the SM.  Asynchronous: cp.async (LDGSTS) double buffer.  Measured at 1 M Gaussians / 1080p on B200 (profiles/round2_*):
    //   first version of the asynchronous kernel (81 registers = 2 blocks per SM)            0.308-0.310 ms   vs synchronous 0.281-0.290 ms
    //   asynchronous kernel capped at 80 registers (3 blocks per SM), [n,12] rows (3 x 16 B)  0.277 ms         vs synchronous 0.290 ms
    // so the asynchronous staging is the default for the row layout (what the fused renderers and the sharded renderer use) and for the
    // has_hit_any_pixels variant; the separate-array layout (eight 4/8-byte LDGSTS per splat) stays synchronous (DESIGN.md §5.4).
    // the row layout is [x, y, depth, A, B, C, comp, opacity, r, g, b, radius] (include/b200gs.h); 16-byte copies need 16-byte aligned rows
    const bool rows16 = row_stride == 12 && CH == 3 && conic == xy + 3 && opacity == xy + 7 && colors == xy + 8 && (reinterpret_cast<uintptr_t>(xy) & 15) == 0;
    if (rows16 || hit_any != nullptr) {
#define B200GS_FWD_ARGS width, height, gx, (const int2*)ranges, ids, st, xy, conic, opacity, colors, bg, image, ps, cs, final_T, n_contrib, alpha, hit_any
#define B200GS_FWD_LAUNCH(G, R)                                                                                                   \
    do {                                                                                                                           \
        if (hit_any) blend_fwd_async_kernel<CH, G, R, true><<<grid, BLOCK_PIX, 0, s>>>(B200GS_FWD_ARGS);                          \
        else blend_fwd_async_kernel<CH, G, R, false><<<grid, BLOCK_PIX, 0, s>>>(B200GS_FWD_ARGS);                                 \
    } while (0)
        if (rows16) {
            if constexpr (CH == 3) {
                if (mode == B200GS_MODE_GSPLAT) B200GS_FWD_LAUNCH(true, true);
                else B200GS_FWD_LAUNCH(false, true);
            }
        } else {
            if (mode == B200GS_MODE_GSPLAT) B200GS_FWD_LAUNCH(true, false);
            else B200GS_FWD_LAUNCH(false, false);
        }
#undef B200GS_FWD_LAUNCH
#undef B200GS_FWD_ARGS
        B200GS_LAUNCH_CHECK();
        return B200GS_OK;
    }
    if (mode == B200GS_MODE_GSPLAT)
        blend_fwd_kernel<CH, true><<<grid, BLOCK_PIX, 0, s>>>(width, height, gx, (const int2*)ranges, ids, st, xy, conic,
                                                              opacity, colors, bg, image, ps, cs, final_T, n_contrib, alpha);
    else
        blend_fwd_kernel<CH, false><<<grid, BLOCK_PIX, 0, s>>>(width, height, gx, (const int2*)ranges, ids, st, xy, conic,
                                                               opacity, colors, bg, image, ps, cs, final_T, n_contrib, alpha);
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

template <int CH>
int bwd_dispatch(int mode, int width, int height, const int32_t* ranges, const int32_t* ids, int row_stride, const float* xy, const float* conic,
                 const float* opacity, const float* colors, const float* bg, const float* final_T, const int32_t* n_contrib,
                 const float* v_image, int64_t ps, int64_t cs, const float* v_alpha, float sx, float sy, float* v_xy,
                 float* v_conic, float* v_opacity, float* v_colors, float* v_xy_abs, cudaStream_t s) {
    const int gx = div_up(width, TILE), gy = div_up(height, TILE);
    dim3 grid(gx * gy);
    const SplatStrides st = row_stride > 0 ? SplatStrides{row_stride, row_stride, row_stride, row_stride} : SplatStrides{2, 3, 1, CH};
    const SplatStrides so = st;   // the gradients have the layout of the inputs
    // gradient outputs that are the columns of one 16-byte aligned [n,12] row buffer leave as 128-bit reductions
    const bool vrows = CH == 3 && row_stride == B200GS_ROW_FLOATS && v_conic == v_xy + B200GS_ROW_CONIC && v_opacity == v_xy + B200GS_ROW_OPACITY &&
                       v_colors == v_xy + B200GS_ROW_RGB && (reinterpret_cast<uintptr_t>(v_xy) & 15) == 0;
#define B200GS_BWD_ARGS width, height, gx, (const int2*)ranges, ids, st, so, xy, conic, opacity, colors, bg, final_T, n_contrib, \
                        v_image, ps, cs, v_alpha, sx, sy, v_xy, v_conic, v_opacity, v_colors, v_xy_abs
    static const cudaError_t attr_rc = []() {
        cudaError_t e = cudaSuccess;
        auto set = [&e](const void* f, size_t bytes) {
            if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        };
        set((const void*)blend_bwd_tr_kernel<CH, true, false, false>, sizeof(TrSmem<false>));
        set((const void*)blend_bwd_tr_kernel<CH, false, false, false>, sizeof(TrSmem<false>));
        set((const void*)blend_bwd_tr_kernel<CH, true, true, false>, sizeof(TrSmem<true>));
        set((const void*)blend_bwd_tr_kernel<CH, false, true, false>, sizeof(TrSmem<true>));
        if constexpr (CH == 3) {
            set((const void*)blend_bwd_tr_kernel<CH, true, false, true>, sizeof(TrSmem<false>));
            set((const void*)blend_bwd_tr_kernel<CH, false, false, true>, sizeof(TrSmem<false>));
        }
        return e;
    }();
    if (attr_rc != cudaSuccess) {
        set_error("blend_bwd: cudaFuncSetAttribute failed: %s", cudaGetErrorString(attr_rc));
        return B200GS_ECUDA;
    }
#define B200GS_BWD_LAUNCH(G, A, V) blend_bwd_tr_kernel<CH, G, A, V><<<grid, BLOCK_PIX, sizeof(TrSmem<A>), s>>>(B200GS_BWD_ARGS)
    const bool gs = mode == B200GS_MODE_GSPLAT, ab = v_xy_abs != nullptr;
    if (vrows) {
        if constexpr (CH == 3) {   // the row entry point has no absgrad output
            if (gs) B200GS_BWD_LAUNCH(true, false, true);
            else B200GS_BWD_LAUNCH(false, false, true);
        }
    } else {
        if (gs) { if (ab) B200GS_BWD_LAUNCH(true, true, false); else B200GS_BWD_LAUNCH(true, false, false); }
        else    { if (ab) B200GS_BWD_LAUNCH(false, true, false); else B200GS_BWD_LAUNCH(false, false, false); }
    }
#undef B200GS_BWD_LAUNCH
#undef B200GS_BWD_ARGS
    B200GS_LAUNCH_CHECK();
    return B200GS_OK;
}

}  // namespace

int launch_blend_fwd(int mode, int width, int height, int channels, const int32_t* ranges, const int32_t* ids, int row_stride, const float* xy,
                     const float* conic, const float* opacity, const float* colors, const float* bg, float* image,
                     int64_t pix_stride, int64_t ch_stride, float* final_T, int32_t* n_contrib, float* alpha, cudaStream_t s,
                     uint8_t* hit_any) {
    switch (channels) {
        case 1: return fwd_dispatch<1>(mode, width, height, ranges, ids, row_stride, xy, conic, opacity, colors, bg, image, pix_stride, ch_stride, final_T, n_contrib, alpha, hit_any, s);
        case 2: return fwd_dispatch<2>(mode, width, height, ranges, ids, row_stride, xy, conic, opacity, colors, bg, image, pix_stride, ch_stride, final_T, n_contrib, alpha, hit_any, s);
        case 3: return fwd_dispatch<3>(mode, width, height, ranges, ids, row_stride, xy, conic, opacity, colors, bg, image, pix_stride, ch_stride, final_T, n_contrib, alpha, hit_any, s);
        case 4: return fwd_dispatch<4>(mode, width, height, ranges, ids, row_stride, xy, conic, opacity, colors, bg, image, pix_stride, ch_stride, final_T, n_contrib, alpha, hit_any, s);
    }
    set_error("blend_fwd: unsupported channel count %d (1..4)", channels);
    return B200GS_EINVAL;
}

int launch_blend_bwd(int mode, int width, int height, int channels, const int32_t* ranges, const int32_t* ids, int row_stride, const float* xy,
                     const float* conic, const float* opacity, const float* colors, const float* bg, const float* final_T,
                     const int32_t* n_contrib, const float* v_image, int64_t pix_stride, int64_t ch_stride, const float* v_alpha,
                     float sx, float sy, float* v_xy, float* v_conic, float* v_opacity, float* v_colors, float* v_xy_abs,
                     cudaStream_t s) {
#define B200GS_BWD_CALL(C) bwd_dispatch<C>(mode, width, height, ranges, ids, row_stride, xy, conic, opacity, colors, bg, final_T, n_contrib, v_image, \
                                           pix_stride, ch_stride, v_alpha, sx, sy, v_xy, v_conic, v_opacity, v_colors, v_xy_abs, s)
    switch (channels) {
        case 1: return B200GS_BWD_CALL(1);
        case 2: return B200GS_BWD_CALL(2);
        case 3: return B200GS_BWD_CALL(3);
        case 4: return B200GS_BWD_CALL(4);
    }
#undef B200GS_BWD_CALL
    set_error("blend_bwd: unsupported channel count %d (1..4)", channels);
    return B200GS_EINVAL;
}

}  // namespace b200gs
