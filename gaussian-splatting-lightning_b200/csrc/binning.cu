// K2-K5: tile binning.
//
// The reference backends sort I (tile,Gaussian) pairs on a 64-bit (tile | depth-bits) key: ~6 radix passes over
// 12 B pairs (SURVEY §8d: I*152 B, the largest pure-bandwidth term of their forward).  The same total order — tile
// major, then depth bits, ties in Gaussian-id order — is produced here hierarchically, and the fine pairs are written
// exactly once, already in place:
//   A. depth keys (32-bit float bits; off-screen -> 0xFFFFFFFF), stable radix sort of the N keys, scan of the
//      per-Gaussian COARSE cell counts in depth order (a coarse cell = 8x8 tiles = 128x128 px); a 32-byte record per
//      Gaussian (one L2 sector) holds everything phase B needs
//   B. emit (coarse cell, {64-bit tile mask, id}) pairs in depth order — the mask = which of the cell's 64 tiles the splat
//      can reach (row spans of the alpha >= 1/255 ellipse, or the plain 3-sigma rect with culling off) — and
//      stable-partition them by cell: ONE 8-bit radix pass over ~2 pairs per visible Gaussian for every image up to
//      2048x2048 (<= 256 cells)
//   C. per 256-entry chunk of a cell's list: per-tile counts (warp bit-matrix transpose + popcount)
//   D. per cell: prefix of the chunk counts; one scan over the tiles -> tile_ranges and the pair total
//   E. every chunk writes its splat ids to sorted_ids at (tile start + chunk prefix + rank inside the chunk), ranks
//      from the transposed bit sets in list order, staged so that every run is one coalesced store
// A stable multi-split keeps the depth order inside every tile, so the result equals the oracle's torch.sort(stable)
// of the 64-bit keys element for element (tests/test_gpu_parity.py::test_binning_exact).
//
// Every kernel here is ours, including the device-wide primitives (onesweep.cuh: chained scan, onesweep radix passes):
//   phase A  depth_keys (order-preserving compaction of the visible Gaussians through a chained scan; {depth key, id} records
//            + the 32-byte record)  ->  hist4  ->  4 onesweep passes over the V visible records
//   phase B  emit_cells (chained scan of the coarse-cell counts in depth order; per-cell histogram)  ->  cell_table (cell
//            ranges, chunk table, digit histograms)  ->  1 onesweep pass by cell (2 above 256 cells)  ->  chunk_counts  ->
//            chunk_prefix  ->  scatter_ids
#include "common.cuh"
#include "onesweep.cuh"

namespace b200gs {

namespace {

constexpr int SUPER_SHIFT = 3;             // coarse cell = 8 x 8 tiles
constexpr int SUPER = 1 << SUPER_SHIFT;
constexpr int CELL_TILES = SUPER * SUPER;  // 64: one bit per tile in a uint64_t mask
constexpr int CHUNK = 256;                 // list entries per block of the count / scatter kernels

// What phase B needs to know about a Gaussian, packed by phase A into ONE 32-byte L2 sector (phase B visits the
// Gaussians in depth order, i.e. at random addresses).
struct __align__(16) SplatRec {
    float x, y, A, B, C, opacity;
    int32_t radius, ncells;
};
static_assert(sizeof(SplatRec) == 32, "SplatRec must be one sector");

// value type of the coarse partition: {tile mask lo, tile mask hi, Gaussian id, unused}
typedef uint4 CellEntry;

constexpr int DEPTH_IPT = 8;                         // records per thread of a depth-sort tile (uint2: 4096 per tile, 32 KB of staging)
constexpr int CELL_IPT = 4;                          // records per thread of a cell-partition tile (uint4: 2048 per tile, 32 KB of staging)
constexpr int DEPTH_TILE = sweep::PASS_THREADS * DEPTH_IPT;
constexpr int CELL_TILE = sweep::PASS_THREADS * CELL_IPT;

struct LayoutA {
    size_t rec_a, rec_b, recs, zero, zero_bytes, hist, tickets, scan_state, lookback, total;
    int64_t tiles, blocks;
};
struct LayoutB {
    size_t entries_in, entries, offsets, zero, zero_bytes, cell_hist, tickets, scan_state, lookback, digit_hist, cell_ranges, chunk_base, chunk_cell,
        chunk_cnt, chunk_pre, tile_start, total;
    int64_t max_chunks, tiles, blocks, scan_blocks;
};

inline int bits_for(int n_values) {
    int b = 1;
    while ((1 << b) < n_values) ++b;
    return b;
}

struct Taker {
    size_t off = 0;
    size_t operator()(size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    }
};

LayoutA make_layout_a(int64_t n) {
    static thread_local int64_t cached_n = -1;
    static thread_local LayoutA cached{};
    if (n == cached_n) return cached;
    LayoutA L{};
    Taker take;
    const size_t nn = (size_t)(n > 0 ? n : 1);
    L.tiles = (int64_t)div_up64((int64_t)nn, DEPTH_TILE);
    L.blocks = (int64_t)div_up64((int64_t)nn, 256 * 8);      // depth_keys_kernel: 256 threads x DK_ITEMS Gaussians
    L.rec_a = take(nn * 8);
    L.rec_b = take(nn * 8);
    L.recs = take(nn * sizeof(SplatRec));
    // one contiguous zero-initialised region: digit histograms, tickets, chained-scan state, look-back words of the 4 passes
    L.zero = take(0);
    L.hist = take(4 * sweep::RADIX * 4);
    L.tickets = take(16 * 4);
    L.scan_state = take((size_t)L.blocks * 4);
    L.lookback = take((size_t)4 * L.tiles * sweep::RADIX * 4);
    L.zero_bytes = take.off - L.zero;
    L.total = take.off;
    cached = L;
    cached_n = n;
    return L;
}

// The sort payload is the Gaussian id; when the id fits 24 bits and a rect can cover at most 255 coarse cells, the cell count of the
// rect rides in the top byte ({key, ncells << 24 | id}): rank_offsets then reads its counts from the sorted records it streams through
// anyway instead of gathering one random 32-byte sector per rank (0.65 M L2 requests = most of that kernel's 21 us).  Decided from
// (n, width, height) alone, so bin_count and bin_sort agree.
inline bool pack_ncells(int64_t n, int width, int height) {
    const int gx = div_up(width, TILE), gy = div_up(height, TILE);
    const int cells = div_up(gx, 1 << 3) * div_up(gy, 1 << 3);
    return n < (int64_t(1) << 24) && cells <= 255;
}
constexpr uint32_t ID_MASK = (1u << 24) - 1u;

inline void cell_grid(int width, int height, int& grid_x, int& grid_y, int& cgrid_x, int& cgrid_y) {
    grid_x = div_up(width, TILE);
    grid_y = div_up(height, TILE);
    cgrid_x = div_up(grid_x, SUPER);
    cgrid_y = div_up(grid_y, SUPER);
}

LayoutB make_layout_b(int64_t n, int64_t max_coarse, int width, int height) {
    static thread_local int64_t cached_p = -1, cached_n = -1;
    static thread_local int cached_w = -1, cached_h = -1;
    static thread_local LayoutB cached{};
    if (max_coarse == cached_p && n == cached_n && width == cached_w && height == cached_h) return cached;
    int grid_x, grid_y, cgrid_x, cgrid_y;
    cell_grid(width, height, grid_x, grid_y, cgrid_x, cgrid_y);
    const size_t n_cells = (size_t)cgrid_x * cgrid_y, n_tiles = (size_t)grid_x * grid_y;
    LayoutB L{};
    Taker take;
    const size_t pp = (size_t)(max_coarse > 0 ? max_coarse : 1);
    L.max_chunks = (int64_t)(pp / CHUNK + n_cells + 1);
    L.tiles = (int64_t)div_up64((int64_t)pp, CELL_TILE);
    L.blocks = (int64_t)div_up64(n > 0 ? n : 1, 256);
    L.scan_blocks = (int64_t)div_up64(n > 0 ? n : 1, 256 * 8);   // rank_offsets_kernel: 256 threads x RO_ITEMS ranks
    L.entries_in = take(pp * sizeof(CellEntry));
    L.entries = take(pp * sizeof(CellEntry));
    L.offsets = take((size_t)(n > 0 ? n : 1) * 4);
    L.zero = take(0);
    L.cell_hist = take(n_cells * 4);
    L.tickets = take(16 * 4);
    L.scan_state = take((size_t)L.scan_blocks * 4);
    L.lookback = take((size_t)2 * L.tiles * sweep::RADIX * 4);
    L.zero_bytes = take.off - L.zero;
    L.digit_hist = take(2 * sweep::RADIX * 4);
    L.cell_ranges = take(n_cells * 8);
    L.chunk_base = take((n_cells + 1) * 4);
    L.chunk_cell = take((size_t)L.max_chunks * 4);
    L.chunk_cnt = take((size_t)L.max_chunks * CELL_TILES * 2);
    L.chunk_pre = take((size_t)L.max_chunks * CELL_TILES * 4);
    L.tile_start = take(n_tiles * 8);
    L.total = take.off;
    cached = L;
    cached_p = max_coarse;
    cached_n = n;
    cached_w = width;
    cached_h = height;
    return cached;
}

// ---- exact tile culling ------------------------------------------------------------------------------------------------
// A (tile, splat) pair can only contribute if some pixel sample p of the tile has alpha = o * exp(-q(p - mu)) >= 1/255,
// q(d) = (A dx^2 + C dy^2)/2 + B dx dy, i.e. if the tile's box of pixel samples meets the ellipse E = {q <= ln(255 o)}.
// E and a tile ROW (a band of 16 sample rows) are convex, so the tiles of that row that meet E are exactly those whose
// sample columns meet the x-extent of (E ∩ band): one interval per row, from two clamped evaluations of the ellipse's
// left/right boundary.  Cost O(rows) per Gaussian instead of O(tiles); every pair dropped would have been skipped by
// the blend loop at all 256 pixels, so images and gradients are bit-identical while the pair list (staging, blend
// evaluations) shrinks ~1.8x on the benchmark scene.  The test only has to be conservative: the threshold carries a
// relative margin of 1e-4 (+1e-3), the interval a 0.01 px slack — orders of magnitude above the error of the
// approximate sqrt used here and of the fp32 / ex2.approx rounding of the blend loop.  Each pair's verdict is computed
// exactly once (emit_cells_kernel) and travels with the pair, so no two kernels ever have to agree on it.
// Per-Gaussian inputs of phase A, with element strides: separate contiguous arrays ({2,1,1,3,1}) or columns of one
// [n,12] row buffer ({12,12,12,12,12}).
struct BinSrc {
    const float* xy; const float* depth; const int32_t* radii; const float* conic; const float* opacity;
    int xs, ds, rs, cs, os;
    // rows that arrive in fixed-size blocks (the sharded exchange): block b holds blk_cnt[b] valid rows, the rest of its blk_rows
    // rows is stale memory and reads as culled — no padding pass over the receive buffer
    const int64_t* blk_cnt; int blk_rows;
    __device__ __forceinline__ float2 get_xy(int64_t i) const { return *reinterpret_cast<const float2*>(xy + i * xs); }
    __device__ __forceinline__ float get_depth(int64_t i) const { return depth[i * ds]; }
    __device__ __forceinline__ int get_radius(int64_t i) const {
        if (blk_cnt != nullptr) {
            const int b = (int)i / blk_rows;
            if ((int)i - b * blk_rows >= (int)blk_cnt[b]) return 0;
        }
        return radii[i * rs];
    }
};

struct CullE {
    float mx, my, B, iA, two_tA, det, ymax, yR;
    int mode;  // 0: full rect (culling off / degenerate conic), 1: spans, 2: nothing visible (opacity <= 1/255)
};

__device__ __forceinline__ CullE make_cull(const SplatRec& r, bool cull) {
    CullE e;
    e.mx = r.x; e.my = r.y;
    e.B = 0.f; e.iA = 1.f; e.two_tA = 0.f; e.det = 1.f; e.ymax = 0.f; e.yR = 0.f;
    e.mode = 0;
    if (!cull) return e;
    const float A = r.A, B = r.B, C = r.C;
    const float o255 = 255.0f * r.opacity;
    if (o255 <= 1.0f) { e.mode = 2; return e; }
    // alpha >= 1/255  <=>  q <= ln(255 o); margin covers every rounding here and in the blend loop
    const float t = __logf(o255) * 1.0001f + 1e-3f;
    const float det = A * C - B * B;
    if (!(det > 0.f) || !(A > 0.f) || !(C > 0.f) || !(t < 3.0e38f)) return e;  // degenerate / NaN: keep the full rect
    const float idet = __frcp_rn(det);
    e.B = B; e.iA = __frcp_rn(A);
    e.two_tA = 2.0f * t * A;
    e.det = det;
    e.ymax = __fsqrt_rn(e.two_tA * idet);
    const float xext = __fsqrt_rn(2.0f * t * C * idet);
    e.yR = -B * xext * __frcp_rn(C);  // the ellipse's rightmost point sits at y = yR, leftmost at -yR
    e.mode = 1;
    return e;
}

__device__ __forceinline__ float sqrt_fast(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// tiles [a, b) of tile row ty (clipped to [x0, x1)) whose pixel samples can meet the ellipse
template <bool GSPLAT>
__device__ __forceinline__ bool row_span(const CullE& e, int ty, int x0, int x1, int& a, int& b) {
    a = x0; b = x1;
    if (e.mode == 0) return true;
    const float off = GSPLAT ? 0.5f : 0.0f;
    const float Y0 = float(ty * TILE) + off - e.my;
    const float ya = fmaxf(Y0, -e.ymax), yb = fminf(Y0 + float(TILE - 1), e.ymax);
    if (ya > yb) { b = a; return false; }
    const float yr = fminf(yb, fmaxf(ya, e.yR)), yl = fminf(yb, fmaxf(ya, -e.yR));
    const float dr = sqrt_fast(fmaxf(0.f, e.two_tA - e.det * yr * yr));
    const float dl = sqrt_fast(fmaxf(0.f, e.two_tA - e.det * yl * yl));
    const float xr = (dr - e.B * yr) * e.iA;    // right end of E ∩ band (relative to mu)
    const float xl = (-e.B * yl - dl) * e.iA;   // left end
    // tile tx holds sample columns [16 tx + off, 16 tx + off + 15]
    const float inv = 1.0f / float(TILE);
    const float fa = ceilf((xl + e.mx - (off + float(TILE - 1) + 0.01f)) * inv);
    const float fb = floorf((xr + e.mx - off + 0.01f) * inv);
    if (!(fa <= fb)) {  // also catches NaN
        if (fa == fa && fb == fb) { b = a; return false; }
        return true;    // NaN: keep the whole row
    }
    a = max(x0, (int)fmaxf(fa, -1.0e9f));
    b = min(x1, (int)fminf(fb, 1.0e9f) + 1);
    if (a >= b) { b = a; return false; }
    return true;
}

// tile rect -> rect of coarse cells
__device__ __forceinline__ void coarsen_rect(int x0, int y0, int x1, int y1, int& cx0, int& cy0, int& cx1, int& cy1) {
    cx0 = x0 >> SUPER_SHIFT;
    cy0 = y0 >> SUPER_SHIFT;
    cx1 = ((x1 - 1) >> SUPER_SHIFT) + 1;
    cy1 = ((y1 - 1) >> SUPER_SHIFT) + 1;
}

// Phase A, blocks in ticket order, 2048 consecutive Gaussians per block (the chained scan advances 32..128 blocks per round trip to
// L2, so its length in BLOCKS is what bounds the kernel's latency — profiles/round2b: 53 us with 256-Gaussian blocks).  The block
// walks its Gaussians in DK_ITEMS STRIPED rounds (round k, thread t: Gaussian 256 k + t), so every load and the 32-byte record
// stores are coalesced (the first version gave each thread 8 consecutive Gaussians: 384-byte lane stride, 32 sectors per request).
// The visible Gaussians (non-empty tile rect) are compacted in index order into {depth key, id} records: rank = visible Gaussians
// of the rounds before (per-(round, warp) ballot counts, one 64-entry scan) + lanes below in the own ballot + the chained scan over
// the blocks.  Each visible Gaussian gets the 32-byte record phase B works from (indexed by Gaussian id: written right away); the
// histograms of the four key bytes (what the radix passes start from) are accumulated on the way — the two high bytes, which take
// only a handful of values in a scene, with warp-aggregated increments (match.any), the low bytes with plain shared-memory atomics.
// counts[0] += tiles of the rect (the reference's pair count I: an upper bound of the culled count, exact without culling),
// counts[1] += coarse cells, counts[3] = V.
constexpr int DK_ITEMS = 8;

// ROWS16: the inputs are the columns of one 16-byte aligned [n,12] row buffer (b200gs.h row layout): three 128-bit loads per Gaussian
template <bool GSPLAT, bool ROWS16>
__global__ void __launch_bounds__(256) depth_keys_kernel(int64_t n, int grid_x, int grid_y, int pack, const BinSrc src, uint2* __restrict__ keyrec,
                                                         SplatRec* __restrict__ recs, uint32_t* __restrict__ ticket,
                                                         uint32_t* __restrict__ scan_state, uint32_t* __restrict__ hist,
                                                         unsigned long long* __restrict__ counts) {
    __shared__ unsigned long long s_area[8], s_cells[8];
    __shared__ int s_cnt[DK_ITEMS * 8];      // visible Gaussians of (round, warp); then their exclusive scan
    __shared__ int s_tile;
    __shared__ uint32_t s_excl;
    __shared__ uint32_t s_h[4][sweep::RADIX];
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    for (int i = threadIdx.x; i < 4 * sweep::RADIX; i += 256) (&s_h[0][0])[i] = 0;
    __syncthreads();
    const int t = s_tile;
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const int64_t base_i = int64_t(t) * (256 * DK_ITEMS) + threadIdx.x;
    unsigned long long area_sum = 0, cell_sum = 0;
    uint32_t key[DK_ITEMS];
    uint32_t hi8[DK_ITEMS];          // pack: the rect's cell count << 24 (rides in the top byte of the sort payload), else 0
    unsigned vis_bits = 0;           // bit k: this thread's Gaussian of round k is visible
    unsigned below[DK_ITEMS];        // visible lanes below this one in round k's ballot
#pragma unroll
    for (int k = 0; k < DK_ITEMS; ++k) {
        const int64_t i = base_i + k * 256;
        key[k] = 0xFFFFFFFFu;
        hi8[k] = 0u;
        bool vis = false;
        if (i < n) {
            float px, py, dep, A = 1.f, B = 0.f, C = 1.f, o = 1.f;
            int r;
            if (ROWS16) {
                const float4* row = reinterpret_cast<const float4*>(src.xy + i * B200GS_ROW_FLOATS);
                const float4 q0 = row[0], q1 = row[1], q2 = row[2];
                px = q0.x; py = q0.y; dep = q0.z; A = q0.w; B = q1.x; C = q1.y; o = q1.w;
                r = __float_as_int(q2.w);
                if (src.blk_cnt != nullptr) {
                    const int b = (int)i / src.blk_rows;
                    if ((int)i - b * src.blk_rows >= (int)src.blk_cnt[b]) r = 0;
                }
            } else {
                r = src.get_radius(i);
                const float2 pp = src.get_xy(i);
                px = pp.x; py = pp.y;
                dep = src.get_depth(i);
                if (src.conic != nullptr) {
                    const float* q = src.conic + i * src.cs;
                    A = q[0]; B = q[1]; C = q[2];
                    o = src.opacity[i * src.os];
                }
            }
            if (r > 0) {
                int x0, y0, x1, y1;
                tile_rect<GSPLAT>(px, py, (float)r, grid_x, grid_y, x0, y0, x1, y1);
                const int area = max(0, x1 - x0) * max(0, y1 - y0);
                if (area > 0) {
                    int cx0, cy0, cx1, cy1;
                    coarsen_rect(x0, y0, x1, y1, cx0, cy0, cx1, cy1);
                    const int ncell = (cx1 - cx0) * (cy1 - cy0);
                    key[k] = __float_as_uint(dep);
                    hi8[k] = pack ? ((uint32_t)ncell << 24) : 0u;
                    area_sum += (unsigned long long)area;
                    cell_sum += (unsigned long long)ncell;
                    vis = true;
                    float4* out = reinterpret_cast<float4*>(recs + i);
                    out[0] = make_float4(px, py, A, B);
                    out[1] = make_float4(C, o, __int_as_float(r), __int_as_float(ncell));
                }
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, vis);
        below[k] = __popc(bal & ((1u << lane) - 1u));
        vis_bits |= vis ? (1u << k) : 0u;
        if (lane == 0) s_cnt[k * 8 + w] = __popc(bal);
        // byte histograms: bytes 3 and 2 (few distinct values per scene) warp-aggregated, bytes 1 and 0 with plain atomics
        const unsigned grp = __match_any_sync(0xffffffffu, vis ? (key[k] >> 16) : 0xFFFFFFFFu);
        if (vis) {
            if ((grp & ((1u << lane) - 1u)) == 0u) atomicAdd(&s_h[2][(key[k] >> 16) & 255u], (uint32_t)__popc(grp));
            atomicAdd(&s_h[1][(key[k] >> 8) & 255u], 1u);
            atomicAdd(&s_h[0][key[k] & 255u], 1u);
        }
        const unsigned grp3 = __match_any_sync(0xffffffffu, vis ? (key[k] >> 24) : 0xFFFFFFFFu);
        if (vis && (grp3 & ((1u << lane) - 1u)) == 0u) atomicAdd(&s_h[3][key[k] >> 24], (uint32_t)__popc(grp3));
    }
    __syncthreads();
    if (threadIdx.x < 32) {     // warp 0: scan of the 64 (round, warp) counts, then the warp-wide look-back over the preceding blocks
        const int c0 = s_cnt[2 * lane], c1 = s_cnt[2 * lane + 1];
        int inc = c0 + c1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o);
            if ((int)lane >= o) inc += v;
        }
        const int block_vis = __shfl_sync(0xffffffffu, inc, 31);
        s_cnt[2 * lane] = inc - c0 - c1;
        s_cnt[2 * lane + 1] = inc - c1;
        const uint32_t excl = sweep::chained_exclusive(scan_state, t, (uint32_t)block_vis);
        if (threadIdx.x == 0) {
            s_excl = excl;
            if (t == (int)gridDim.x - 1) counts[3] = (unsigned long long)(excl + (uint32_t)block_vis);
        }
    }
    __syncthreads();
    const uint32_t base = s_excl;
#pragma unroll
    for (int k = 0; k < DK_ITEMS; ++k) {
        if (!((vis_bits >> k) & 1u)) continue;
        keyrec[base + (uint32_t)s_cnt[k * 8 + w] + below[k]] = make_uint2(key[k], (uint32_t)(base_i + k * 256) | hi8[k]);
    }
    unsigned long long a = area_sum, c = cell_sum;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if ((threadIdx.x & 31) == 0) { s_area[threadIdx.x >> 5] = a; s_cells[threadIdx.x >> 5] = c; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long ta = 0, tc = 0;
#pragma unroll
        for (int w2 = 0; w2 < 8; ++w2) { ta += s_area[w2]; tc += s_cells[w2]; }
        if (ta) atomicAdd(counts, ta);
        if (tc) atomicAdd(counts + 1, tc);
    }
    for (int i = threadIdx.x; i < 4 * sweep::RADIX; i += 256) {
        const uint32_t v = (&s_h[0][0])[i];
        if (v) atomicAdd(hist + i, v);
    }
}

// Exclusive prefix of the coarse-cell counts over the depth-ranked Gaussians: offsets[rank] = first entry slot of that rank.  Big
// tiles (RO_ITEMS consecutive ranks per thread) for the same reason as above; the cell count of a rank is gathered from its record.
constexpr int RO_ITEMS = 8;

__global__ void __launch_bounds__(256) rank_offsets_kernel(const int64_t* __restrict__ d_visible, int pack, const uint2* __restrict__ order,
                                                          const SplatRec* __restrict__ recs, uint32_t* __restrict__ offsets,
                                                          uint32_t* __restrict__ ticket, uint32_t* __restrict__ scan_state) {
    __shared__ int s_scan[sweep::WARPS + 1];
    __shared__ int s_tile;
    __shared__ uint32_t s_excl;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int t = s_tile;
    const int64_t n = *d_visible;
    const int64_t r0 = (int64_t(t) * blockDim.x + threadIdx.x) * RO_ITEMS;
    if (int64_t(t) * blockDim.x * RO_ITEMS >= n) return;
    int nc[RO_ITEMS];
    int mine = 0;
#pragma unroll
    for (int k = 0; k < RO_ITEMS; ++k) {
        nc[k] = 0;
        if (r0 + k < n) {
            const uint32_t y = order[r0 + k].y;
            nc[k] = pack ? (int)(y >> 24) : __ldg(&recs[y].ncells);
        }
        mine += nc[k];
    }
    int block_total;
    int local = sweep::block_exclusive(mine, s_scan, &block_total);
    if (threadIdx.x < 32) {
        const uint32_t excl = sweep::chained_exclusive(scan_state, t, (uint32_t)block_total);
        if (threadIdx.x == 0) s_excl = excl;
    }
    __syncthreads();
    uint32_t run = s_excl + (uint32_t)local;
#pragma unroll
    for (int k = 0; k < RO_ITEMS; ++k) {
        if (r0 + k < n) offsets[r0 + k] = run;
        run += (uint32_t)nc[k];
    }
}

// Phase B, one block (in ticket order) per 256 depth-ranked Gaussians: emits their (coarse cell, {tile mask, id}) entries, cells
// in row-major order.  The first slot of a rank is the exclusive prefix of the cell counts in depth order: block scan +
// chained scan over the blocks, so the block's ranks own one contiguous window of the entry array; the entries are
// assembled in shared memory and written back with coalesced stores.  The expensive part — one ellipse/row-band
// intersection per tile row of every rect — is spread over the block as (rank, row) work items, so a warp never waits
// for the one lane that owns a large splat.  The block also counts its entries per cell (the histogram the partition and
// the cell ranges are derived from).
constexpr int EMIT_SLOTS = 2048;
constexpr int EMIT_ITEMS = 2048;  // (rank, row) work items resolved through a table instead of a binary search
constexpr int EMIT_HIST = 1024;   // cells counted in shared memory (images up to 4096 x 4096); larger grids count straight in global memory

template <bool GSPLAT>
__global__ void __launch_bounds__(256) emit_cells_kernel(const int64_t* __restrict__ d_visible, int pack, int grid_x, int grid_y, int cgrid_x, int cull,
                                                         int64_t max_coarse, const uint2* __restrict__ order, const SplatRec* __restrict__ recs,
                                                         const uint32_t* __restrict__ offsets, CellEntry* __restrict__ entries, int n_cells,
                                                         uint32_t* __restrict__ cell_hist) {
    __shared__ unsigned short s_k[EMIT_SLOTS];
    __shared__ int32_t s_id[EMIT_SLOTS];
    __shared__ unsigned long long s_mask[EMIT_SLOTS];
    __shared__ float s_f[8][256];        // mx, my, B, iA, two_tA, det, ymax, yR
    __shared__ int s_mode[256], s_xr[256], s_yr[256], s_start[256];   // x0 | x1 << 16, y0 | y1 << 16, first slot - block_lo
    __shared__ int s_rowoff[260];
    __shared__ unsigned char s_item[EMIT_ITEMS];   // work item -> rank of the block (when the block has <= EMIT_ITEMS tile rows)
    __shared__ int s_warp[8];
    __shared__ uint32_t s_hist[EMIT_HIST];
    const int tid = threadIdx.x;
    const unsigned lane = tid & 31u, w = tid >> 5;
    const int64_t n = *d_visible;
    const int64_t rank0 = int64_t(blockIdx.x) * blockDim.x;
    if (rank0 >= n) return;
    const bool smem_hist = n_cells <= EMIT_HIST;
    if (smem_hist)
        for (int i = tid; i < n_cells; i += 256) s_hist[i] = 0;
    const int64_t rnk = rank0 + tid;
    int g = -1, x0 = 0, y0 = 0, x1 = 0, y1 = 0, t = 0, nrows = 0;
    CullE e{};
    if (rnk < n) {
        g = (int)(pack ? (order[rnk].y & ID_MASK) : order[rnk].y);
        const float4* rp = reinterpret_cast<const float4*>(recs + g);
        const float4 r0 = __ldg(rp), r1 = __ldg(rp + 1);
        SplatRec rec;
        rec.x = r0.x; rec.y = r0.y; rec.A = r0.z; rec.B = r0.w; rec.C = r1.x; rec.opacity = r1.y;
        rec.radius = __float_as_int(r1.z); rec.ncells = __float_as_int(r1.w);
        t = rec.ncells;
        if (t > 0) {
            tile_rect<GSPLAT>(rec.x, rec.y, (float)rec.radius, grid_x, grid_y, x0, y0, x1, y1);
            e = make_cull(rec, cull != 0);
            nrows = (e.mode == 2) ? 0 : y1 - y0;
        }
    }
    // first slot of this rank = cells of the ranks before it (rank_offsets_kernel); the block's ranks own one contiguous window
    const int64_t block_lo = (int64_t)offsets[rank0];
    const int64_t last_rank = min(rank0 + (int64_t)blockDim.x, n) - 1;
    const uint32_t last_y = order[last_rank].y;
    const int block_cells = (int)((int64_t)offsets[last_rank] + (pack ? (int)(last_y >> 24) : __ldg(&recs[last_y].ncells)) - block_lo);
    const int local_start = (rnk < n) ? (int)((int64_t)offsets[rnk] - block_lo) : block_cells;
    // exclusive scan of the row counts
    int inc = nrows;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if ((int)lane >= o) inc += v;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    int wbase = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) wbase += (k < (int)w) ? s_warp[k] : 0;
    __syncthreads();   // every warp has read s_warp before anything below is stored (racecheck, round 2: a slow warp's read of
                       // s_warp raced with the stores that follow in a fast warp)
    s_rowoff[tid] = wbase + inc - nrows;
    if (tid == 255) s_rowoff[256] = wbase + inc;
    s_f[0][tid] = e.mx; s_f[1][tid] = e.my; s_f[2][tid] = e.B; s_f[3][tid] = e.iA;
    s_f[4][tid] = e.two_tA; s_f[5][tid] = e.det; s_f[6][tid] = e.ymax; s_f[7][tid] = e.yR;
    s_mode[tid] = e.mode;
    s_xr[tid] = x0 | (x1 << 16);
    s_yr[tid] = y0 | (y1 << 16);
    s_start[tid] = local_start;
    const int cx0 = x0 >> SUPER_SHIFT, cy0 = y0 >> SUPER_SHIFT;
    const int cw = t > 0 ? ((x1 - 1) >> SUPER_SHIFT) - cx0 + 1 : 1;
    __syncthreads();
    const int total_rows = s_rowoff[256];
    const bool item_table = total_rows <= EMIT_ITEMS;
    if (item_table) {     // rank tid owns items [s_rowoff[tid], s_rowoff[tid] + nrows)
        const int o = s_rowoff[tid];
        for (int k = 0; k < nrows; ++k) s_item[o + k] = (unsigned char)tid;
    }                     // visible to the item loop after the barrier that follows the cell/id stores below
    const int64_t block_hi = min(block_lo + block_cells, max_coarse);
    for (int64_t lo = block_lo; lo < block_hi; lo += EMIT_SLOTS) {
        const int cn = (int)min((int64_t)EMIT_SLOTS, block_hi - lo);
        const int wlo = (int)(lo - block_lo);       // window = local slots [wlo, wlo + cn)
        for (int i = tid; i < cn; i += 256) s_mask[i] = 0ull;
        // cells and ids of this rank's slots
        {
            const int ls = local_start;
            int k = max(0, wlo - ls);
            const int kend = min(t, wlo + cn - ls);
            int cy = cy0 + k / cw, cx = cx0 + k % cw;
            for (; k < kend; ++k) {
                const int cell = cy * cgrid_x + cx;
                s_k[ls + k - wlo] = (unsigned short)cell;
                s_id[ls + k - wlo] = g;
                if (smem_hist) atomicAdd(&s_hist[cell], 1u); else atomicAdd(cell_hist + cell, 1u);
                if (++cx == cx0 + cw) { cx = cx0; ++cy; }
            }
        }
        __syncthreads();
        // (rank, row) work items
        for (int it = tid; it < total_rows; it += 256) {
            int r = 0;
            if (item_table) {
                r = s_item[it];
            } else {
#pragma unroll
                for (int step = 128; step >= 1; step >>= 1)
                    if (s_rowoff[r + step] <= it) r += step;
            }
            CullE q;
            q.mx = s_f[0][r]; q.my = s_f[1][r]; q.B = s_f[2][r]; q.iA = s_f[3][r];
            q.two_tA = s_f[4][r]; q.det = s_f[5][r]; q.ymax = s_f[6][r]; q.yR = s_f[7][r];
            q.mode = s_mode[r];
            const int xr = s_xr[r], yr = s_yr[r];
            const int rx0 = xr & 0xffff, rx1 = xr >> 16, ry0 = yr & 0xffff;
            const int ty = ry0 + (it - s_rowoff[r]);
            int a, b;
            if (!row_span<GSPLAT>(q, ty, rx0, rx1, a, b)) continue;
            const int rcx0 = rx0 >> SUPER_SHIFT, rcw = ((rx1 - 1) >> SUPER_SHIFT) - rcx0 + 1;
            const int row_slot = s_start[r] + ((ty >> SUPER_SHIFT) - (ry0 >> SUPER_SHIFT)) * rcw - rcx0 - wlo;
            for (int cx = a >> SUPER_SHIFT; cx <= (b - 1) >> SUPER_SHIFT; ++cx) {
                const int slot = row_slot + cx;
                if (slot < 0 || slot >= cn) continue;
                const int wx0 = cx << SUPER_SHIFT;
                const int ca = max(a, wx0) - wx0, cb = min(b, wx0 + SUPER) - wx0;
                const unsigned bits = ((1u << (cb - ca)) - 1u) << ca;
                reinterpret_cast<unsigned char*>(s_mask)[slot * 8 + (ty & (SUPER - 1))] = (unsigned char)bits;
            }
        }
        __syncthreads();
        for (int i = tid; i < cn; i += 256) {
            const unsigned long long m = s_mask[i];
            entries[lo + i] = make_uint4((uint32_t)m, (uint32_t)(m >> 32), (uint32_t)s_id[i], (uint32_t)s_k[i]);
        }
        __syncthreads();
    }
    if (smem_hist)
        for (int i = tid; i < n_cells; i += 256) {
            const uint32_t c = s_hist[i];
            if (c) atomicAdd(cell_hist + i, c);
        }
}

// One block, after the emit: from the per-cell entry counts -> cell ranges (exclusive scan), the chunk table
// (chunk_base[c] = number of CHUNK-entry chunks of the cells before c; chunk_cell[chunk] = its cell), the digit histograms
// of the partition passes (low / high byte of the cell id), zeroed tile totals.
__global__ void __launch_bounds__(1024) cell_table_kernel(int n_cells, const uint32_t* __restrict__ cell_hist, int2* __restrict__ cell_ranges,
                                                          int32_t* __restrict__ chunk_base, int32_t* __restrict__ chunk_cell,
                                                          uint32_t* __restrict__ digit_hist, int n_tiles, int64_t* __restrict__ tile_total) {
    __shared__ int s_warp[32], s_warp2[32];
    __shared__ int s_carry, s_carry2;
    __shared__ uint32_t s_dh[2][sweep::RADIX];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) { s_carry = 0; s_carry2 = 0; }
    for (int i = tid; i < 2 * sweep::RADIX; i += 1024) (&s_dh[0][0])[i] = 0;
    __syncthreads();
    for (int base = 0; base < n_cells; base += 1024) {
        const int i = base + tid;
        int cnt = 0, v = 0;
        if (i < n_cells) {
            cnt = (int)cell_hist[i];
            v = (cnt + CHUNK - 1) / CHUNK;
            if (cnt) { atomicAdd(&s_dh[0][i & 255], (uint32_t)cnt); atomicAdd(&s_dh[1][(i >> 8) & 255], (uint32_t)cnt); }
        }
        int inc = v, inc2 = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            const int t2 = __shfl_up_sync(0xffffffffu, inc2, o);
            if (lane >= o) { inc += t; inc2 += t2; }
        }
        if (lane == 31) { s_warp[w] = inc; s_warp2[w] = inc2; }
        __syncthreads();
        if (w == 0) {
            int ws = s_warp[lane], winc = ws, ws2 = s_warp2[lane], winc2 = ws2;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, winc, o);
                const int t2 = __shfl_up_sync(0xffffffffu, winc2, o);
                if (lane >= o) { winc += t; winc2 += t2; }
            }
            s_warp[lane] = winc - ws;
            s_warp2[lane] = winc2 - ws2;
        }
        __syncthreads();
        const int excl = s_carry + s_warp[w] + inc - v;
        const int excl2 = s_carry2 + s_warp2[w] + inc2 - cnt;
        if (i < n_cells) {
            chunk_base[i] = excl;
            cell_ranges[i] = cnt > 0 ? make_int2(excl2, excl2 + cnt) : make_int2(0, 0);
        }
        __syncthreads();
        if (tid == 1023) { s_carry = excl + v; s_carry2 = excl2 + cnt; }
        __syncthreads();
    }
    const int total = s_carry;
    if (tid == 0) chunk_base[n_cells] = total;
    for (int i = tid; i < 2 * sweep::RADIX; i += 1024) digit_hist[i] = (&s_dh[0][0])[i];
    for (int i = tid; i < n_tiles; i += 1024) tile_total[i] = 0;    // accumulated by chunk_counts_kernel
    __syncthreads();                                                // chunk_base (written by this block) is visible
    __shared__ int s_cb[1024];                                      // chunk_base of up to 1024 cells (images up to 4096 x 4096): the
    const bool in_smem = n_cells <= 1024;                           // binary search below is a chain of dependent loads per chunk
    if (in_smem) {
        if (tid < n_cells) s_cb[tid] = chunk_base[tid];
        __syncthreads();
    }
    for (int c = tid; c < total; c += 1024) {
        int lo = 0, hi = n_cells;   // invariant: chunk_base[lo] <= c < chunk_base[hi]; cells without entries own no chunk
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((in_smem ? s_cb[mid] : chunk_base[mid]) <= c) lo = mid; else hi = mid;
        }
        chunk_cell[c] = lo;
    }
}

// 32x32 bit-matrix transpose across a warp: lane l passes row l, lane t receives column t
// (bit l of the result = bit t of lane l's input).
__device__ __forceinline__ uint32_t transpose32(uint32_t x, unsigned lane) {
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
        const uint32_t m = (j == 16) ? 0x0000FFFFu : (j == 8) ? 0x00FF00FFu : (j == 4) ? 0x0F0F0F0Fu : (j == 2) ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
        x = (lane & j) ? ((x & ~m) | ((y >> j) & m)) : ((x & m) | ((y << j) & ~m));
    }
    return x;
}

// Phase C: one block per chunk (256 consecutive entries of one cell's depth-ordered list): per-tile entry counts.
// Each warp transposes the masks of its 32 entries: lane t then holds, for tiles t and t+32, the bit set of the warp's
// entries that reach the tile.
__global__ void __launch_bounds__(CHUNK) chunk_counts_kernel(int n_cells, int cgrid_x, int grid_x, int grid_y, const int2* __restrict__ cell_ranges,
                                                             const int32_t* __restrict__ chunk_base, const int32_t* __restrict__ chunk_cell,
                                                             const CellEntry* __restrict__ entries, uint16_t* __restrict__ chunk_cnt,
                                                             int64_t* __restrict__ tile_total) {
    __shared__ uint16_t s_cnt[CHUNK / 32][CELL_TILES];
    const int c = blockIdx.x;
    if (c >= __ldg(chunk_base + n_cells)) return;
    const int cell = __ldg(chunk_cell + c);
    const int2 r = cell_ranges[cell];
    const int e = r.x + (c - __ldg(chunk_base + cell)) * CHUNK + (int)threadIdx.x;
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    uint32_t lo = 0, hi = 0;
    if (e < r.y) {
        const uint2 m = __ldg(reinterpret_cast<const uint2*>(entries + e));
        lo = m.x; hi = m.y;
    }
    s_cnt[w][lane] = (uint16_t)__popc(transpose32(lo, lane));
    s_cnt[w][lane + 32] = (uint16_t)__popc(transpose32(hi, lane));
    __syncthreads();
    if (threadIdx.x < CELL_TILES) {
        int sum = 0;
#pragma unroll
        for (int k = 0; k < CHUNK / 32; ++k) sum += s_cnt[k][threadIdx.x];
        chunk_cnt[int64_t(c) * CELL_TILES + threadIdx.x] = (uint16_t)sum;
        const int t = threadIdx.x;
        const int tx = ((cell % cgrid_x) << SUPER_SHIFT) + (t & (SUPER - 1));
        const int ty = ((cell / cgrid_x) << SUPER_SHIFT) + (t >> SUPER_SHIFT);
        if (sum > 0 && tx < grid_x && ty < grid_y)
            atomicAdd(reinterpret_cast<unsigned long long*>(tile_total + int64_t(ty) * grid_x + tx), (unsigned long long)sum);
    }
}

// Phase D.  Blocks [0, n_cells): thread (j, t) of a cell's block computes the prefix over the cell's chunks of tile t's
// counts, the chunk list split into 16 contiguous parts j so that the sequential walks stay short.  Block n_cells, at the
// same time: exclusive scan of the tile totals (accumulated by chunk_counts_kernel) in tile-id order, in place -> tile
// starts; tile_ranges (clamped to the capacity of sorted_ids; empty tiles (0,0) like dgr's zero-filled ranges); counts[2].
__global__ void __launch_bounds__(1024) chunk_prefix_kernel(int n_cells, int n_tiles, const int32_t* __restrict__ chunk_base,
                                                            const uint16_t* __restrict__ chunk_cnt, uint32_t* __restrict__ chunk_pre,
                                                            int64_t* __restrict__ tile_start, int64_t max_pairs,
                                                            int2* __restrict__ tile_ranges, int64_t* __restrict__ d_counts) {
    __shared__ uint32_t s_part[16][CELL_TILES];
    __shared__ int64_t s_warp[32];
    __shared__ int64_t s_carry;
    const int tid = threadIdx.x;
    if ((int)blockIdx.x < n_cells) {
        const int cell = blockIdx.x;
        const int t = tid & (CELL_TILES - 1), j = tid >> 6;
        const int c0 = chunk_base[cell], c1 = chunk_base[cell + 1];
        const int per = (c1 - c0 + 15) >> 4;
        const int a = min(c1, c0 + j * per), b = min(c1, a + per);
        // the walk is a chain of dependent L2 round trips unless the loads are issued together: up to PRE_REG counts per thread live in
        // registers (all loads in flight at once, read once), longer parts fall back to the two-pass loop
        constexpr int PRE_REG = 16;
        uint32_t sum = 0;
        if (per <= PRE_REG) {
            uint32_t v[PRE_REG];
#pragma unroll
            for (int q = 0; q < PRE_REG; ++q) v[q] = (a + q < b) ? (uint32_t)chunk_cnt[int64_t(a + q) * CELL_TILES + t] : 0u;
#pragma unroll
            for (int q = 0; q < PRE_REG; ++q) sum += v[q];
            s_part[j][t] = sum;
            __syncthreads();
            uint32_t run = 0;
            for (int k = 0; k < j; ++k) run += s_part[k][t];
#pragma unroll
            for (int q = 0; q < PRE_REG; ++q) {
                if (a + q < b) chunk_pre[int64_t(a + q) * CELL_TILES + t] = run;
                run += v[q];
            }
            return;
        }
#pragma unroll 4
        for (int c = a; c < b; ++c) sum += chunk_cnt[int64_t(c) * CELL_TILES + t];
        s_part[j][t] = sum;
        __syncthreads();
        uint32_t run = 0;
        for (int k = 0; k < j; ++k) run += s_part[k][t];
#pragma unroll 4
        for (int c = a; c < b; ++c) {
            const uint32_t v = chunk_cnt[int64_t(c) * CELL_TILES + t];
            chunk_pre[int64_t(c) * CELL_TILES + t] = run;
            run += v;
        }
        return;
    }
    if (tid == 0) s_carry = 0;
    __syncthreads();
    const int lane = tid & 31, w = tid >> 5;
    for (int base = 0; base < n_tiles; base += 8192) {
        const int i0 = base + tid * 8;
        int64_t v[8];
        if (i0 + 8 <= n_tiles) {
            const longlong2* p = reinterpret_cast<const longlong2*>(tile_start + i0);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const longlong2 q = p[k];
                v[2 * k] = q.x; v[2 * k + 1] = q.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = (i0 + k < n_tiles) ? tile_start[i0 + k] : 0;
        }
        int64_t sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) sum += v[k];
        int64_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_warp[w] = inc;
        __syncthreads();
        if (w == 0) {
            const int64_t ws = s_warp[lane];
            int64_t winc = ws;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t t = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += t;
            }
            s_warp[lane] = winc - ws;
        }
        __syncthreads();
        int64_t run = s_carry + s_warp[w] + inc - sum;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (i0 + k < n_tiles) {
                tile_start[i0 + k] = run;
                tile_ranges[i0 + k] = v[k] > 0 ? make_int2((int)min(run, max_pairs), (int)min(run + v[k], max_pairs)) : make_int2(0, 0);
            }
            run += v[k];
        }
        __syncthreads();
        if (tid == 1023) s_carry = run;
        __syncthreads();
    }
    if (tid == 0) d_counts[2] = s_carry;
}

// Phase E: one block per chunk; sorted_ids[tile start + chunk prefix + rank in chunk] = id.  After the warp transpose,
// lane t owns the bit sets of tiles t / t+32 over the warp's 32 entries; walking their set bits in order yields the
// tile's ids in list order.  The chunk's output is first laid out in shared memory in (tile, rank) order — the order it
// has in global memory, where tile t's part is one contiguous run — so each run leaves the SM as one coalesced store
// instead of one partial-sector write per id.
constexpr int SCATTER_STAGE = 4096;

__global__ void __launch_bounds__(CHUNK) scatter_ids_kernel(int n_cells, int cgrid_x, int grid_x, int grid_y, int64_t max_pairs,
                                                            const int2* __restrict__ cell_ranges, const int32_t* __restrict__ chunk_base,
                                                            const int32_t* __restrict__ chunk_cell, const CellEntry* __restrict__ entries,
                                                            const uint32_t* __restrict__ chunk_pre, const int64_t* __restrict__ tile_start,
                                                            int32_t* __restrict__ sorted_ids) {
    constexpr int WARPS = CHUNK / 32;
    __shared__ uint16_t s_cnt[WARPS][CELL_TILES];
    __shared__ int s_wbase[WARPS][CELL_TILES];    // offset of (warp, tile) inside the tile's run of this chunk
    __shared__ int s_off[CELL_TILES + 1];         // offset of tile t's run inside the staged output
    __shared__ int64_t s_gbase[CELL_TILES];       // global position of tile t's run
    __shared__ int32_t s_id[CHUNK];
    __shared__ int32_t s_out[SCATTER_STAGE];
    const int c = blockIdx.x;
    if (c >= __ldg(chunk_base + n_cells)) return;
    const unsigned lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const int cell = __ldg(chunk_cell + c);
    const int2 r = cell_ranges[cell];
    const int e = r.x + (c - __ldg(chunk_base + cell)) * CHUNK + (int)threadIdx.x;
    uint32_t mlo = 0, mhi = 0;
    if (e < r.y) {
        const uint4 v = __ldg(entries + e);
        mlo = v.x; mhi = v.y;
        s_id[threadIdx.x] = (int)v.z;
    }
    uint32_t wlo = transpose32(mlo, lane), whi = transpose32(mhi, lane);   // entries of this warp reaching tile lane / lane + 32
    s_cnt[w][lane] = (uint16_t)__popc(wlo);
    s_cnt[w][lane + 32] = (uint16_t)__popc(whi);
    __syncthreads();
    if (threadIdx.x < CELL_TILES) {
        const int t = threadIdx.x;
        const int tx = ((cell % cgrid_x) << SUPER_SHIFT) + (t & (SUPER - 1));
        const int ty = ((cell / cgrid_x) << SUPER_SHIFT) + (t >> SUPER_SHIFT);
        s_gbase[t] = (tx < grid_x && ty < grid_y) ? tile_start[int64_t(ty) * grid_x + tx] + chunk_pre[int64_t(c) * CELL_TILES + t] : 0;
        int run = 0;
#pragma unroll
        for (int k = 0; k < WARPS; ++k) {
            s_wbase[k][t] = run;
            run += s_cnt[k][t];
        }
        int inc = run;   // inclusive scan of the tile totals inside each of the two warps
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o);
            if ((int)lane >= o) inc += v;
        }
        s_off[t + 1] = inc;
    }
    __syncthreads();
    const int half = s_off[32];       // total of tiles 0..31
    __syncthreads();
    if (threadIdx.x >= 32 && threadIdx.x < CELL_TILES) s_off[threadIdx.x + 1] += half;
    if (threadIdx.x == 0) s_off[0] = 0;
    __syncthreads();
    const int total = s_off[CELL_TILES];
    const int32_t* ids = s_id + w * 32;
    if (total <= SCATTER_STAGE) {
        int p = s_off[lane] + s_wbase[w][lane];
        for (; wlo; wlo &= wlo - 1) s_out[p++] = ids[__ffs(wlo) - 1];
        p = s_off[lane + 32] + s_wbase[w][lane + 32];
        for (; whi; whi &= whi - 1) s_out[p++] = ids[__ffs(whi) - 1];
        __syncthreads();
        for (int t = (int)w; t < CELL_TILES; t += WARPS) {     // warp w flushes the runs of tiles w, w+8, ...
            const int o = s_off[t], len = s_off[t + 1] - o;
            const int64_t gb = s_gbase[t];
            for (int k = (int)lane; k < len; k += 32)
                if (gb + k < max_pairs) sorted_ids[gb + k] = s_out[o + k];
        }
    } else {   // a chunk of very large splats: write straight to global memory
        int64_t p = s_gbase[lane] + s_wbase[w][lane];
        for (; wlo; wlo &= wlo - 1, ++p)
            if (p < max_pairs) sorted_ids[p] = ids[__ffs(wlo) - 1];
        p = s_gbase[lane + 32] + s_wbase[w][lane + 32];
        for (; whi; whi &= whi - 1, ++p)
            if (p < max_pairs) sorted_ids[p] = ids[__ffs(whi) - 1];
    }
}

}  // namespace

size_t bin_count_workspace_bytes(int64_t n) { return make_layout_a(n).total; }
size_t bin_sort_workspace_bytes(int64_t n, int64_t max_coarse, int width, int height) { return make_layout_b(n, max_coarse, width, height).total; }

static BinSrc make_src(int row_stride, const float* xy, const float* depth, const int32_t* radii, const float* conic, const float* opacity,
                       const int64_t* block_counts, int64_t block_rows) {
    if (block_rows <= 0) block_counts = nullptr;
    if (row_stride > 0)
        return BinSrc{xy, depth, radii, conic, opacity, row_stride, row_stride, row_stride, row_stride, row_stride, block_counts, (int)block_rows};
    return BinSrc{xy, depth, radii, conic, opacity, 2, 1, 1, 3, 1, block_counts, (int)block_rows};
}

// Counter read-back.  For pinned (mapped) host memory the counters are PUBLISHED by a kernel with system-scope stores
// instead of a cudaMemcpyAsync: an in-stream D2H copy is serviced by a copy engine, and queues behind whatever bulk
// transfer the application has in flight on it (e.g. the H2D prefetch of the next training image) — which would stall
// the whole forward behind a 32-byte copy.  Pageable host memory falls back to the copy.
__global__ void publish_counts_kernel(const int64_t* __restrict__ d_counts, volatile int64_t* __restrict__ host_counts) {
    if (threadIdx.x < 4) host_counts[threadIdx.x] = d_counts[threadIdx.x];
    __threadfence_system();
}

__global__ void publish_i64_kernel(const int64_t* __restrict__ src, volatile int64_t* __restrict__ dst, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    __threadfence_system();
}

static int copy_counts(const int64_t* d_counts, int64_t* host_counts, int sync_host, cudaStream_t s) {
    if (host_counts != nullptr) {
        cudaPointerAttributes attr{};
        const cudaError_t e = cudaPointerGetAttributes(&attr, host_counts);
        if (e == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer != nullptr) {
            publish_counts_kernel<<<1, 32, 0, s>>>(d_counts, (volatile int64_t*)attr.devicePointer);
            B200GS_LAUNCH_CHECK();
        } else {
            (void)cudaGetLastError();
            B200GS_CUDA(cudaMemcpyAsync(host_counts, d_counts, 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        }
        if (sync_host) B200GS_CUDA(cudaStreamSynchronize(s));
    }
    return B200GS_OK;
}

int publish_i64(const int64_t* d_values, int64_t* host_values, int n, cudaStream_t s) {
    cudaPointerAttributes attr{};
    const cudaError_t e = cudaPointerGetAttributes(&attr, host_values);
    if (e == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer != nullptr) {
        publish_i64_kernel<<<1, 64, 0, s>>>(d_values, (volatile int64_t*)attr.devicePointer, n);
        B200GS_LAUNCH_CHECK();
    } else {
        (void)cudaGetLastError();
        B200GS_CUDA(cudaMemcpyAsync(host_values, d_values, sizeof(int64_t) * (size_t)n, cudaMemcpyDeviceToHost, s));
    }
    return B200GS_OK;
}

int bin_count(int mode, int width, int height, int64_t n, int row_stride, const float* xy, const float* depth, const int32_t* radii,
              const float* conic, const float* opacity, void* ws, size_t ws_bytes, int64_t* d_counts, int64_t* host_counts,
              int sync_host, cudaStream_t s, const int64_t* block_counts, int64_t block_rows) {
    const LayoutA L = make_layout_a(n);
    if (ws_bytes < L.total) {
        set_error("bin_count: workspace too small (%zu < %zu)", ws_bytes, L.total);
        return B200GS_ENOSPACE;
    }
    if (n >= (int64_t(1) << 30)) {
        set_error("bin_count: %lld Gaussians exceed the 2^30 limit of the look-back words", (long long)n);
        return B200GS_ENOSPACE;
    }
    char* w = (char*)ws;
    uint2* rec_a = (uint2*)(w + L.rec_a);
    uint2* rec_b = (uint2*)(w + L.rec_b);
    SplatRec* recs = (SplatRec*)(w + L.recs);
    uint32_t* hist = (uint32_t*)(w + L.hist);
    uint32_t* tickets = (uint32_t*)(w + L.tickets);
    uint32_t* scan_state = (uint32_t*)(w + L.scan_state);
    uint32_t* lookback = (uint32_t*)(w + L.lookback);
    const int grid_x = div_up(width, TILE), grid_y = div_up(height, TILE);
    B200GS_CUDA(cudaMemsetAsync(d_counts, 0, 4 * sizeof(int64_t), s));
    if (n > 0) {
        B200GS_CUDA(cudaMemsetAsync(w + L.zero, 0, L.zero_bytes, s));
        const unsigned blocks = (unsigned)L.blocks;
        const BinSrc src = make_src(row_stride, xy, depth, radii, conic, opacity, block_counts, block_rows);
        // all five inputs are columns of one 16-byte aligned [n,12] row buffer -> 128-bit row loads
        const bool rows16 = row_stride == B200GS_ROW_FLOATS && conic != nullptr && depth == xy + B200GS_ROW_DEPTH && conic == xy + B200GS_ROW_CONIC &&
                            opacity == xy + B200GS_ROW_OPACITY && reinterpret_cast<const float*>(radii) == xy + B200GS_ROW_RADIUS &&
                            (reinterpret_cast<uintptr_t>(xy) & 15) == 0;
        const int pack = pack_ncells(n, width, height) ? 1 : 0;
#define B200GS_DK_LAUNCH(G, R) depth_keys_kernel<G, R><<<blocks, 256, 0, s>>>(n, grid_x, grid_y, pack, src, rec_a, recs, tickets, scan_state, hist, (unsigned long long*)d_counts)
        if (mode == B200GS_MODE_GSPLAT) { if (rows16) B200GS_DK_LAUNCH(true, true); else B200GS_DK_LAUNCH(true, false); }
        else                            { if (rows16) B200GS_DK_LAUNCH(false, true); else B200GS_DK_LAUNCH(false, false); }
#undef B200GS_DK_LAUNCH
        B200GS_LAUNCH_CHECK();
        // stable LSD sort of the V visible {depth key, id} records (V = d_counts[3], known on the device only; byte histograms from above)
        const int64_t* d_visible = d_counts + 3;
        uint2* src_rec = rec_a;
        uint2* dst_rec = rec_b;
        for (int pass = 0; pass < 4; ++pass) {
            sweep::onesweep_pass_kernel<uint2, DEPTH_IPT><<<(unsigned)L.tiles, sweep::PASS_THREADS, 0, s>>>(
                src_rec, dst_rec, d_visible, n, 8 * pass, hist + pass * sweep::RADIX, lookback + (size_t)pass * L.tiles * sweep::RADIX, tickets + 1 + pass);
            B200GS_LAUNCH_CHECK();
            uint2* tmp = src_rec; src_rec = dst_rec; dst_rec = tmp;
        }
        // 4 passes: the sorted records are back in rec_a
    }
    return copy_counts(d_counts, host_counts, sync_host, s);
}

int bin_sort(int mode, int width, int height, int64_t n, int cull, int64_t max_coarse, int64_t max_pairs, int64_t* d_counts,
             const void* ws_a, void* ws_b, size_t ws_bytes, int32_t* sorted_ids, int32_t* tile_ranges, int64_t* host_counts,
             int sync_host, cudaStream_t s) {
    int grid_x, grid_y, cgrid_x, cgrid_y;
    cell_grid(width, height, grid_x, grid_y, cgrid_x, cgrid_y);
    const int n_tiles = grid_x * grid_y, n_cells = cgrid_x * cgrid_y;
    if (max_pairs >= (int64_t(1) << 30) || max_coarse >= (int64_t(1) << 30)) {
        set_error("bin_sort: capacity %lld / %lld exceeds 2^30", (long long)max_coarse, (long long)max_pairs);
        return B200GS_ENOSPACE;
    }
    if (n_cells > 65536) {
        set_error("bin_sort: %d coarse cells exceed 65536 (image too large)", n_cells);
        return B200GS_ENOSPACE;
    }
    if (max_coarse == 0 || n == 0) {   // nothing on screen (or nothing can be stored): empty lists; counts[2] stays 0
        B200GS_CUDA(cudaMemsetAsync(tile_ranges, 0, sizeof(int32_t) * 2 * (size_t)n_tiles, s));
        return copy_counts(d_counts, host_counts, sync_host, s);
    }
    const LayoutA LA = make_layout_a(n);
    const LayoutB L = make_layout_b(n, max_coarse, width, height);
    if (ws_bytes < L.total) {
        set_error("bin_sort: workspace too small (%zu < %zu)", ws_bytes, L.total);
        return B200GS_ENOSPACE;
    }
    const char* wa = (const char*)ws_a;
    char* w = (char*)ws_b;
    const uint2* order = (const uint2*)(wa + LA.rec_a);
    const SplatRec* recs = (const SplatRec*)(wa + LA.recs);
    CellEntry* entries_in = (CellEntry*)(w + L.entries_in);
    CellEntry* entries = (CellEntry*)(w + L.entries);
    uint32_t* offsets = (uint32_t*)(w + L.offsets);
    uint32_t* cell_hist = (uint32_t*)(w + L.cell_hist);
    uint32_t* tickets = (uint32_t*)(w + L.tickets);
    uint32_t* scan_state = (uint32_t*)(w + L.scan_state);
    uint32_t* lookback = (uint32_t*)(w + L.lookback);
    uint32_t* digit_hist = (uint32_t*)(w + L.digit_hist);
    int2* cell_ranges = (int2*)(w + L.cell_ranges);
    int32_t* chunk_base = (int32_t*)(w + L.chunk_base);
    int32_t* chunk_cell = (int32_t*)(w + L.chunk_cell);
    uint16_t* chunk_cnt = (uint16_t*)(w + L.chunk_cnt);
    uint32_t* chunk_pre = (uint32_t*)(w + L.chunk_pre);
    int64_t* tile_start = (int64_t*)(w + L.tile_start);
    const int64_t* d_visible = d_counts + 3;
    const int64_t* d_coarse = d_counts + 1;

    // B: coarse entries with their tile masks in depth order; per-cell counts
    B200GS_CUDA(cudaMemsetAsync(w + L.zero, 0, L.zero_bytes, s));
    const bool two_pass = n_cells > sweep::RADIX;
    CellEntry* emit_dst = two_pass ? entries : entries_in;   // one pass: in -> entries; two passes: entries -> in -> entries
    const int pack = pack_ncells(n, width, height) ? 1 : 0;
    rank_offsets_kernel<<<(unsigned)L.scan_blocks, 256, 0, s>>>(d_visible, pack, order, recs, offsets, tickets, scan_state);
    B200GS_LAUNCH_CHECK();
    if (mode == B200GS_MODE_GSPLAT)
        emit_cells_kernel<true><<<(unsigned)L.blocks, 256, 0, s>>>(d_visible, pack, grid_x, grid_y, cgrid_x, cull, max_coarse, order, recs, offsets, emit_dst,
                                                                    n_cells, cell_hist);
    else
        emit_cells_kernel<false><<<(unsigned)L.blocks, 256, 0, s>>>(d_visible, pack, grid_x, grid_y, cgrid_x, cull, max_coarse, order, recs, offsets, emit_dst,
                                                                     n_cells, cell_hist);
    B200GS_LAUNCH_CHECK();
    cell_table_kernel<<<1, 1024, 0, s>>>(n_cells, cell_hist, cell_ranges, chunk_base, chunk_cell, digit_hist, n_tiles, tile_start);
    B200GS_LAUNCH_CHECK();
    // stable partition by cell: one onesweep pass per byte of the cell id (the entry carries its cell in .w)
    if (two_pass) {
        sweep::onesweep_pass_kernel<CellEntry, CELL_IPT><<<(unsigned)L.tiles, sweep::PASS_THREADS, 0, s>>>(entries, entries_in, d_coarse, max_coarse, 0, digit_hist,
                                                                                                      lookback, tickets + 1);
        B200GS_LAUNCH_CHECK();
        sweep::onesweep_pass_kernel<CellEntry, CELL_IPT><<<(unsigned)L.tiles, sweep::PASS_THREADS, 0, s>>>(
            entries_in, entries, d_coarse, max_coarse, 8, digit_hist + sweep::RADIX, lookback + (size_t)L.tiles * sweep::RADIX, tickets + 2);
    } else {
        sweep::onesweep_pass_kernel<CellEntry, CELL_IPT><<<(unsigned)L.tiles, sweep::PASS_THREADS, 0, s>>>(entries_in, entries, d_coarse, max_coarse, 0, digit_hist,
                                                                                                      lookback, tickets + 1);
    }
    B200GS_LAUNCH_CHECK();

    // C: per-chunk tile counts;  D: chunk prefixes, tile starts / ranges / total;  E: ids in place
    const unsigned chunks = (unsigned)L.max_chunks;
    chunk_counts_kernel<<<chunks, CHUNK, 0, s>>>(n_cells, cgrid_x, grid_x, grid_y, cell_ranges, chunk_base, chunk_cell, entries, chunk_cnt, tile_start);
    B200GS_LAUNCH_CHECK();
    chunk_prefix_kernel<<<(unsigned)n_cells + 1, 1024, 0, s>>>(n_cells, n_tiles, chunk_base, chunk_cnt, chunk_pre, tile_start, max_pairs,
                                                               (int2*)tile_ranges, d_counts);
    B200GS_LAUNCH_CHECK();
    scatter_ids_kernel<<<chunks, CHUNK, 0, s>>>(n_cells, cgrid_x, grid_x, grid_y, max_pairs, cell_ranges, chunk_base, chunk_cell, entries, chunk_pre,
                                                tile_start, sorted_ids);
    B200GS_LAUNCH_CHECK();
    return copy_counts(d_counts, host_counts, sync_host, s);
}

// ---- row packing for the Gaussian-sharded exchange -------------------------------------------------------------------
namespace {

// scan[i] = number of entries with radius > 0 before i: block scan + chained scan over the blocks (ticket order).  VS_ITEMS
// consecutive entries per thread: the chained scan's latency is its length in BLOCKS (round 2, N = 2: with 256-entry blocks the
// 11.7 k blocks of a 3 M-entry scan made this kernel most of a 0.41 ms pack stage).
constexpr int VS_ITEMS = 8;

__global__ void __launch_bounds__(256) visible_scan_kernel(int64_t n, const int32_t* __restrict__ radii, int32_t* __restrict__ scan,
                                                           uint32_t* __restrict__ ticket, uint32_t* __restrict__ state) {
    __shared__ int s_scan[sweep::WARPS + 1];
    __shared__ int s_tile;
    __shared__ uint32_t s_excl;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int t = s_tile;
    const int64_t i0 = (int64_t(t) * blockDim.x + threadIdx.x) * VS_ITEMS;
    int vis[VS_ITEMS];
    int mine = 0;
    const bool vec = i0 + VS_ITEMS <= n && (reinterpret_cast<uintptr_t>(radii) & 15u) == 0;    // i0 is a multiple of 8
    if (vec) {
        const int4 a = __ldg(reinterpret_cast<const int4*>(radii + i0)), b = __ldg(reinterpret_cast<const int4*>(radii + i0) + 1);
        vis[0] = a.x > 0; vis[1] = a.y > 0; vis[2] = a.z > 0; vis[3] = a.w > 0;
        vis[4] = b.x > 0; vis[5] = b.y > 0; vis[6] = b.z > 0; vis[7] = b.w > 0;
    } else {
#pragma unroll
        for (int k = 0; k < VS_ITEMS; ++k) vis[k] = (i0 + k < n && radii[i0 + k] > 0) ? 1 : 0;
    }
#pragma unroll
    for (int k = 0; k < VS_ITEMS; ++k) mine += vis[k];
    int block_total;
    const int local = sweep::block_exclusive(mine, s_scan, &block_total);
    if (threadIdx.x < 32) {
        const uint32_t excl = sweep::chained_exclusive(state, t, (uint32_t)block_total);
        if (threadIdx.x == 0) s_excl = excl;
    }
    __syncthreads();
    int run = (int)(s_excl + (uint32_t)local);
    int out[VS_ITEMS];
#pragma unroll
    for (int k = 0; k < VS_ITEMS; ++k) { out[k] = run; run += vis[k]; }
    if (vec) {                       // scan is the library's own workspace: aligned
        reinterpret_cast<int4*>(scan + i0)[0] = make_int4(out[0], out[1], out[2], out[3]);
        reinterpret_cast<int4*>(scan + i0)[1] = make_int4(out[4], out[5], out[6], out[7]);
    } else {
#pragma unroll
        for (int k = 0; k < VS_ITEMS; ++k)
            if (i0 + k < n) scan[i0 + k] = out[k];
    }
}

// scan[i] = number of visible entries before i.  Plain layout (seg_cap == 0): row index = scan[i], d_count[0] = total.
// Segmented layout (seg_cap > 0; a segment = the seg_len entries of one camera = the rows for one destination rank):
// segment j owns rows [j*seg_cap, (j+1)*seg_cap) — a fixed-size send block, so the all-to-all needs no size exchange;
// rows past the capacity are dropped and reported through d_count[j] = visible entries of segment j (the caller compares
// with seg_cap); unused rows of a block are zero-filled (radius 0 = culled for the binning that reads them in place).
// row_index[i] is what the backward uses to find entry i's gradient row.
__global__ void __launch_bounds__(256) pack_rows_kernel(int64_t n, int64_t seg_len, int64_t seg_cap, const float2* __restrict__ xy,
                                                        const float* __restrict__ depth, const float* __restrict__ conic,
                                                        const float* __restrict__ comp, const float* __restrict__ opacity,
                                                        const float* __restrict__ rgb, const int32_t* __restrict__ radii,
                                                        const int32_t* __restrict__ scan, int32_t* __restrict__ row_index,
                                                        float* __restrict__ rows, int64_t* __restrict__ d_count) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int r = radii[i];
    int64_t o = scan[i];
    if (seg_cap > 0) {
        const int64_t seg = i / seg_len, first = seg * seg_len;
        const int64_t k = o - scan[first];
        if (i == min(n, first + seg_len) - 1) d_count[seg] = k + (r > 0 ? 1 : 0);
        o = (k < seg_cap) ? seg * seg_cap + k : -1;
    } else if (i == n - 1) {
        *d_count = o + (r > 0 ? 1 : 0);
    }
    row_index[i] = (int32_t)o;
    if (r <= 0 || o < 0) return;
    float4* out = reinterpret_cast<float4*>(rows + o * B200GS_ROW_FLOATS);
    const float2 p = xy[i];
    out[0] = make_float4(p.x, p.y, depth[i], conic[3 * i]);
    out[1] = make_float4(conic[3 * i + 1], conic[3 * i + 2], comp ? comp[i] : 1.0f, opacity[i]);
    out[2] = make_float4(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], __int_as_float(r));
}

// zero the unused tail of every fixed-size block
__global__ void __launch_bounds__(256) pad_rows_kernel(int64_t segments, int64_t seg_cap, const int64_t* __restrict__ d_count,
                                                       float* __restrict__ rows) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;    // one float4 per thread, 3 per row
    if (i >= segments * seg_cap * 3) return;
    const int64_t row = i / 3, seg = row / seg_cap, k = row - seg * seg_cap;
    if (k < d_count[seg]) return;
    reinterpret_cast<float4*>(rows)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

}  // namespace

static size_t pack_scan_state_bytes(int64_t n) { return align_up((size_t)div_up64(n > 0 ? n : 1, 256) * 4 + 64, 256); }

size_t pack_rows_workspace_bytes(int64_t n) { return pack_scan_state_bytes(n) + align_up((size_t)(n > 0 ? n : 1) * 4, 256); }

int pack_rows(int64_t n, int64_t seg_len, int64_t seg_cap, const float* xy, const float* depth, const float* conic, const float* comp,
              const float* opacity, const float* rgb, const int32_t* radii, void* ws, size_t ws_bytes, int32_t* row_index, float* rows,
              int64_t* d_count, cudaStream_t s) {
    const int64_t segments = seg_cap > 0 ? div_up64(n, seg_len) : 1;
    if (n == 0) {
        B200GS_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int64_t) * (size_t)segments, s));
        return B200GS_OK;
    }
    const size_t state_bytes = pack_scan_state_bytes(n);
    (void)ws_bytes;
    uint32_t* ticket = (uint32_t*)ws;               // [0]: ticket, [16..]: chained-scan state of the blocks
    uint32_t* state = ticket + 16;
    int32_t* scan = (int32_t*)((char*)ws + state_bytes);
    B200GS_CUDA(cudaMemsetAsync(ws, 0, state_bytes, s));
    visible_scan_kernel<<<(unsigned)div_up64(n, 256 * VS_ITEMS), 256, 0, s>>>(n, radii, scan, ticket, state);
    B200GS_LAUNCH_CHECK();
    pack_rows_kernel<<<(unsigned)div_up64(n, 256), 256, 0, s>>>(n, seg_cap > 0 ? seg_len : n, seg_cap, (const float2*)xy, depth,
                                                               conic, comp, opacity, rgb, radii, scan, row_index, rows, d_count);
    B200GS_LAUNCH_CHECK();
    if (seg_cap > 0) {
        pad_rows_kernel<<<(unsigned)div_up64(segments * seg_cap * 3, 256), 256, 0, s>>>(segments, seg_cap, d_count, rows);
        B200GS_LAUNCH_CHECK();
    }
    return B200GS_OK;
}

}  // namespace b200gs
