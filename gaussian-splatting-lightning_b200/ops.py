"""torch.autograd.Function wrappers over the C ABI (``libb200gs.so``).

PyTorch is used for device memory (its caching allocator owns every buffer, including workspaces), the current CUDA
stream and autograd bookkeeping only; all arithmetic of the hot path runs in the hand-written kernels.

Functions
  rasterize_vanilla(...)      the whole dgr-semantics pipeline as ONE autograd node (what
                              ``diff_gaussian_rasterization.GaussianRasterizer`` is; vanilla_renderer.py:111-120)
  project_gaussians(...)      gsplat v0 ``project_gaussians``          (gsplat_renderer.py:64-79)
  spherical_harmonics(...)    gsplat ``spherical_harmonics``           (gsplat_renderer.py:105)
  rasterize_gaussians(...)    gsplat v0 ``rasterize_gaussians``        (gsplat_renderer.py:86-99)
"""
import ctypes
import os
import threading
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import MODE_GSPLAT, MODE_VANILLA, TILE, B200gsView, check, lib, ptr

ROW_FLOATS = 12   # include/b200gs.h B200GS_ROW_FLOATS


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device (raw handle; ~20x cheaper than current_stream())."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


class StageTimer:
    """Optional per-stage CUDA-event timing on the launching stream (used by bench.py for the roofline numbers)."""

    def __init__(self):
        self.events = {}
        self.calls = {}

    class _Ctx:
        __slots__ = ("timer", "name", "start")

        def __init__(self, timer, name):
            self.timer, self.name = timer, name

        def __enter__(self):
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()

        def __exit__(self, *exc):
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            self.timer.events.setdefault(self.name, []).append((self.start, end))
            return False

    def stage(self, name):
        return StageTimer._Ctx(self, name)

    def reset(self):
        self.events.clear()

    def summary_ms(self):
        torch.cuda.synchronize()
        return {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in self.events.items()}, {k: len(v) for k, v in self.events.items()}


class _Null:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NULL = _Null()
_TIMER: Optional[StageTimer] = None


def set_stage_timer(timer: Optional[StageTimer]):
    global _TIMER
    _TIMER = timer


def _stage(name):
    return _NULL if _TIMER is None else _TIMER.stage(name)


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {t.dtype}")
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor (b200gs has no CPU path)")
    return t.contiguous()


def make_view(mode: int, width: int, height: int, *, fx: float = 0.0, fy: float = 0.0, cx: float = 0.0, cy: float = 0.0,
              tanfovx: float = 0.0, tanfovy: float = 0.0, viewmatrix=None, projmatrix=None, campos=None,
              sh_degree: int = 0, sh_stride: int = 1, scale_modifier: float = 1.0, eps2d: float = 0.3,
              near_plane: float = -1.0) -> B200gsView:
    """Pack a host-side B200gsView.  ``viewmatrix`` / ``projmatrix`` are the reference's transposed 4x4 tensors
    (Camera.world_to_camera / Camera.full_projection); they are copied to the host here (16 floats)."""
    v = B200gsView()
    v.width, v.height, v.mode = int(width), int(height), int(mode)
    v.sh_degree, v.sh_stride = int(sh_degree), int(sh_stride)
    v.fx, v.fy, v.cx, v.cy = float(fx), float(fy), float(cx), float(cy)
    v.tanfovx, v.tanfovy = float(tanfovx), float(tanfovy)
    v.scale_modifier, v.eps2d, v.near_plane = float(scale_modifier), float(eps2d), float(near_plane)
    if viewmatrix is not None:
        vm = viewmatrix.detach().to("cpu", torch.float32).reshape(-1).tolist()
        v.viewmatrix[:] = vm
    if projmatrix is not None:
        pm = projmatrix.detach().to("cpu", torch.float32).reshape(-1).tolist()
        v.projmatrix[:] = pm
    if campos is not None:
        cp = campos.detach().to("cpu", torch.float32).reshape(-1).tolist()
        v.campos[:] = cp
    return v


def _copy_view(v: B200gsView, **updates) -> B200gsView:
    out = B200gsView()
    ctypes.memmove(ctypes.byref(out), ctypes.byref(v), ctypes.sizeof(B200gsView))
    for k, val in updates.items():
        setattr(out, k, val)
    return out


# ----------------------------------------------------------------------------------------------------------------------
# binning helper (no autograd)
# ----------------------------------------------------------------------------------------------------------------------
class Binning:
    """Result of K2-K5 for one view: depth-sorted per-tile Gaussian id lists.  `rect_pairs` = the reference's pair count
    (every tile of the 3-sigma rects; bounds `total`), `coarse_pairs` = (8x8-tile cell, Gaussian) pairs of the first
    binning level, `total` = number of listed pairs.  In lazy mode the counters arrive asynchronously: rect/coarse are
    None until resolve(), `total` waits for its own copy when first read (see bin_gaussians)."""
    __slots__ = ("sorted_ids", "tile_ranges", "rect_pairs", "coarse_pairs", "_total", "_pending", "_host", "_event_b")

    def __init__(self, sorted_ids, tile_ranges, total=None, host=None, pending=None, event_b=None):
        self.sorted_ids, self.tile_ranges, self._total = sorted_ids, tile_ranges, total
        self.rect_pairs = self.coarse_pairs = None
        self._host, self._pending, self._event_b = host, pending, event_b
        if host is not None and pending is None:
            self.rect_pairs, self.coarse_pairs = int(host[0]), int(host[1])

    @property
    def total(self):
        if self._total is None and self._host is not None:
            if self._event_b is not None:
                self._event_b.synchronize()
            self._total = int(self._host[6])
        return self._total

    def resolve(self) -> bool:
        """Lazy mode: wait for phase A's counters (the GPU is far past that point when this is called after the blend has
        been enqueued).  Returns False when a counter exceeds the capacity the lists were built with — pairs were
        dropped and the caller must re-bin in exact mode.  The check uses the RECT pair count, which bounds the listed
        pairs and is known right after phase A, so it never waits for the binning itself."""
        if self._pending is None:
            return True
        event_a, key, cap_coarse, cap_pairs = self._pending
        self._pending = None
        event_a.synchronize()
        self.rect_pairs, self.coarse_pairs = int(self._host[0]), int(self._host[1])
        with _state_lock:
            _last_total[key] = (self.coarse_pairs, self.rect_pairs)
        return self.coarse_pairs <= cap_coarse and self.rect_pairs <= cap_pairs

    def __del__(self):
        try:
            if self._host is not None:
                _return_host_counts(self._host)
        except Exception:      # interpreter shutdown
            pass


_host_counts_pool = []  # pinned int64[8] buffers: [0:4] phase A's copy of the counters, [4:8] phase B's
_last_total = {}       # key -> (coarse pairs, rect pairs) of the previous view: sizes the next view's buffers in lazy mode
_state_lock = threading.RLock()   # the two process-wide structures above are shared by every thread that renders (trainer + viewer threads)

LAZY_SLACK = 1.15      # lazy mode: capacity = slack x previous count


def _host_counts():
    with _state_lock:
        if _host_counts_pool:
            return _host_counts_pool.pop()
    return torch.zeros(8, dtype=torch.int64).pin_memory()


def _return_host_counts(buf):
    with _state_lock:
        if len(_host_counts_pool) < 32:
            _host_counts_pool.append(buf)


def _bin(key, mode, width, height, n, dev, cull, lazy, count_call) -> Binning:
    L = lib()
    st = _stream()
    gx, gy = (width + TILE - 1) // TILE, (height + TILE - 1) // TILE
    ws_a = torch.empty(L.b200gs_bin_count_workspace_bytes(n), dtype=torch.uint8, device=dev)
    d_counts = torch.empty(4, dtype=torch.int64, device=dev)
    ranges = torch.empty(gx * gy, 2, dtype=torch.int32, device=dev)
    host = _host_counts()
    with _state_lock:
        prev = _last_total.get(key) if lazy else None
    sync = prev is None
    with _stage("bin_count"):
        count_call(ptr(ws_a), ws_a.numel(), ptr(d_counts), host.data_ptr(), 1 if sync else 0, st)
    if sync:
        cap_coarse, cap_pairs = int(host[1]), int(host[0])    # exact / an upper bound: cannot overflow
        with _state_lock:
            _last_total[key] = (cap_coarse, cap_pairs)
        pending = None
    else:
        event_a = torch.cuda.Event()
        event_a.record()
        cap_coarse = int(prev[0] * LAZY_SLACK) + 4096
        cap_pairs = int(prev[1] * LAZY_SLACK) + 4096
        pending = (event_a, key, cap_coarse, cap_pairs)
    sorted_ids = torch.empty(max(cap_pairs, 1), dtype=torch.int32, device=dev)
    ws_b = torch.empty(L.b200gs_bin_sort_workspace_bytes(n, cap_coarse, width, height), dtype=torch.uint8, device=dev)
    with _stage("bin_sort"):
        check(L.b200gs_bin_sort(mode, width, height, n, 1 if cull else 0, cap_coarse, cap_pairs, ptr(d_counts), ptr(ws_a), ptr(ws_b),
                                ws_b.numel(), ptr(sorted_ids), ptr(ranges), host.data_ptr() + 32, 1 if sync else 0, st), "b200gs_bin_sort")
    if sync:
        return Binning(sorted_ids, ranges, int(host[6]), host)
    event_b = torch.cuda.Event()
    event_b.record()
    return Binning(sorted_ids, ranges, None, host, pending, event_b)


def bin_gaussians(mode: int, width: int, height: int, xy: torch.Tensor, depth: torch.Tensor, radii: torch.Tensor,
                  conic: Optional[torch.Tensor] = None, opacity: Optional[torch.Tensor] = None, lazy: bool = False) -> Binning:
    """K2-K5.  Passing conic+opacity enables exact tile culling (see include/b200gs.h).

    lazy=False: the counters are read back synchronously (host syncs, like the reference backends) and the buffers can
    never overflow.  lazy=True: buffers are sized from the previous view's counts (x LAZY_SLACK), nothing blocks here;
    call Binning.resolve() once the rest of the forward is enqueued — it returns False in the rare case a capacity was
    exceeded and the forward has to be redone with lazy=False."""
    L = lib()
    if conic is None or opacity is None:
        conic = opacity = None
    n = xy.shape[0]

    def count_call(ws_a, ws_a_bytes, d_counts, host, sync, st):
        check(L.b200gs_bin_count(mode, width, height, n, ptr(xy), ptr(depth), ptr(radii), ptr(conic), ptr(opacity), ws_a, ws_a_bytes,
                                 d_counts, host, sync, st), "b200gs_bin_count")

    cull = conic is not None
    return _bin((mode, width, height, n, cull), mode, width, height, n, xy.device, cull, lazy, count_call)


def bin_rows(mode: int, width: int, height: int, rows: torch.Tensor, cull: bool = True, lazy: bool = False, block_counts=None,
             block_rows: int = 0) -> Binning:
    """K2-K5 on a [n,12] splat-row buffer read in place (b200gs_bin_count_rows); same lazy protocol as bin_gaussians.
    block_counts (int64 device tensor) / block_rows: the rows come in fixed-size blocks of which only the first block_counts[b] rows
    are valid (the sharded exchange)."""
    L = lib()
    n = rows.shape[0]

    def count_call(ws_a, ws_a_bytes, d_counts, host, sync, st):
        check(L.b200gs_bin_count_rows(mode, width, height, n, ptr(rows), int(cull), ws_a, ws_a_bytes, d_counts, host, sync, st,
                                      ptr(block_counts), int(block_rows) if block_counts is not None else 0), "b200gs_bin_count_rows")

    return _bin(("rows", mode, width, height, bool(cull)), mode, width, height, n, rows.device, bool(cull), lazy, count_call)


def blend_forward_rows(mode, width, height, binning: Binning, rows, bg, planar=False):
    """K6 on rows -> image [H,W,3] (planar: [3,H,W]), final_T, n_contrib."""
    L = lib()
    dev = rows.device
    image = torch.empty((3, height, width) if planar else (height, width, 3), dtype=torch.float32, device=dev)
    final_T = torch.empty(height, width, dtype=torch.float32, device=dev)
    n_contrib = torch.empty(height, width, dtype=torch.int32, device=dev)
    pix_stride, ch_stride = (1, height * width) if planar else (3, 1)
    with _stage("blend_fwd"):
        check(L.b200gs_blend_fwd_rows(mode, width, height, ptr(binning.tile_ranges), ptr(binning.sorted_ids), ptr(rows), ptr(bg), ptr(image),
                                      pix_stride, ch_stride, ptr(final_T), ptr(n_contrib), None, _stream()), "b200gs_blend_fwd_rows")
    return image, final_T, n_contrib


def bin_and_blend_rows(mode, width, height, rows, bg, cull=True, planar=False, block_counts=None, block_rows=0):
    binning = bin_rows(mode, width, height, rows, cull, lazy=True, block_counts=block_counts, block_rows=block_rows)
    out = blend_forward_rows(mode, width, height, binning, rows, bg, planar)
    if not binning.resolve():
        binning = bin_rows(mode, width, height, rows, cull, lazy=False, block_counts=block_counts, block_rows=block_rows)
        out = blend_forward_rows(mode, width, height, binning, rows, bg, planar)
    return binning, out


def bin_and_blend(mode, width, height, xy, depth, radii, conic, opacity, colors, bg, planar, want_alpha):
    """Forward binning + blend with the lazy (sync-free) pair count; falls back to an exact re-run on overflow."""
    binning = bin_gaussians(mode, width, height, xy, depth, radii, conic, opacity, lazy=True)
    out = blend_forward(mode, width, height, binning, xy, conic, opacity, colors, bg, planar, want_alpha)
    if not binning.resolve():
        binning = bin_gaussians(mode, width, height, xy, depth, radii, conic, opacity, lazy=False)
        out = blend_forward(mode, width, height, binning, xy, conic, opacity, colors, bg, planar, want_alpha)
    return binning, out


# ----------------------------------------------------------------------------------------------------------------------
# raw stage calls (no autograd) — also used directly by tests
# ----------------------------------------------------------------------------------------------------------------------
def project_forward(view: B200gsView, means, scales, quats, shs=None, want_comp=False, want_cov3d=False):
    L = lib()
    n = means.shape[0]
    dev = means.device
    xy = torch.empty(n, 2, dtype=torch.float32, device=dev)
    depth = torch.empty(n, dtype=torch.float32, device=dev)
    radii = torch.empty(n, dtype=torch.int32, device=dev)
    conic = torch.empty(n, 3, dtype=torch.float32, device=dev)
    tiles = torch.empty(n, dtype=torch.int32, device=dev)
    comp = torch.empty(n, dtype=torch.float32, device=dev) if want_comp else None
    cov3d = torch.empty(n, 6, dtype=torch.float32, device=dev) if want_cov3d else None
    rgb = clamped = None
    if shs is not None:
        rgb = torch.empty(n, 3, dtype=torch.float32, device=dev)
        clamped = torch.empty(n, dtype=torch.uint8, device=dev)
    with _stage("project_fwd"):
        check(L.b200gs_project_fwd(ctypes.byref(view), n, ptr(means), ptr(scales), ptr(quats), ptr(shs), ptr(xy), ptr(depth),
                                   ptr(radii), ptr(conic), ptr(comp), ptr(tiles), ptr(cov3d), ptr(rgb), ptr(clamped), _stream()),
              "b200gs_project_fwd")
    return xy, depth, radii, conic, comp, tiles, cov3d, rgb, clamped


def project_backward(view: B200gsView, means, scales, quats, shs, radii, clamped, v_xy, v_depth, v_conic, v_comp, v_rgb):
    L = lib()
    n = means.shape[0]
    dev = means.device
    v_means = torch.empty(n, 3, dtype=torch.float32, device=dev)
    v_scales = torch.empty(n, 3, dtype=torch.float32, device=dev)
    v_quats = torch.empty(n, 4, dtype=torch.float32, device=dev)
    v_shs = torch.empty_like(shs) if shs is not None else None
    with _stage("project_bwd"):
        check(L.b200gs_project_bwd(ctypes.byref(view), n, ptr(means), ptr(scales), ptr(quats), ptr(shs), ptr(radii), ptr(clamped),
                                   ptr(v_xy), ptr(v_depth), ptr(v_conic), ptr(v_comp), ptr(v_rgb), ptr(v_means), ptr(v_scales),
                                   ptr(v_quats), ptr(v_shs), _stream()), "b200gs_project_bwd")
    return v_means, v_scales, v_quats, v_shs


def blend_forward(mode, width, height, binning: Binning, xy, conic, opacity, colors, bg, planar: bool, want_alpha: bool, hit_any=None):
    """planar=True -> image [C,H,W] (vanilla); else [H,W,C] (gsplat).  hit_any: zero-filled uint8 [N] that receives 1 for every splat
    that contributed to a pixel (b200gs_blend_fwd_hits)."""
    L = lib()
    ch = colors.shape[1]
    dev = xy.device
    if planar:
        image = torch.empty(ch, height, width, dtype=torch.float32, device=dev)
        ps, cs = 1, height * width
    else:
        image = torch.empty(height, width, ch, dtype=torch.float32, device=dev)
        ps, cs = ch, 1
    final_T = torch.empty(height, width, dtype=torch.float32, device=dev)
    n_contrib = torch.empty(height, width, dtype=torch.int32, device=dev)
    alpha = torch.empty(height, width, dtype=torch.float32, device=dev) if want_alpha else None
    with _stage("blend_fwd"):
        if hit_any is None:
            check(L.b200gs_blend_fwd(mode, width, height, ch, ptr(binning.tile_ranges), ptr(binning.sorted_ids), ptr(xy), ptr(conic),
                                     ptr(opacity), ptr(colors), ptr(bg), ptr(image), ps, cs, ptr(final_T), ptr(n_contrib), ptr(alpha),
                                     _stream()), "b200gs_blend_fwd")
        else:
            check(L.b200gs_blend_fwd_hits(mode, width, height, ch, ptr(binning.tile_ranges), ptr(binning.sorted_ids), ptr(xy), ptr(conic),
                                          ptr(opacity), ptr(colors), ptr(bg), ptr(image), ps, cs, ptr(final_T), ptr(n_contrib), ptr(alpha),
                                          ptr(hit_any), _stream()), "b200gs_blend_fwd_hits")
    return image, final_T, n_contrib, alpha


def blend_backward(mode, width, height, binning: Binning, xy, conic, opacity, colors, bg, final_T, n_contrib, v_image, v_alpha,
                   planar: bool, xy_scale=(1.0, 1.0), want_abs: bool = False):
    L = lib()
    n, ch = colors.shape
    dev = xy.device
    # one zero-filled slab for all atomically accumulated outputs
    width_cols = 2 + 3 + 1 + ch + (2 if want_abs else 0)
    slab = torch.zeros(n * width_cols, dtype=torch.float32, device=dev)
    o = 0
    v_xy = slab[o:o + 2 * n].view(n, 2); o += 2 * n
    v_conic = slab[o:o + 3 * n].view(n, 3); o += 3 * n
    v_opacity = slab[o:o + n]; o += n
    v_colors = slab[o:o + ch * n].view(n, ch); o += ch * n
    v_abs = slab[o:o + 2 * n].view(n, 2) if want_abs else None
    ps, cs = (1, height * width) if planar else (ch, 1)
    with _stage("blend_bwd"):
        check(L.b200gs_blend_bwd(mode, width, height, ch, ptr(binning.tile_ranges), ptr(binning.sorted_ids), ptr(xy), ptr(conic),
                                 ptr(opacity), ptr(colors), ptr(bg), ptr(final_T), ptr(n_contrib), ptr(v_image), ps, cs,
                                 ptr(v_alpha), float(xy_scale[0]), float(xy_scale[1]), ptr(v_xy), ptr(v_conic), ptr(v_opacity),
                                 ptr(v_colors), ptr(v_abs), _stream()), "b200gs_blend_bwd")
    return v_xy, v_conic, v_opacity, v_colors, v_abs


# ----------------------------------------------------------------------------------------------------------------------
# vanilla: one autograd node for the whole pipeline (diff_gaussian_rasterization semantics)
# ----------------------------------------------------------------------------------------------------------------------
class _RasterizeVanilla(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, shs, colors_precomp, opacities, scales, rotations, bg, view: B200gsView):
        n = means3D.shape[0]
        means3D = _f32c(means3D, "means3D")
        scales = _f32c(scales, "scales")
        rotations = _f32c(rotations, "rotations")
        opac = _f32c(opacities, "opacities").reshape(-1)
        bg = _f32c(bg, "bg")
        use_sh = shs is not None
        if use_sh:
            shs = _f32c(shs, "shs")
            view = _copy_view(view, sh_stride=int(shs.shape[1]))
        else:
            colors_precomp = _f32c(colors_precomp, "colors_precomp")
        W, H = view.width, view.height
        xy, depth, radii, conic, _, tiles, _, rgb, clamped = project_forward(view, means3D, scales, rotations, shs if use_sh else None)
        colors = rgb if use_sh else colors_precomp
        binning, (image, final_T, n_contrib, _) = bin_and_blend(MODE_VANILLA, W, H, xy, depth, radii, conic, opac, colors, bg, True, False)
        ctx.view = view
        ctx.use_sh = use_sh
        ctx.binning = binning
        ctx.means2D_shape = tuple(means2D.shape)
        ctx.opac_shape = tuple(opacities.shape)
        ctx.save_for_backward(means3D, scales, rotations, shs if use_sh else colors_precomp, opac, bg, xy, conic, radii,
                              clamped if use_sh else None, rgb if use_sh else None, final_T, n_contrib)
        ctx.mark_non_differentiable(radii)
        return image, radii

    @staticmethod
    def backward(ctx, v_image, _v_radii):
        means3D, scales, rotations, sh_or_col, opac, bg, xy, conic, radii, clamped, rgb, final_T, n_contrib = ctx.saved_tensors
        view = ctx.view
        W, H = view.width, view.height
        use_sh = ctx.use_sh
        colors = rgb if use_sh else sh_or_col
        v_image = _f32c(v_image, "grad_image")
        # dgr stores dL/dmean2D in NDC-scaled units: pixel gradient x (0.5 W, 0.5 H)
        v_xy, v_conic, v_opacity, v_colors, _ = blend_backward(MODE_VANILLA, W, H, ctx.binning, xy, conic, opac, colors, bg,
                                                              final_T, n_contrib, v_image, None, True, (0.5 * W, 0.5 * H))
        v_means, v_scales, v_quats, v_shs = project_backward(view, means3D, scales, rotations, sh_or_col if use_sh else None,
                                                             radii, clamped, v_xy, None, v_conic, None, v_colors if use_sh else None)
        n = means3D.shape[0]
        v_means2D = torch.zeros(ctx.means2D_shape, dtype=torch.float32, device=means3D.device)
        v_means2D[:, :2] = v_xy
        return (v_means, v_means2D, v_shs if use_sh else None, None if use_sh else v_colors, v_opacity.reshape(ctx.opac_shape),
                v_scales, v_quats, None, None)


def rasterize_vanilla(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, bg, view: B200gsView):
    """-> (color [3,H,W], radii int32 [N]).  Exactly one of shs / colors_precomp."""
    if (shs is None) == (colors_precomp is None):
        raise ValueError("Please provide exactly one of either SHs or precomputed colors!")
    if scales is None or rotations is None:
        raise NotImplementedError("cov3D_precomp is not supported by b200gs; pass scales and rotations")
    return _RasterizeVanilla.apply(means3D, means2D, shs, colors_precomp, opacities, scales, rotations, bg, view)


# ----------------------------------------------------------------------------------------------------------------------
# vanilla, activations fused: the same node fed with the model's RAW parameter tensors (b200gs_project_*_rows)
# ----------------------------------------------------------------------------------------------------------------------
class _RasterizeRaw(torch.autograd.Function):
    """The whole renderer step as ONE autograd node on the model's RAW parameters, either constant set: K1 (activations + SH fused)
    writes one [N,12] row per Gaussian, K2-K6 read the rows in place; backward: K7 accumulates [N,12] gradient rows (128-bit
    reductions), K8 reads them in place.  `means2D` is the viewspace-points tensor of the renderer contract ([N,3] zeros in vanilla
    mode, [N,2] in gsplat mode where it is also filled with the projected means): its `.grad` receives d loss / d mean2D."""

    @staticmethod
    def forward(ctx, mode, means3D, means2D, shs_dc, shs_rest, opacity_logits, log_scales, raw_quats, bg, view: B200gsView, anti_aliased):
        means3D = _f32c(means3D, "means3D")
        log_scales = _f32c(log_scales, "scales")
        raw_quats = _f32c(raw_quats, "rotations")
        ol = _f32c(opacity_logits, "opacities").reshape(-1)
        shs_dc = _f32c(shs_dc, "shs_dc")
        shs_rest = _f32c(shs_rest, "shs_rest")
        bg = _f32c(bg, "bg")
        view = _copy_view(view, sh_stride=int(shs_dc.shape[1] + shs_rest.shape[1]))
        W, H = view.width, view.height
        n, dev = means3D.shape[0], means3D.device
        rows = torch.empty(n, ROW_FLOATS, dtype=torch.float32, device=dev)
        radii = torch.empty(n, dtype=torch.int32, device=dev)
        clamped = torch.empty(n, dtype=torch.uint8, device=dev)
        with _stage("project_fwd"):
            check(lib().b200gs_project_fwd_rows(ctypes.byref(view), n, ptr(means3D), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc),
                                                ptr(shs_rest), int(bool(anti_aliased)), ptr(rows), ptr(radii), ptr(clamped), None, _stream()),
                  "b200gs_project_fwd_rows")
        binning, (image, final_T, n_contrib) = bin_and_blend_rows(mode, W, H, rows, bg, True, mode == MODE_VANILLA)
        if mode == MODE_GSPLAT:
            means2D.detach()[:, :2].copy_(rows[:, 0:2])     # the gsplat renderers hand the projected means out as `viewspace_points`
        ctx.view, ctx.mode, ctx.aa = view, mode, bool(anti_aliased)
        ctx.binning = binning
        ctx.means2D_shape = tuple(means2D.shape)
        ctx.opac_shape = tuple(opacity_logits.shape)
        ctx.save_for_backward(means3D, log_scales, raw_quats, ol, shs_dc, shs_rest, bg, rows, radii, clamped, final_T, n_contrib)
        ctx.mark_non_differentiable(radii)
        return image, radii

    @staticmethod
    def backward(ctx, v_image, _v_radii):
        means3D, log_scales, raw_quats, ol, shs_dc, shs_rest, bg, rows, radii, clamped, final_T, n_contrib = ctx.saved_tensors
        view, mode = ctx.view, ctx.mode
        W, H = view.width, view.height
        v_image = _f32c(v_image, "grad_image")
        n = means3D.shape[0]
        dev = means3D.device
        v_rows = torch.zeros(n, ROW_FLOATS, dtype=torch.float32, device=dev)
        L = lib()
        if mode == MODE_VANILLA:      # [3,H,W] image, mean2D gradient in NDC units (the vanilla rasterizer's convention)
            pix_stride, ch_stride, gsx, gsy = 1, H * W, 0.5 * W, 0.5 * H
        else:                         # [H,W,3] image, mean2D gradient in pixels
            pix_stride, ch_stride, gsx, gsy = 3, 1, 1.0, 1.0
        with _stage("blend_bwd"):
            check(L.b200gs_blend_bwd_rows(mode, W, H, ptr(ctx.binning.tile_ranges), ptr(ctx.binning.sorted_ids), ptr(rows), ptr(bg), ptr(final_T),
                                          ptr(n_contrib), ptr(v_image), pix_stride, ch_stride, None, gsx, gsy, ptr(v_rows), _stream()),
                  "b200gs_blend_bwd_rows")
        v_means = torch.empty(n, 3, dtype=torch.float32, device=dev)
        v_ls = torch.empty(n, 3, dtype=torch.float32, device=dev)
        v_q = torch.empty(n, 4, dtype=torch.float32, device=dev)
        v_ol = torch.empty(n, dtype=torch.float32, device=dev)
        v_dc, v_rest = torch.empty_like(shs_dc), torch.empty_like(shs_rest)
        # d loss / d mean2D (`viewspace_points.grad`): K8 writes it while it has the gradient row in registers
        cols = int(ctx.means2D_shape[1])
        v_means2D = torch.empty(n, cols, dtype=torch.float32, device=dev) if (ctx.needs_input_grad[2] and cols in (2, 3)) else None
        with _stage("project_bwd"):
            check(L.b200gs_project_bwd_rows(ctypes.byref(view), n, ptr(means3D), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc), ptr(shs_rest),
                                            int(ctx.aa), ptr(radii), ptr(clamped), None, ptr(v_rows), 0, ptr(v_means), ptr(v_ls), ptr(v_q), ptr(v_ol),
                                            ptr(v_dc), ptr(v_rest), ptr(v_means2D), cols if v_means2D is not None else 0, _stream()),
                  "b200gs_project_bwd_rows")
        if v_means2D is None and ctx.needs_input_grad[2]:
            v_means2D = torch.zeros(ctx.means2D_shape, dtype=torch.float32, device=dev)
            v_means2D[:, :2] = v_rows[:, 0:2]
        return None, v_means, v_means2D, v_dc, v_rest, v_ol.reshape(ctx.opac_shape), v_ls, v_q, None, None, None


def rasterize_vanilla_raw(means3D, means2D, shs_dc, shs_rest, opacity_logits, log_scales, raw_quats, bg, view: B200gsView):
    """Fused-activation variant of rasterize_vanilla: inputs are the model's RAW parameters
    (means, shs_dc [N,1,3], shs_rest [N,K-1,3], opacity logits, log-scales, un-normalised quaternions)."""
    return _RasterizeRaw.apply(MODE_VANILLA, means3D, means2D, shs_dc, shs_rest, opacity_logits, log_scales, raw_quats, bg, view, False)


def rasterize_gsplat_raw(means3D, means2D, shs_dc, shs_rest, opacity_logits, log_scales, raw_quats, bg, view: B200gsView, anti_aliased=True):
    """The gsplat-semantics counterpart: -> ([H,W,3] image, radii); `means2D` [N,2] receives the projected means (values) and
    d loss / d mean2D in pixels (`.grad`)."""
    return _RasterizeRaw.apply(MODE_GSPLAT, means3D, means2D, shs_dc, shs_rest, opacity_logits, log_scales, raw_quats, bg, view, anti_aliased)


# ----------------------------------------------------------------------------------------------------------------------
# gsplat v0 surface
# ----------------------------------------------------------------------------------------------------------------------
class _ProjectGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3d, scales, quats, view: B200gsView):
        means3d = _f32c(means3d, "means3d")
        scales = _f32c(scales, "scales")
        quats = _f32c(quats, "quats")
        xy, depth, radii, conic, comp, tiles, cov3d, _, _ = project_forward(view, means3d, scales, quats, None, True, True)
        ctx.view = view
        ctx.save_for_backward(means3d, scales, quats, radii)
        ctx.mark_non_differentiable(radii, tiles, cov3d)
        return xy, depth, radii, conic, comp, tiles, cov3d

    @staticmethod
    def backward(ctx, v_xy, v_depth, _v_radii, v_conic, v_comp, _v_tiles, _v_cov3d):
        means3d, scales, quats, radii = ctx.saved_tensors
        n = means3d.shape[0]
        dev = means3d.device

        def z(t, shape):
            return torch.zeros(shape, dtype=torch.float32, device=dev) if t is None else _f32c(t, "grad")

        v_means, v_scales, v_quats, _ = project_backward(ctx.view, means3d, scales, quats, None, radii, None, z(v_xy, (n, 2)),
                                                         z(v_depth, (n,)), z(v_conic, (n, 3)), z(v_comp, (n,)), None)
        return v_means, v_scales, v_quats, None


def project_gaussians(means3d, scales, glob_scale, quats, viewmat, fx, fy, cx, cy, img_height, img_width, block_width=16,
                      clip_thresh=0.01, filter_2d_kernel_size=0.3, view: Optional[B200gsView] = None):
    """gsplat v0 ``project_gaussians``: -> (xys [N,2], depths [N], radii int32 [N], conics [N,3], compensation [N],
    num_tiles_hit int32 [N], cov3d [N,6]).  ``viewmat`` is the standard [3|4,4] world-to-camera (rows R|t), i.e.
    ``camera.world_to_camera.T[:3,:]`` as the reference passes it (gsplat_renderer.py:69)."""
    if block_width != TILE:
        raise ValueError(f"b200gs supports block_width {TILE} only (the reference default, gsplat_renderer.py:7)")
    if view is None:
        vm = torch.eye(4, dtype=torch.float32)
        vm[:viewmat.shape[0], :] = viewmat.detach().to("cpu", torch.float32)
        view = make_view(MODE_GSPLAT, img_width, img_height, fx=fx, fy=fy, cx=cx, cy=cy, viewmatrix=vm.T.contiguous(),
                         scale_modifier=glob_scale, eps2d=filter_2d_kernel_size, near_plane=clip_thresh)
    return _ProjectGaussians.apply(means3d, scales, quats, view)


class _SphericalHarmonics(torch.autograd.Function):
    @staticmethod
    def forward(ctx, degree: int, dirs, coeffs):
        dirs = _f32c(dirs, "dirs")
        coeffs = _f32c(coeffs, "coeffs")
        n, k = coeffs.shape[0], coeffs.shape[1]
        rgb = torch.empty(n, 3, dtype=torch.float32, device=coeffs.device)
        check(lib().b200gs_sh_fwd(int(degree), k, n, ptr(dirs), ptr(coeffs), ptr(rgb), _stream()), "b200gs_sh_fwd")
        ctx.degree = int(degree)
        ctx.save_for_backward(dirs, coeffs)
        return rgb

    @staticmethod
    def backward(ctx, v_rgb):
        dirs, coeffs = ctx.saved_tensors
        n, k = coeffs.shape[0], coeffs.shape[1]
        v_rgb = _f32c(v_rgb, "grad")
        v_coeffs = torch.empty_like(coeffs)
        v_dirs = torch.empty_like(dirs) if ctx.needs_input_grad[1] else None
        check(lib().b200gs_sh_bwd(ctx.degree, k, n, ptr(dirs), ptr(coeffs), ptr(v_rgb), ptr(v_coeffs), ptr(v_dirs), _stream()),
              "b200gs_sh_bwd")
        return None, v_dirs, v_coeffs


def spherical_harmonics(degrees_to_use: int, dirs: torch.Tensor, coeffs: torch.Tensor, masks: Optional[torch.Tensor] = None) -> torch.Tensor:
    """gsplat ``spherical_harmonics(deg, dirs[N,3], coeffs[N,K,3], masks=None) -> [N,3]`` (directions normalised inside).  `masks`
    (gsplat skips the masked-out rows) is accepted for call compatibility; every row is evaluated, the caller only reads the visible ones."""
    if coeffs.shape[-1] != 3 or coeffs.dim() != 3:
        raise ValueError("coeffs must be [N, K, 3]")
    return _SphericalHarmonics.apply(degrees_to_use, dirs, coeffs)


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xys, depths, radii, conics, colors, opacity, img_height, img_width, background, return_alpha, absgrad):
        xys = _f32c(xys, "xys")
        depths = _f32c(depths, "depths")
        conics = _f32c(conics, "conics")
        colors = _f32c(colors, "colors")
        opac = _f32c(opacity, "opacity").reshape(-1)
        radii = radii.contiguous()
        bg = _f32c(background, "background") if background is not None else None
        H, W = int(img_height), int(img_width)
        binning, (image, final_T, n_contrib, alpha) = bin_and_blend(MODE_GSPLAT, W, H, xys, depths, radii, conics, opac, colors, bg, False, True)
        ctx.binning = binning
        ctx.hw = (H, W)
        ctx.absgrad = absgrad
        ctx.opac_shape = tuple(opacity.shape)
        ctx.save_for_backward(xys, conics, colors, opac, bg, final_T, n_contrib)
        ctx.xys_ref = xys
        return image, alpha

    @staticmethod
    def backward(ctx, v_image, v_alpha):
        xys, conics, colors, opac, bg, final_T, n_contrib = ctx.saved_tensors
        H, W = ctx.hw
        v_image = _f32c(v_image, "grad_image")
        v_alpha = _f32c(v_alpha, "grad_alpha") if v_alpha is not None else None
        v_xy, v_conic, v_opacity, v_colors, v_abs = blend_backward(MODE_GSPLAT, W, H, ctx.binning, xys, conics, opac, colors, bg,
                                                                   final_T, n_contrib, v_image, v_alpha, False, (1.0, 1.0),
                                                                   ctx.absgrad)
        if ctx.absgrad:
            ctx.xys_ref.absgrad = v_abs
        return v_xy, None, None, v_conic, v_colors, v_opacity.reshape(ctx.opac_shape), None, None, None, None, None


def rasterize_gaussians(xys, depths, radii, conics, num_tiles_hit, colors, opacity, img_height, img_width, block_width=16,
                        background=None, return_alpha=False, absgrad=False):
    """gsplat v0 ``rasterize_gaussians`` -> [H,W,D] (and alpha [H,W] when return_alpha)."""
    if block_width != TILE:
        raise ValueError(f"b200gs supports block_width {TILE} only")
    if colors.dim() != 2 or not (1 <= colors.shape[1] <= 4):
        raise ValueError("colors must be [N, D] with 1 <= D <= 4")
    if background is not None and background.shape[0] != colors.shape[1]:
        raise ValueError("background must have one entry per colour channel")
    image, alpha = _RasterizeGaussians.apply(xys, depths, radii, conics, colors, opacity, img_height, img_width, background,
                                             return_alpha, absgrad)
    return (image, alpha) if return_alpha else image


class _RasterizeBinned(torch.autograd.Function):
    """K6 / K7 on a binning computed beforehand (gsplat v1: isect_tiles + isect_offset_encode once, rasterize_to_pixels several
    times with different colour sets — gsplat_v1_renderer.py:176-196,326-352).  <= 4 channels per call."""

    @staticmethod
    def forward(ctx, xys, conics, colors, opacity, background, binning, hw, absgrad, want_hits):
        xys = _f32c(xys, "means2d")
        conics = _f32c(conics, "conics")
        colors = _f32c(colors, "colors")
        opac = _f32c(opacity, "opacities").reshape(-1)
        bg = _f32c(background, "background") if background is not None else None
        H, W = hw
        hits = torch.zeros(xys.shape[0], dtype=torch.uint8, device=xys.device) if want_hits else None
        image, final_T, n_contrib, alpha = blend_forward(MODE_GSPLAT, W, H, binning, xys, conics, opac, colors, bg, False, True, hits)
        ctx.binning, ctx.hw, ctx.absgrad, ctx.opac_shape = binning, hw, bool(absgrad), tuple(opacity.shape)
        ctx.save_for_backward(xys, conics, colors, opac, bg, final_T, n_contrib)
        ctx.xys_ref = xys
        ctx.mark_non_differentiable(*([hits] if hits is not None else []))
        return (image, alpha, hits) if hits is not None else (image, alpha)

    @staticmethod
    def backward(ctx, v_image, v_alpha, *_):
        xys, conics, colors, opac, bg, final_T, n_contrib = ctx.saved_tensors
        H, W = ctx.hw
        v_image = _f32c(v_image, "grad_image")
        v_alpha = _f32c(v_alpha, "grad_alpha") if v_alpha is not None else None
        v_xy, v_conic, v_opacity, v_colors, v_abs = blend_backward(MODE_GSPLAT, W, H, ctx.binning, xys, conics, opac, colors, bg, final_T,
                                                                   n_contrib, v_image, v_alpha, False, (1.0, 1.0), ctx.absgrad)
        if ctx.absgrad:   # channel groups of one render accumulate (|.| per group: an upper bound of gsplat's all-channel value when D > 4)
            prev = getattr(ctx.xys_ref, "absgrad", None)
            ctx.xys_ref.absgrad = v_abs if prev is None else prev + v_abs
        return v_xy, v_conic, v_colors, v_opacity.reshape(ctx.opac_shape), None, None, None, None, None


def rasterize_binned(means2d, conics, colors, opacities, binning: Binning, img_height: int, img_width: int, background=None,
                     absgrad: bool = False, want_hits: bool = False):
    """-> (image [H,W,D], alpha [H,W], hits uint8 [N] or None) for any D >= 1: the channels are composited in groups of <= 4 over the
    same per-tile lists (alpha / hits come from the first group; `means2d.absgrad`, when requested, accumulates every group's)."""
    if colors.dim() != 2 or colors.shape[1] < 1:
        raise ValueError("colors must be [N, D] with D >= 1")
    if background is not None and background.shape[0] != colors.shape[1]:
        raise ValueError("background must have one entry per colour channel")
    D = colors.shape[1]
    images, alpha, hits, abs_total = [], None, None, None
    for c0 in range(0, D, 4):
        c1 = min(D, c0 + 4)
        out = _RasterizeBinned.apply(means2d, conics, colors[:, c0:c1], opacities, None if background is None else background[c0:c1], binning,
                                     (int(img_height), int(img_width)), absgrad, want_hits and c0 == 0)
        images.append(out[0])
        if c0 == 0:
            alpha = out[1]
            hits = out[2] if want_hits else None
    return (images[0] if len(images) == 1 else torch.cat(images, dim=-1)), alpha, hits


def knn_mean_dist2(points: torch.Tensor) -> torch.Tensor:
    """``simple_knn._C.distCUDA2(points [N,3]) -> [N]``: mean squared distance to the 3 nearest neighbours (vanilla_gaussian.py:122-125)."""
    pts = _f32c(points, "points")
    if pts.dim() != 2 or pts.shape[1] != 3:
        raise ValueError("points must be [N, 3]")
    L = lib()
    n = pts.shape[0]
    out = torch.empty(n, dtype=torch.float32, device=pts.device)
    ws = torch.empty(max(int(L.b200gs_knn_workspace_bytes(n)), 256), dtype=torch.uint8, device=pts.device)
    check(L.b200gs_knn_mean_dist2(n, ptr(pts), ptr(out), ptr(ws), ws.numel(), _stream()), "b200gs_knn_mean_dist2")
    return out


# ----------------------------------------------------------------------------------------------------------------------
# fused L1 + SSIM loss (csrc/loss.cu; the metric the reference computes right after the renderer, vanilla_metrics.py:57-80)
# ----------------------------------------------------------------------------------------------------------------------
class _L1SSIMLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image, target, lambda_dssim):
        L = lib()
        image, target = _f32c(image, "image"), _f32c(target, "target")
        if image.dim() != 3 or image.shape != target.shape:
            raise ValueError("image and target must both be [C,H,W]")
        C, H, W = image.shape
        dev = image.device
        blocks = int(L.b200gs_loss_blocks(C, W, H))
        dmaps = torch.empty(3, C, H, W, dtype=torch.float32, device=dev)
        partials = torch.empty(blocks, 2, dtype=torch.float32, device=dev)
        with _stage("loss_fwd"):
            check(L.b200gs_loss_fwd(C, W, H, ptr(image), ptr(target), ptr(dmaps), ptr(partials), _stream()), "b200gs_loss_fwd")
        sums = partials.sum(dim=0) / float(C * H * W)                   # [mean |a-b|, mean SSIM]; fixed summation order
        loss = (1.0 - lambda_dssim) * sums[0] + lambda_dssim * (1.0 - sums[1])
        ctx.save_for_backward(image, target, dmaps)
        ctx.lambda_dssim = float(lambda_dssim)
        ctx.mark_non_differentiable(sums)
        return loss, sums

    @staticmethod
    def backward(ctx, v_loss, _v_sums):
        L = lib()
        image, target, dmaps = ctx.saved_tensors
        C, H, W = image.shape
        v_image = torch.empty_like(image)
        v = _f32c(v_loss.reshape(1), "grad_loss")
        with _stage("loss_bwd"):
            check(L.b200gs_loss_bwd(C, W, H, ptr(image), ptr(target), ptr(dmaps), ctx.lambda_dssim, ptr(v), ptr(v_image), _stream()),
                  "b200gs_loss_bwd")
        return v_image, None, None


def l1_ssim_loss(image: torch.Tensor, target: torch.Tensor, lambda_dssim: float = 0.2):
    """(1 - lambda) * L1 + lambda * (1 - SSIM) of `VanillaMetricsImpl._get_basic_metrics` (vanilla_metrics.py:57-74) in two
    kernels; returns (loss, stats) with stats = [mean |image - target|, mean SSIM].  image/target: [C,H,W] fp32 CUDA."""
    return _L1SSIMLoss.apply(image, target, float(lambda_dssim))
