#!/usr/bin/env python
"""Benchmark of the rasterizer hot path: train-views/sec (forward + backward) @ N Gaussians, 1080p.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200gs|reference] [--mode vanilla|gsplat]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workloads are the BASELINE.json config shapes on the deterministic synthetic scene of SURVEY.md §8(d) (G(N, seed 0) in
[-1.3,1.3]^3, 32-pose camera ring, a fresh pose every step: parameters + per-view buffers > L2, no L2 flush needed):
  N = 1 (default)   configs[1] "Mip-NeRF360 garden, 1920x1080, ~1M Gaussians, SH deg 3, 1xB200 fwd+bwd" — the metric's config
  N = 2, 4, 8       configs[3] "bicycle, ~3M Gaussians, 1600x1063, Gaussian-sharded across 2/4/8 GPUs" (gsplat semantics, like the
                    reference's distributed renderer); at N = 8 configs[4] (10M, 1920x1080, tile culling on) is measured too and
                    reported under "other_workloads"
  --config K / --n --width --height select any other shape (configs[0] 30k/800x800, configs[2] 5M/1080p, ...).
The N = 1 line also carries "scaling_base": configs[3] on ONE GPU in gsplat mode — the like-for-like denominator of the
multi-GPU lines (same workload, same kernels); the N > 1 lines repeat it as measured on rank 0 alone in the same run.

One "step" = what `GaussianSplatting.training_step` asks of the renderer (internal/gaussian_splatting.py:344,380):
renderer.forward(camera, model, bg) from RAW parameters (activations included) and backward of a fixed random
cotangent G[3,H,W] ~ U(-1,1) down to the gradients of the six raw parameter tensors.  No loss, optimizer, dataloader.

Keys of the JSON line: see the driver contract.  `value` times K steps with everything resident in HBM; `e2e` times the
same steps through the public plug-in API with that step's cotangent image coming from pinned host memory (H2D inside
the timed region, standing for the ground-truth image upload of gaussian_splatting.py:250-264) and the step's scalar
result read back (D2H).  `roofline` is for the kernel with the largest share of the step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "train-views/sec (fwd+bwd) @ N Gaussians, 1080p"
UNIT = "views/s"

# BASELINE.json "configs", as (label, N Gaussians, width, height)
CONFIGS = {
    0: ("configs[0] shape: nerf_synthetic/lego, 30k Gaussians, 800x800", 30_000, 800, 800),
    1: ("configs[1] shape: Mip-NeRF360 garden, ~1M Gaussians, 1920x1080", 1_000_000, 1920, 1080),
    2: ("configs[2] shape: synthetic 5M Gaussians, 1920x1080", 5_000_000, 1920, 1080),
    3: ("configs[3] shape: Mip-NeRF360 bicycle, ~3M Gaussians, 1600x1063", 3_000_000, 1600, 1063),
    4: ("configs[4] shape: MatrixCity aerial block, 10M Gaussians, 1920x1080", 10_000_000, 1920, 1080),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200gs", choices=["b200gs", "reference"])
    ap.add_argument("--mode", default=None, choices=["vanilla", "gsplat"], help="default: vanilla on one GPU, gsplat when sharded")
    ap.add_argument("--config", type=int, default=None, choices=sorted(CONFIGS), help="BASELINE.json configs[K] shape; default 1 (N=1) / 3 (N>1)")
    ap.add_argument("--n", type=int, default=None)
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--no-extras", action="store_true", help="skip the scaling_base / single-GPU / configs[4] side measurements")
    ap.add_argument("--cpu-sample-iters", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parallelism", default="sharded", choices=["sharded", "replicas"],
                    help="N>1 only. sharded: the reference's Gaussian-sharded scheme (gsplat_distributed_renderer.py): scene split by "
                         "index across ranks, one camera per rank, all-to-all of the visible projected splats, gsplat semantics. "
                         "replicas: every rank holds the whole scene (configs/ddp.yaml style), no data-path collective.")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy, float32: "
                         "the image, and radii / view-space gradient / raw-parameter gradients of a fixed seeded sample of Gaussians")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.config is None:
        args.config = 1 if world == 1 else 3
    label, n, w, h = CONFIGS[args.config]
    custom = any(v is not None for v in (args.n, args.width, args.height))
    args.n = n if args.n is None else args.n
    args.width = w if args.width is None else args.width
    args.height = h if args.height is None else args.height
    args.workload_label = label if not custom else f"custom shape ({args.n} Gaussians, {args.width}x{args.height})"
    if args.mode is None:
        args.mode = "gsplat" if (world > 1 and args.parallelism == "sharded") else "vanilla"
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own CPU-runnable part of the path (BASELINE.md §3): projection + SH, forward + autograd
# backward, as restated (and pinned against the reference) in oracle/gs_oracle.py
# ----------------------------------------------------------------------------------------------------------------------
def _reference_modules():
    """internal/utils/gaussian_projection.py and sh_utils.py of the UNMODIFIED reference, from baseline/_ref (the offline
    pip --target install of /root/reference; git-ignored, shipped to the GPU box).  None when it is not there."""
    base = os.path.join(ROOT, "baseline", "_ref", "internal", "utils")
    if not os.path.exists(os.path.join(base, "gaussian_projection.py")):
        return None
    import importlib.util
    mods = []
    for name in ("gaussian_projection", "sh_utils"):
        spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(base, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        mods.append(m)
    return tuple(mods)


def cpu_projection_views_per_sec(n, width, height, mode_name, iters, warm=2, prefer_reference=True):
    from oracle import gs_oracle as O
    from b200gs.scene import activate, make_ring_cameras, make_scene
    mode = O.MODE_GSPLAT if mode_name == "gsplat" else O.MODE_VANILLA
    sc = activate(make_scene(n, 0))
    cams = make_ring_cameras(width, height)
    g = torch.Generator().manual_seed(1)
    c_xy, c_con, c_rgb = torch.randn(n, 2, generator=g), torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)
    ref = _reference_modules() if prefer_reference else None

    def one(it):
        cam = cams[it % len(cams)]
        ins = {k: sc[k].clone().requires_grad_(True) for k in ("means", "scales", "rotations", "shs")}
        if ref is not None:
            # the UNMODIFIED reference code (baseline/_ref): PythonPreprocessGSplatRenderer's projection + SH
            # (internal/renderers/pypreprocess_gsplat_renderer.py:20-38), forward + autograd backward, on the CPU
            gp, shu = ref
            t0 = time.perf_counter()
            out = gp.project_gaussians(means_3d=ins["means"], scales=ins["scales"], scale_modifier=1.0, quaternions=ins["rotations"],
                                       world_to_camera=cam.world_to_camera, fx=cam.fx, fy=cam.fy, cx=cam.cx, cy=cam.cy,
                                       img_height=cam.height, img_width=cam.width, block_width=16)
            dirs = ins["means"].detach() - cam.camera_center
            dirs = dirs / dirs.norm(dim=-1, keepdim=True)
            col = torch.clamp_min(shu.eval_sh(3, ins["shs"].transpose(1, 2), dirs) + 0.5, 0.0)
            ((out[0] * c_xy).sum() + (out[3] * c_con).sum() + (col * c_rgb).sum()).backward()
            return time.perf_counter() - t0
        ov = O.make_view(cam.R, cam.T, float(cam.fx), float(cam.fy), float(cam.cx), float(cam.cy), width, height)
        t0 = time.perf_counter()
        p = O.project(mode, ins["means"], ins["scales"], ins["rotations"], ov)
        col = O.sh_colors(3, ins["shs"], ins["means"], cam.camera_center, detach_dir=(mode == O.MODE_GSPLAT))
        ((p["xy"] * c_xy).sum() + (p["conic"] * c_con).sum() + (col * c_rgb).sum()).backward()
        return time.perf_counter() - t0

    # use all the host threads that help: torch's intra-op pool stops scaling (and can regress) well below 128 threads
    # on these elementwise passes, so probe a few pool sizes and keep the fastest
    ncpu = os.cpu_count() or 1
    best_t, best_threads = None, 1
    for th in sorted({min(ncpu, c) for c in (8, 16, 32, 64)}):   # 128 threads measured 36 s/view on the B200 host: not probed
        torch.set_num_threads(th)
        t = one(0)
        if best_t is None or t < best_t:
            best_t, best_threads = t, th
    torch.set_num_threads(best_threads)
    times = [one(it) for it in range(warm + iters)][warm:]
    times.sort()
    med = times[len(times) // 2]
    return 1.0 / med, med, best_threads, ("reference" if ref is not None else "port")


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)
    vps, med, cores, kind = cpu_projection_views_per_sec(args.n, args.width, args.height, args.mode, steps, warm=warm)
    sample = (f"the reference's CPU-runnable part of the path (pypreprocess projection + SH, forward + autograd backward; it has no "
              f"CPU blend/sort: BASELINE.md §3), {steps} views of the same workload, median; "
              + ("unmodified reference code from baseline/_ref" if kind == "reference" else "oracle port (baseline/_ref absent)"))
    line = {
        "impl": "reference", "metric": METRIC, "value": vps, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, "single" if world == 1 else "sharded-by-gaussian-index+exchange-of-projected-splats(peer stores over NVLink; all-to-all fallback)"),
        "cpu_baseline": {"value": vps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": vps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, parallelism):
    return {"workload": f"{args.workload_label}: synthetic G({args.n}, seed 0) SH deg 3, {args.width}x{args.height}, 32-pose ring, "
                        f"{args.mode} semantics, fwd+bwd from raw parameters",
            "n_gaussians": args.n, "width": args.width, "height": args.height, "mode": args.mode, "parallelism": parallelism,
            "l2": "inputs larger than L2 (236 MB parameters + fresh camera every step); no explicit flush"}


# bytes per view, SURVEY.md §8(d) / BASELINE.md §5 (V visible, I pairs, P pixels, N total; SH degree 3)
def algorithmic_bytes(stage, N, V, I, P, n_tiles, C=None):
    """I = (tile, Gaussian) pairs the stage actually processes (after exact tile culling)."""
    C = C if C is not None else int(2.5 * V)
    return {
        "project_fwd": V * 268 + N * 16,
        # phase A: xy/depth/radius/conic/opacity read (36 B per Gaussian, 24 more per visible one), {key, id} + 32 B record per
        # visible Gaussian, histogram read (8 B), 4 radix passes over the V records (8 B read + 8 B write each)
        "bin_count": N * 12 + V * (24 + 8 + 32 + 8 + 4 * 16),
        # phase B, C = (8x8-tile cell, Gaussian) entries (~2 per visible splat): emit reads {key,id} 8 B + the 32 B record per
        # visible Gaussian and writes 16 B per entry; one partition pass (16 B read + 16 B write); chunk counts read 8 B, write
        # 2 B x 64 tiles per 256-entry chunk; scatter reads 16 B; every fine pair's id written ONCE (4 B); tile starts / ranges
        "bin_sort": V * 40 + C * (16 + 32 + 8 + 16) + I * 4 + n_tiles * 24,
        "blend_fwd": I * 40 + P * 20,
        "blend_bwd": I * 76 + P * 20,
        "project_bwd": V * 552,
        "pack": N * 57 + V * 48,                       # sharded path: visibility scan + SoA read + [V,12] row write
    }.get(stage, 0)


def _launch_count():
    """Number of kernels libb200gs.so has launched so far in this process (counted inside the library at every launch)."""
    from b200gs._lib import lib
    fn = getattr(lib(), "b200gs_launch_count", None)
    return int(fn()) if fn is not None else None


class Workload:
    """One (shape, mode, parallelism) measurement on the current process group."""

    def __init__(self, n, width, height, mode, rank, world, local, sharded):
        from b200gs.renderers import B200GSplatRenderer, B200VanillaRenderer
        from b200gs.scene import SyntheticGaussians, make_ring_cameras, make_scene
        self.N, self.W, self.H, self.mode, self.rank, self.world, self.sharded = n, width, height, mode, rank, world, sharded
        self.dev = dev = torch.device("cuda", local)
        raw = make_scene(n, 0)
        self.cams = [c.to_device(dev) for c in make_ring_cameras(width, height)]
        if sharded:
            from b200gs.distributed import B200DistributedRenderer, shard_range
            lo, hi = shard_range(n, world, rank)
            self.model = SyntheticGaussians({k: v[lo:hi].contiguous() for k, v in raw.items()}).to(dev)
            self.renderer = B200DistributedRenderer().to(dev)
        else:
            self.model = SyntheticGaussians(raw).to(dev)
            self.renderer = (B200VanillaRenderer() if mode == "vanilla" else B200GSplatRenderer()).to(dev)
        del raw
        self.bg = torch.zeros(3, device=dev)
        gen = torch.Generator().manual_seed(1)
        self.cot_host = (torch.rand(3, height, width, generator=gen) * 2 - 1).pin_memory()
        self.cot = self.cot_host.to(dev)
        # e2e pipeline, the shape of the reference's training input path (dataset.py:150-305 prefetches, gaussian_splatting.py:
        # 250-264 copies to the device): step i's input image is uploaded from pinned memory on a copy stream while step i-1
        # computes (double buffer), and every step's scalar result is read back (its D2H lands one step later, so the host
        # never stalls the GPU).  Every byte is moved inside the timed region.  (The 32 camera poses — 40 floats each — are
        # device-resident before the loop, as a training set's cameras are.)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.read_stream = torch.cuda.Stream(device=dev)   # the result read-back never sits in the compute stream
        self.loss_ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.in_bufs = [torch.empty_like(self.cot), torch.empty_like(self.cot)]
        self.in_ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.loss_hosts = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]
        self.loss_done = [torch.cuda.Event(), torch.cuda.Event()]
        self.loss_dev = [torch.zeros(1, device=dev), torch.zeros(1, device=dev)]
        self.results = []
        self.fwd_done = torch.cuda.Event()
        self.step_done = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(self, i):
        # called right after step i-1's forward has been enqueued: the upload overlaps that step's backward (compute-bound
        # kernels) instead of the next forward's projection/binning (bandwidth- and latency-bound: measured 1.68 vs 1.58
        # ms/step, profiles/tools/e2e_probe.py).  The buffer's previous consumer (step i-2) precedes the event in stream order.
        self.fwd_done.record()
        self.copy_stream.wait_event(self.fwd_done)
        with torch.cuda.stream(self.copy_stream):
            self.in_bufs[i & 1].copy_(self.cot_host, non_blocking=True)
            self.in_ready[i & 1].record(self.copy_stream)

    def step(self, i, e2e=False, more=False):
        cam = self.cams[(i * self.world + self.rank) % len(self.cams)]   # each rank renders a different pose
        for p in self.model.parameters():
            p.grad = None
        out = self.renderer(cam, self.model, self.bg)
        if e2e:
            # the uploaded image is first needed by the loss, not by the renderer: the compute stream waits for it HERE, so an upload
            # that takes longer than the previous step's backward (24.9 MB over PCIe ~ 0.5 ms vs ~0.57 ms of backward) runs on under
            # this step's forward instead of stalling it (round 2: e2e fell to 490 views/s in some runs with the wait in front)
            torch.cuda.current_stream().wait_event(self.in_ready[i & 1])
            c = self.in_bufs[i & 1]
        else:
            c = self.cot
        if e2e and more:
            self.prefetch(i + 1)
        loss = (out["render"] * c).sum()
        loss.backward()
        if e2e:
            self.loss_dev[i & 1].copy_(loss.detach().reshape(1))
            self.loss_ready[i & 1].record()
            self.read_stream.wait_event(self.loss_ready[i & 1])
            with torch.cuda.stream(self.read_stream):
                self.loss_hosts[i & 1].copy_(self.loss_dev[i & 1], non_blocking=True)
                self.loss_done[i & 1].record(self.read_stream)
        return out

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, k, e2e, keep_last=False):
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if e2e:
            self.prefetch(0)
        for i in range(k):
            out = self.step(i, e2e, i + 1 < k)
            if keep_last and i + 1 == k:
                self.last_out = out
            del out
            if not e2e:
                self.step_done[i & 1].record()
            if i > 0:   # the host stays at most one step ahead in both loops, like a training loop that logs its loss
                if e2e:                                         # the user reads the previous step's result
                    self.loss_done[(i - 1) & 1].synchronize()
                    self.results.append(float(self.loss_hosts[(i - 1) & 1][0]))
                else:
                    self.step_done[(i - 1) & 1].synchronize()
        if e2e:
            self.loss_done[(k - 1) & 1].synchronize()
            self.results.append(float(self.loss_hosts[(k - 1) & 1][0]))
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms

    def run(self, steps, warmup, e2e=True, stages=True, keep_outputs=False):
        """-> dict(ms_total, ms_e2e, launches, stage_ms).  W untimed warm-up steps, then EXACTLY `steps` timed steps.
        keep_outputs: self.outputs = host copies of what the last timed step computed (see host_outputs)."""
        from b200gs import ops
        for i in range(max(warmup, 3)):
            self.step(i)
        self.timed(min(steps, 16), False)      # untimed: lets the caching allocator settle into the timed loop's pattern
        l0 = _launch_count()
        ms_total = self.timed(steps, False, keep_last=keep_outputs)
        l1 = _launch_count()
        if keep_outputs:     # before the steps below overwrite the gradients
            self.outputs = self.host_outputs(self.last_out)
            del self.last_out
        ms_e2e = self.timed(steps, True) if e2e else None
        stage_ms = {}
        if stages:    # per-stage timing (CUDA events on the launching stream) for the roofline numbers
            timer = ops.StageTimer()
            ops.set_stage_timer(timer)
            for i in range(min(steps, 32)):
                self.step(i)
            stage_ms, _ = timer.summary_ms()
            ops.set_stage_timer(None)
        return {"ms_total": ms_total, "ms_e2e": ms_e2e, "launches": (l1 - l0) if l0 is not None else None, "stage_ms": stage_ms}

    DUMP_ROWS = 1 << 16            # Gaussians sampled for the per-Gaussian arrays (16.5 MB at SH degree 3)
    DUMP_IMAGE_BYTES = 32 << 20    # a larger image is sampled at a fixed seeded set of pixels

    def host_outputs(self, out):
        """Float32 host copies of what the caller of one step receives: the rendered image [3,H,W], and for a fixed seeded sample of
        this rank's Gaussians (sorted indices) the radii, the view-space gradient and the gradients of the raw parameter tensors."""
        n = self.model.gaussians["means"].shape[0]
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:self.DUMP_ROWS].sort().values.to(self.dev)
        img = out["render"].detach()
        if img.numel() * 4 > self.DUMP_IMAGE_BYTES:
            pix = torch.randperm(img[0].numel(), generator=torch.Generator().manual_seed(1))[:self.DUMP_IMAGE_BYTES // 12]
            img = img.reshape(img.shape[0], -1)[:, pix.sort().values.to(self.dev)]
        res = {"render": img, "radii": out["radii"][rows]}
        if out["viewspace_points"].grad is not None:
            res["viewspace_points_grad"] = out["viewspace_points"].grad[rows]
        for k, p in self.model.gaussians.items():
            res[f"grad_{k}"] = p.grad[rows]
        return {k: v.float().cpu().numpy() for k, v in res.items()}

    def views_per_s(self, ms, steps):
        return steps * self.world / (ms * 1e-3)


def loss_stage(width, height, dev, iters=20):
    """The op right after the renderer in a training step (SURVEY §8f rank 2): (1-l) L1 + l (1 - SSIM) forward + backward on a [3,H,W]
    image.  Ours (two fused kernels) next to the reference's own torch implementation (internal/utils/ssim.py + vanilla_metrics.py:57-74,
    the code in baseline/_ref) on the same GPU.  Not part of `value`."""
    from b200gs import ops
    g = torch.Generator().manual_seed(3)
    gt = torch.rand(3, height, width, generator=g).to(dev)
    img = (gt + 0.1 * torch.randn(3, height, width, generator=g).to(dev)).clamp(0, 1)
    ref_path = os.path.join(ROOT, "baseline", "_ref", "internal", "utils", "ssim.py")
    kind = "reference (baseline/_ref internal/utils/ssim.py, torch on the GPU)"
    if os.path.exists(ref_path):
        import importlib.util
        spec = importlib.util.spec_from_file_location("ref_ssim", ref_path)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        ssim = m.ssim
    else:
        ssim, kind = None, "unavailable (baseline/_ref absent): only the fused kernels were timed"

    def ours():
        x = img.clone().requires_grad_(True)
        loss, _ = ops.l1_ssim_loss(x, gt, 0.2)
        loss.backward()
        return loss

    def theirs():
        x = img.clone().requires_grad_(True)
        loss = 0.8 * torch.abs(x - gt).mean() + 0.2 * (1.0 - ssim(x, gt))
        loss.backward()
        return loss

    out = {}
    for name, fn in (("fused_ms", ours), ("torch_ms", theirs)):
        if fn is theirs and ssim is None:
            continue
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            val = fn()
        e1.record()
        torch.cuda.synchronize()
        out[name] = round(e0.elapsed_time(e1) / iters, 4)
        out[name.replace("_ms", "_loss")] = float(val)
    out["torch_impl"] = kind
    out["what"] = f"L1 + SSIM training loss forward + backward on a [3,{height},{width}] image (includes the clone of the input), CUDA events, {iters} iterations"
    return out


def scene_statistics(n, width, height, mode, dev):
    """V, I (rect pairs), I after exact culling, coarse pairs of pose 0 on the full scene (one GPU, no collectives)."""
    from b200gs import ops
    from b200gs.renderers import camera_view
    from b200gs.scene import SyntheticGaussians, make_ring_cameras, make_scene
    model = SyntheticGaussians(make_scene(n, 0)).to(dev)
    cam = make_ring_cameras(width, height)[0].to_device(dev)
    mode_id = 0 if mode == "vanilla" else 1
    view = camera_view(cam, mode_id)
    with torch.no_grad():
        xy, depth, radii, conic, comp, tiles, _, _, _ = ops.project_forward(view, model.get_xyz.detach(), model.get_scaling.detach().contiguous(),
                                                                            model.get_rotation.detach().contiguous(), None, True)
        V, I = int((radii > 0).sum()), int(tiles.sum())
        opac_act = model.get_opacity.detach().reshape(-1).contiguous() * (comp if mode == "gsplat" else 1.0)
        binned = ops.bin_gaussians(mode_id, width, height, xy, depth, radii, conic, opac_act.contiguous())
        return V, I, binned.total, binned.coarse_pairs


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (b200gs has no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    N, W, H = args.n, args.width, args.height
    sharded = world > 1 and args.parallelism == "sharded"
    extras = {}

    # like-for-like single-GPU number of the same workload and mode (rank 0 alone; the other ranks wait): the denominator
    # the multi-GPU value should be read against
    if sharded and not args.no_extras:
        if rank == 0:
            solo = Workload(N, W, H, args.mode, 0, 1, local, False)
            r = solo.run(min(args.steps, 24), 3, e2e=False, stages=False)
            extras["single_gpu_same_workload"] = {"value": solo.views_per_s(r["ms_total"], min(args.steps, 24)), "unit": UNIT, "mode": args.mode,
                                                  "note": "the whole scene on rank 0 alone, same shape/mode/kernels, measured in this run"}
            del solo
            torch.cuda.empty_cache()
        dist.barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    wl = Workload(N, W, H, args.mode, rank, world, local, sharded)
    dump = args.dump_outputs is not None and rank == 0
    res = wl.run(args.steps, args.warmup, keep_outputs=dump)
    clocks = sampler.stop() if rank == 0 else None
    if dump:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in wl.outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    ms_total, ms_e2e, stage_ms = res["ms_total"], res["ms_e2e"], res["stage_ms"]
    cot_bytes = int(wl.cot_host.numel() * 4)
    del wl
    torch.cuda.empty_cache()

    # side measurements: configs[4] on 8 GPUs; the scaling base (configs[3], one GPU, gsplat mode) on the single-GPU line
    if not args.no_extras and args.config in (1, 3):
        if sharded and world == 8 and args.config == 3:
            label, n4, w4, h4 = CONFIGS[4]
            w4l = Workload(n4, w4, h4, "gsplat", rank, world, local, True)
            k4 = min(args.steps, 16)
            r4 = w4l.run(k4, 3, e2e=False, stages=False)
            extras["other_workloads"] = [{"workload": f"{label}: synthetic G({n4}, seed 0) SH deg 3, {w4}x{h4}, gsplat semantics, exact tile culling on, "
                                                      f"sharded by Gaussian index over {world} GPUs", "value": w4l.views_per_s(r4["ms_total"], k4),
                                          "unit": UNIT, "steps": k4, "ms_per_step": r4["ms_total"] / k4}]
            del w4l
            torch.cuda.empty_cache()
        elif world == 1 and args.config == 1:
            label, n3, w3, h3 = CONFIGS[3]
            w3l = Workload(n3, w3, h3, "gsplat", 0, 1, local, False)
            k3 = min(args.steps, 24)
            r3 = w3l.run(k3, 3, e2e=False, stages=False)
            extras["scaling_base"] = {"workload": f"{label}: synthetic G({n3}, seed 0), {w3}x{h3}, gsplat semantics, ONE GPU", "value": w3l.views_per_s(r3["ms_total"], k3),
                                      "unit": UNIT, "steps": k3, "note": "denominator for the N = 2/4/8 lines, which run this workload sharded"}
            del w3l
            torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # workload statistics of pose 0 for the algorithmic byte counts (full scene on this GPU, no collectives)
    V, I, I_culled, C_coarse = scene_statistics(N, W, H, args.mode, dev)
    gx, gy = (W + 15) // 16, (H + 15) // 16
    P = W * H
    hbm_peak, peak_src = peaks()
    kernels = {}
    for k, ms in stage_ms.items():
        b = algorithmic_bytes(k, N, V, I_culled, P, gx * gy, C_coarse)
        kernels[k] = {"ms": round(ms, 4), "alg_bytes": b, "gbs": round(b / (ms * 1e-3) / 1e9, 1)}
    top = max(stage_ms, key=stage_ms.get)
    ach = kernels[top]["gbs"]
    traffic, traffic_src, issue = None, None, None
    try:   # DRAM bytes / executed warp instructions per launch of that kernel from the committed ncu --set full capture
        prof = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_traffic.json"))
        if prof:
            with open(os.path.join(ROOT, "profiles", prof[-1])) as f:
                pj = json.load(f)
            traffic = pj.get(top)
            traffic_src = f"static: profiles/{prof[-1]} (ncu --set full capture of this command, configs[1]); not re-measured in this run"
            inst = pj.get(top + "_warp_instructions")
            if inst and clocks and clocks.get("sm_mhz"):
                peak_issue = 148 * 4 * clocks["sm_mhz"] * 1e6            # warp instructions per second: 4 schedulers per SM, 1 per clock
                issue = {"kernel": top, "bound": "issue", "achieved": round(inst / (stage_ms[top] * 1e-3) / 1e9, 1), "peak": round(peak_issue / 1e9, 1),
                         "unit": "G warp-inst/s", "frac": round(inst / (stage_ms[top] * 1e-3) / peak_issue, 4),
                         "source": f"executed warp instructions per launch from profiles/{prof[-1]} / live kernel time"}
    except Exception:
        traffic = None
    views_per_s = args.steps * world / (ms_total * 1e-3)
    e2e_vps = args.steps * world / (ms_e2e * 1e-3)

    line = {
        "metric": METRIC, "value": views_per_s, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, ("sharded-by-gaussian-index+exchange-of-projected-splats(peer stores over NVLink; all-to-all fallback)" if sharded else "replicas") if world > 1 else "single"),
        "e2e": {"value": e2e_vps, "unit": UNIT, "h2d_bytes_per_step": cot_bytes, "d2h_bytes_per_step": 4,
                "note": "per step: the [3,H,W] input image pinned-host->device and the scalar result device->host, inside the timed region; "
                        "the 32 camera poses (40 floats each) are device-resident before the loop, as a training set's cameras are"},
        "gpu_launches": res["launches"],
        "gpu_launches_note": "kernels launched by libb200gs.so inside the timed region, counted by the library at every launch (b200gs_launch_count)",
        "clocks": clocks,
        "roofline": {"kernel": top, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": round(ach / hbm_peak, 4),
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "note": "blend kernels are SM-issue (FP32+MUFU) bound, not HBM bound (SURVEY §8d): see roofline_issue; HBM fraction reported as asked"},
        "roofline_issue": issue,
        "kernels": kernels,
        "scene": {"N": N, "V": V, "I": I, "I_after_exact_culling": I_culled, "coarse_pairs": C_coarse, "P": P, "stage_sum_ms": round(sum(stage_ms.values()), 4)},
    }
    line.update(extras)
    if world > 1:
        line["scaling_note"] = ("N > 1 lines run configs[3] (and configs[4] at N = 8) as the north_star names them; the N = 1 headline line is configs[1], "
                                "a lighter workload: value / (N * value_N1) mixes workloads. The like-for-like single-GPU denominator, measured in this "
                                "run on rank 0 alone, is single_gpu_same_workload.value (also scaling_base.value in the N = 1 line).")
    if world == 1 and not args.no_extras:
        try:
            line["loss_stage"] = loss_stage(W, H, dev)
        except Exception as e:      # the loss is a side measurement: never lose the main line over it
            line["loss_stage"] = {"error": repr(e)}
    if not args.no_cpu_baseline and world == 1:
        vps, med, cores, kind = cpu_projection_views_per_sec(N, W, H, args.mode, args.cpu_sample_iters)
        line["cpu_baseline"] = {"value": vps, "unit": UNIT, "cores": cores, "kind": kind, "host_cpus": os.cpu_count() or 1,
                                "sample": f"reference CPU path (pypreprocess projection + SH, fwd + autograd bwd; no CPU blend exists), "
                                          f"{args.cpu_sample_iters} views, median; " + ("baseline/_ref code" if kind == "reference" else "oracle port")}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
