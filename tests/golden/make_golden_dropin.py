"""Golden vectors for tests/test_gpu_reference_dropin.py: the reference's own classes, run UNMODIFIED on a CUDA device on
the b200gs kernels (``b200gs.compat.install()`` aliases ``diff_gaussian_rasterization`` / ``gsplat`` in ``sys.modules``):
``internal.models.vanilla_gaussian.VanillaGaussian``, ``internal.cameras.cameras.Cameras``,
``internal.renderers.{vanilla,gsplat,pypreprocess_gsplat}_renderer`` and ``internal.utils.ssim``.

    python tests/golden/make_golden_dropin.py <reference checkout> [out.npz]   -> tests/golden/dropin_n6000_320x240.npz

To keep the file small it holds the outputs at a fixed seeded sample of pixels and of visible Gaussians, plus every radius,
the visibility masks and the full-size gradient maxima that the tests' relative errors are taken against.
``lightning`` is only needed by the reference for a type annotation at import time and is stubbed with an empty module.
"""
import math
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
N, W, H, POSE, SCENE_SEED = 6000, 320, 240, 2, 9
N_PIX, N_ROWS = 1024, 128
DEV = "cuda"


def load_reference(ref):
    sys.path.insert(0, ref)
    stub = types.ModuleType("lightning")
    stub.LightningModule = type("LightningModule", (), {})
    sys.modules.setdefault("lightning", stub)
    import b200gs.compat
    b200gs.compat.install()
    from internal.cameras.cameras import Cameras
    from internal.models.vanilla_gaussian import VanillaGaussian
    from internal.renderers.gsplat_renderer import GSPlatRenderer
    from internal.renderers.pypreprocess_gsplat_renderer import PythonPreprocessGSplatRenderer
    from internal.renderers.vanilla_renderer import VanillaRenderer
    from internal.utils.ssim import ssim
    return types.SimpleNamespace(Cameras=Cameras, VanillaGaussian=VanillaGaussian, VanillaRenderer=VanillaRenderer,
                                 GSPlatRenderer=GSPlatRenderer, PythonPreprocessGSplatRenderer=PythonPreprocessGSplatRenderer,
                                 ssim=ssim)


def setup(ref):
    from b200gs.scene import make_scene, ring_pose
    raw = make_scene(N, SCENE_SEED, mean_scale=0.04)
    model = ref.VanillaGaussian(sh_degree=3).instantiate()
    model.setup_from_tensors({k: v.clone() for k, v in raw.items()})
    model.active_sh_degree = 3
    model = model.to(DEV)
    R, T = ring_pose(POSE)
    fx = 0.5 * W / math.tan(math.radians(39.6) * 0.5)
    cams = ref.Cameras(R=R[None], T=T[None], fx=torch.tensor([fx]), fy=torch.tensor([fx]), cx=torch.tensor([W / 2.0]),
                       cy=torch.tensor([H / 2.0]), width=torch.tensor([W], dtype=torch.int32),
                       height=torch.tensor([H], dtype=torch.int32), appearance_id=torch.zeros(1, dtype=torch.int32),
                       normalized_appearance_id=torch.zeros(1), distortion_params=None,
                       camera_type=torch.zeros(1, dtype=torch.int32))
    return model, cams[0].to_device(DEV)


def cotangent():
    return (torch.rand(3, H, W, generator=torch.Generator().manual_seed(1)) * 2 - 1).to(DEV)


def record(d, prefix, out, images, model, vs, pix, rows):
    d[f"{prefix}_keys"] = np.array(sorted(out.keys()))
    for key in images:
        d[f"{prefix}_{key}"] = out[key].detach().reshape(out[key].shape[0], -1)[:, pix].cpu().numpy()
    d[f"{prefix}_radii"] = out["radii"].cpu().numpy()
    for k, p in model.gaussians.items():
        d[f"{prefix}_grad_{k}"] = p.grad[rows].cpu().numpy()
        d[f"{prefix}_gradmax_{k}"] = p.grad.abs().max().cpu().numpy()
        p.grad = None
    d[f"{prefix}_grad_viewspace"] = vs[rows].cpu().numpy()
    d[f"{prefix}_gradmax_viewspace"] = vs.abs().max().cpu().numpy()


def main(ref_path, out_path):
    ref = load_reference(ref_path)
    d = {}
    model, cam = setup(ref)
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    cot = cotangent()

    out = ref.VanillaRenderer()(cam, model, bg)
    out["viewspace_points"].retain_grad()
    (out["render"] * cot).sum().backward()
    pix = torch.randperm(H * W, generator=torch.Generator().manual_seed(2))[:N_PIX].sort().values
    visible = torch.nonzero(out["radii"].cpu() > 0).flatten()
    rows = visible[torch.randperm(visible.numel(), generator=torch.Generator().manual_seed(3))[:N_ROWS]].sort().values
    d["pix"], d["rows"] = pix.numpy(), rows.numpy()
    record(d, "vanilla", out, ("render",), model, out["viewspace_points"].grad, pix, rows)

    out = ref.GSPlatRenderer()(cam, model, bg, render_types=["rgb", "alpha", "acc_depth"])
    out["viewspace_points"].retain_grad()
    ((out["render"] * cot).sum() + out["alpha"].sum() + out["acc_depth"].sum()).backward()
    record(d, "gsplat", out, ("render", "alpha", "acc_depth"), model, out["viewspace_points"].grad, pix, rows)
    d["gsplat_viewspace_points_grad_scale"] = out["viewspace_points_grad_scale"].cpu().numpy()

    with torch.no_grad():
        out = ref.PythonPreprocessGSplatRenderer()(cam, model, bg)
    d["pypreprocess_render"] = out["render"].reshape(3, -1)[:, pix].cpu().numpy()
    d["pypreprocess_visibility_filter"] = out["visibility_filter"].cpu().numpy()

    # the steps of GaussianSplatting.training_step around the renderer, with the reference's model object and ssim
    from b200gs.renderers import B200VanillaRenderer
    model, cam = setup(ref)
    bg = torch.zeros(3, device=DEV)
    renderer = B200VanillaRenderer().to(DEV)
    with torch.no_grad():
        target = renderer(cam, model, bg)["render"].clone()
        model.gaussians["means"].add_(0.003 * torch.randn(N, 3, generator=torch.Generator().manual_seed(4)).to(DEV))
    opt = torch.optim.Adam(model.gaussians.values(), lr=1e-3)
    losses = []
    for _ in range(4):
        out = renderer(cam, model, bg)
        loss = 0.8 * (out["render"] - target).abs().mean() + 0.2 * (1 - ref.ssim(out["render"], target))
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        losses.append(float(loss))
    d["train_losses"] = np.array(losses)
    np.savez_compressed(out_path, **d)
    print("wrote", out_path, "losses", losses)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, f"dropin_n{N}_{W}x{H}.npz"))
