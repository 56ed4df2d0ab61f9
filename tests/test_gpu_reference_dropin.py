"""Drop-in evidence: the b200gs plug-in renderers give the image and gradients that the reference's UNMODIFIED classes —
``internal.renderers.vanilla_renderer.VanillaRenderer``, ``internal.renderers.gsplat_renderer.GSPlatRenderer``,
``internal.renderers.pypreprocess_gsplat_renderer.PythonPreprocessGSplatRenderer``, ``internal.models.vanilla_gaussian.
VanillaGaussian``, ``internal.cameras.cameras.Cameras``, ``internal.utils.ssim`` — produced for the same scene when they ran
on the b200gs kernels through ``b200gs.compat.install()``.  Those outputs are frozen in tests/golden/dropin_n6000_320x240.npz
(tests/golden/make_golden_dropin.py) at a fixed sample of pixels and visible Gaussians; relative errors are taken against the
full-size maxima stored with them.  ``SyntheticGaussians`` and ``make_camera`` stand in for the reference's model and
camera objects (same raw parameters and getters; the camera fields are pinned bit for bit by tests/test_oracle_golden.py)."""
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLDEN, "dropin_n6000_320x240.npz"))


def _setup(n=6000, W=320, H=240, pose=2):
    from b200gs.cameras import make_camera
    from b200gs.scene import SyntheticGaussians, make_scene, ring_pose
    raw = make_scene(n, 9, mean_scale=0.04)
    model = SyntheticGaussians(raw).to(DEV)
    R, T = ring_pose(pose)
    fx = 0.5 * W / math.tan(math.radians(39.6) * 0.5)
    cam = make_camera(R, T, fx, fx, W / 2.0, H / 2.0, W, H)
    return raw, model, cam.to_device(DEV), W, H


def _sampled(img, ref):
    return img.detach().reshape(img.shape[0], -1)[:, torch.from_numpy(ref["pix"]).to(img.device)].cpu()


def _check_grads(ref, prefix, model, vs):
    rows = torch.from_numpy(ref["rows"]).to(DEV)
    for k, p in model.gaussians.items():
        assert _rel(p.grad[rows].cpu(), ref[f"{prefix}_grad_{k}"], ref[f"{prefix}_gradmax_{k}"]) < 2e-3, k
    assert _rel(vs[rows].cpu(), ref[f"{prefix}_grad_viewspace"], ref[f"{prefix}_gradmax_viewspace"]) < 2e-3


def _rel(a, b, bmax):
    return float((a - torch.from_numpy(b)).abs().max() / max(float(bmax), 1e-30))


def test_reference_vanilla_renderer_runs_on_b200gs(ref):
    from b200gs.renderers import B200VanillaRenderer
    raw, model, cam, W, H = _setup()
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    cot = (torch.rand(3, H, W, generator=torch.Generator().manual_seed(1)) * 2 - 1).to(DEV)

    out = B200VanillaRenderer().to(DEV)(cam, model, bg)           # our plug-in (fused-activation path: it IS the vanilla model)
    out["viewspace_points"].retain_grad()
    (out["render"] * cot).sum().backward()
    vs = out["viewspace_points"].grad
    assert out["render"].shape == (3, H, W) and out["radii"].dtype == torch.int32
    assert torch.equal(out["visibility_filter"], out["radii"] > 0)
    assert float(vs[:, 2].abs().max()) == 0 and float(vs[:, :2].abs().max()) > 0
    assert sorted(out.keys()) == ref["vanilla_keys"].tolist()
    assert float((_sampled(out["render"], ref) - torch.from_numpy(ref["vanilla_render"])).abs().max()) < 2e-4
    assert torch.equal(out["radii"].cpu(), torch.from_numpy(ref["vanilla_radii"]))
    _check_grads(ref, "vanilla", model, vs)


def test_reference_gsplat_renderer_runs_on_b200gs(ref):
    from b200gs.renderers import B200GSplatRenderer
    raw, model, cam, W, H = _setup()
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    cot = (torch.rand(3, H, W, generator=torch.Generator().manual_seed(1)) * 2 - 1).to(DEV)

    out = B200GSplatRenderer().to(DEV)(cam, model, bg, render_types=["rgb", "alpha", "acc_depth"])
    out["viewspace_points"].retain_grad()
    ((out["render"] * cot).sum() + out["alpha"].sum() + out["acc_depth"].sum()).backward()
    assert out["render"].shape == (3, H, W) and out["alpha"].shape == (1, H, W)
    assert sorted(out.keys()) == ref["gsplat_keys"].tolist()
    for key in ("render", "alpha", "acc_depth"):
        want = torch.from_numpy(ref[f"gsplat_{key}"])
        assert float((_sampled(out[key], ref) - want).abs().max()) < 2e-4 * max(1.0, float(want.abs().max())), key
    assert torch.equal(out["radii"].cpu(), torch.from_numpy(ref["gsplat_radii"]))
    assert torch.equal(out["viewspace_points_grad_scale"].cpu(), torch.from_numpy(ref["gsplat_viewspace_points_grad_scale"]))
    _check_grads(ref, "gsplat", model, out["viewspace_points"].grad)


def test_reference_python_preprocess_renderer_agrees(ref):
    """configs[0] of BASELINE.json names the reference's PythonPreprocessGSplatRenderer (its own torch projection,
    internal/utils/gaussian_projection.py, feeding the gsplat rasterizer) as the CPU-runnable reference path.  Its picture (torch
    projection on the GPU, our SH + binning + blend underneath through the aliased gsplat modules) is compared with
    B200GSplatRenderer, whose K1 restates the same projection: the two images must agree to fp32-projection noise (the python
    projection is fp32; K1 evaluates the same formulas in fp64)."""
    from b200gs.renderers import B200GSplatRenderer
    raw, model, cam, W, H = _setup()
    bg = torch.tensor([0.1, 0.2, 0.3], device=DEV)
    with torch.no_grad():
        out = B200GSplatRenderer().to(DEV)(cam, model, bg)
    assert out["render"].shape == (3, H, W)
    diff = (torch.from_numpy(ref["pypreprocess_render"]) - _sampled(out["render"], ref)).abs()
    assert float(diff.mean()) < 2e-5 and float(diff.max()) < 2e-2      # isolated radius/threshold flips of the fp32 python projection
    assert int((diff > 1e-3).sum()) < 0.002 * diff.numel()
    same_vis = (torch.from_numpy(ref["pypreprocess_visibility_filter"]) == out["visibility_filter"].cpu()).float().mean()
    assert float(same_vis) > 0.999


def test_training_step_shape_with_reference_objects(ref):
    """The sequence GaussianSplatting.training_step performs around the renderer (internal/gaussian_splatting.py:341-397):
    forward -> L1 + (1 - SSIM) loss -> retain_grad -> backward -> the density controller's read of
    viewspace_points.grad[visibility_filter, :2] / radii (vanilla_density_controller.py:101-123) -> Adam step.  The SSIM is
    oracle/loss_oracle.py on the CPU (pinned to the reference's ssim by tests/test_loss_oracle_golden.py); the losses must follow
    the ones the reference's model object and ssim gave."""
    from oracle.loss_oracle import ssim
    from b200gs.renderers import B200VanillaRenderer
    raw, model, cam, W, H = _setup()
    bg = torch.tensor([0.0, 0.0, 0.0], device=DEV)
    renderer = B200VanillaRenderer().to(DEV)
    with torch.no_grad():
        target = renderer(cam, model, bg)["render"].clone()
        noise = torch.randn(model.gaussians["means"].shape, generator=torch.Generator().manual_seed(4))
        model.gaussians["means"].add_(0.003 * noise.to(DEV))
    opt = torch.optim.Adam(model.gaussians.values(), lr=1e-3)
    losses = []
    max_radii = torch.zeros(model.gaussians["means"].shape[0], device=DEV)
    for step in range(4):
        out = renderer(cam, model, bg)
        loss = 0.8 * (out["render"] - target).abs().mean() + 0.2 * (1 - ssim(out["render"].cpu(), target.cpu()))
        out["viewspace_points"].retain_grad()
        loss.backward()
        vis, radii = out["visibility_filter"], out["radii"]
        grad_norm = out["viewspace_points"].grad[vis, :2].norm(dim=-1)
        assert bool(torch.isfinite(grad_norm).all()) and grad_norm.numel() == int(vis.sum())
        max_radii[vis] = torch.max(max_radii[vis], radii[vis].float())
        opt.step()
        opt.zero_grad(set_to_none=True)
        losses.append(float(loss))
    assert losses[-1] < losses[0]
    np.testing.assert_allclose(losses, ref["train_losses"], rtol=1e-3)
