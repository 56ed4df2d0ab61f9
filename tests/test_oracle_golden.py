"""Pin the oracle: its gsplat-mode projection, SH and sort keys must reproduce the golden vectors produced by the
reference's own code (tests/golden/make_golden.py), including the known-answer fixture of the reference's
tests/gaussian_projection_test.py:30-113, and the reference's autograd gradients."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import gs_oracle as O


def _view_from(w2c, fx, fy, cx, cy, W, H):
    w2c = torch.as_tensor(w2c)
    return O.View(int(W), int(H), float(fx), float(fy), float(cx), float(cy), w2c, torch.zeros(4, 4),
                  torch.linalg.inv(w2c)[3, :3], 0.5 * W / fx, 0.5 * H / fy)


def test_known_answer_fixture():
    d = np.load(os.path.join(GOLDEN, "kat_projection.npz"))
    fx, fy, cx, cy, W, H = d["intr"]
    v = _view_from(d["w2c"], fx, fy, cx, cy, W, H)
    p = O.project(O.MODE_GSPLAT, torch.tensor(d["means"]), torch.tensor(d["scales"]), torch.tensor(d["quats"]), v)
    m = p["mask"]
    # literals asserted by the reference test
    assert torch.equal(p["radii"], torch.tensor(d["expect_radii"]))
    assert torch.equal(p["tiles"][m], torch.tensor(d["expect_tiles_masked"]))
    assert torch.allclose(p["comp"][m], torch.tensor(d["expect_comp_masked"]), rtol=1e-5, atol=1e-7)
    assert torch.allclose(p["conic"][m], torch.tensor(d["expect_conic_masked"]), rtol=1e-4, atol=1e-9)
    up = p["cov3d"][m].reshape(-1, 9)[:, [0, 1, 2, 4, 5, 8]]
    assert torch.allclose(up, torch.tensor(d["expect_cov3d_upper_masked"]), rtol=1e-4, atol=1e-9)
    # the literals for xys come from the older NDC variant: current pixel convention = that + 0.5 (gaussian_projection.py:87-88)
    assert torch.allclose(p["xy"][m] - 0.5, torch.tensor(d["expect_xys_masked_old_ndc_variant"]), rtol=2e-5, atol=2e-3)
    # and the live outputs of the reference code
    assert torch.equal(m, torch.tensor(d["mask"]))
    assert torch.allclose(p["xy"], torch.tensor(d["xys"]), rtol=1e-5, atol=1e-3)
    assert torch.allclose(p["depth"], torch.tensor(d["depths"]), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name", ["scene_n256_64x48", "scene_n4096_256x256", "scene_n30000_800x800"])
def test_projection_matches_reference(name):
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    n, W, H, seed, pose = [int(x) for x in d["meta"]]
    from b200gs.scene import make_scene, activate, make_ring_cameras
    sc = activate(make_scene(n, seed, extent=1.3, mean_scale=0.05 if n <= 4096 else 0.01))
    cam = make_ring_cameras(W, H)[pose]
    v = O.make_view(cam.R, cam.T, float(cam.fx), float(cam.fy), float(cam.cx), float(cam.cy), W, H)
    means = sc["means"].clone().requires_grad_(True)
    scales = sc["scales"].clone().requires_grad_(True)
    quats = sc["rotations"].clone().requires_grad_(True)
    p = O.project(O.MODE_GSPLAT, means, scales, quats, v)
    assert torch.equal(p["mask"], torch.tensor(d["mask"]))
    assert torch.equal(p["radii"], torch.tensor(d["radii"]))
    assert torch.equal(p["tiles"], torch.tensor(d["tiles"]))
    assert torch.equal(p["rect_min"], torch.tensor(d["rect_min"]))
    assert torch.equal(p["rect_max"], torch.tensor(d["rect_max"]))
    assert torch.allclose(p["xy"], torch.tensor(d["xys"]), rtol=1e-5, atol=1e-4)
    assert torch.allclose(p["conic"], torch.tensor(d["conic"]), rtol=1e-4, atol=1e-7)
    assert torch.allclose(p["comp"], torch.tensor(d["comp"]), rtol=1e-4, atol=1e-6)
    assert torch.allclose(p["depth"], torch.tensor(d["depths"]), rtol=1e-6, atol=1e-6)
    if "g_means" in d:
        loss = (p["xy"] * torch.tensor(d["cot_xy"])).sum() + (p["depth"] * torch.tensor(d["cot_depth"])).sum() \
            + (p["conic"] * torch.tensor(d["cot_conic"])).sum() + (p["comp"] * torch.tensor(d["cot_comp"])).sum()
        loss.backward()
        for mine, ref in ((means.grad, d["g_means"]), (scales.grad, d["g_scales"]), (quats.grad, d["g_quats"])):
            ref = torch.tensor(ref)
            scale = ref.abs().max()
            assert (mine - ref).abs().max() <= 2e-4 * scale, ((mine - ref).abs().max(), scale)
        # sort keys: the reference's python triple loop
        gx = (W + 15) // 16
        keys, ids = O.build_sort_keys(p["depth"], p["rect_min"], p["rect_max"], p["tiles"], gx)
        # NB: run today, the reference's builder (gaussian_projection.py:199-203) shifts an *int32* tile id by 32, which
        # wraps to 0 — its keys carry only the depth bits.  The emit order / ids / depth bits are pinned against it;
        # the documented (tile_id << 32) part is pinned against an explicit loop below.
        assert torch.equal(keys & 0xFFFFFFFF, torch.tensor(d["sort_key"]))
        assert torch.equal(ids, torch.tensor(d["sort_ids"]))
        if n <= 256:
            exp_tiles = []
            for g in range(n):
                for ty in range(int(p["rect_min"][g, 1]), int(p["rect_max"][g, 1])):
                    for tx in range(int(p["rect_min"][g, 0]), int(p["rect_max"][g, 0])):
                        if bool(p["mask"][g]):
                            exp_tiles.append(ty * gx + tx)
            assert (keys >> 32).tolist() == exp_tiles


@pytest.mark.parametrize("name", ["scene_n256_64x48", "scene_n4096_256x256"])
def test_sh_matches_reference(name):
    d = np.load(os.path.join(GOLDEN, name + ".npz"))
    n, W, H, seed, pose = [int(x) for x in d["meta"]]
    from b200gs.scene import make_scene, activate, make_ring_cameras
    sc = activate(make_scene(n, seed, extent=1.3, mean_scale=0.05))
    cam = make_ring_cameras(W, H)[pose]
    cot = torch.tensor(d["sh_cot"])
    for deg in range(4):
        shs = sc["shs"].clone().requires_grad_(True)
        dirs = sc["means"] - cam.camera_center
        dirs = (dirs / dirs.norm(dim=-1, keepdim=True)).requires_grad_(True)
        rgb = O.eval_sh(deg, shs, dirs)
        assert torch.allclose(rgb, torch.tensor(d[f"sh_rgb_deg{deg}"]), rtol=1e-5, atol=1e-6)
        (torch.clamp_min(rgb + 0.5, 0.0) * cot).sum().backward()
        assert torch.allclose(shs.grad, torch.tensor(d[f"sh_g_shs_deg{deg}"]), rtol=1e-5, atol=1e-6)
        if deg > 0:
            assert torch.allclose(dirs.grad, torch.tensor(d[f"sh_g_dirs_deg{deg}"]), rtol=1e-4, atol=1e-5)


def test_camera_restatement_matches_product_camera():
    from b200gs.scene import make_ring_cameras
    for cam in make_ring_cameras(1920, 1080)[::5]:
        v = O.make_view(cam.R, cam.T, float(cam.fx), float(cam.fy), float(cam.cx), float(cam.cy), 1920, 1080)
        assert torch.allclose(v.world_to_camera, cam.world_to_camera)
        assert torch.allclose(v.full_projection, cam.full_projection, atol=1e-6)
        assert torch.allclose(v.camera_center, cam.camera_center, atol=1e-6)


def test_product_camera_matches_reference_cameras_class():
    """b200gs.cameras.make_camera against what the reference's own Cameras dataclass derives for the same poses
    (tests/golden/make_golden_cameras.py)."""
    from b200gs.scene import make_ring_cameras
    d = np.load(os.path.join(GOLDEN, "cameras_1920x1080.npz"))
    cams = make_ring_cameras(1920, 1080)
    for k in d["poses"].tolist():
        for name in ("world_to_camera", "full_projection", "camera_center", "fov_x", "fov_y"):
            assert torch.equal(torch.from_numpy(d[f"{name}_{k}"]), getattr(cams[k], name)), (name, k)


def test_sh_degree4_matches_reference():
    """Degree 4 (sh_utils.py:102-111), values and gradients, against the reference's eval_sh (tests/golden/make_golden_sh4.py)."""
    d = np.load(os.path.join(GOLDEN, "sh_deg4.npz"))
    shs = torch.tensor(d["shs"]).requires_grad_(True)
    dirs = torch.tensor(d["dirs"]).requires_grad_(True)
    rgb = O.eval_sh(4, shs, dirs)
    assert torch.allclose(rgb, torch.tensor(d["rgb"]), rtol=1e-5, atol=1e-6)
    (rgb * torch.tensor(d["cot"])).sum().backward()
    assert torch.allclose(shs.grad, torch.tensor(d["g_shs"]), rtol=1e-5, atol=1e-6)
    assert torch.allclose(dirs.grad, torch.tensor(d["g_dirs"]), rtol=1e-4, atol=1e-5)
