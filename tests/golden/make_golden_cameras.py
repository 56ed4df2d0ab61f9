"""Freeze what the reference's own ``Cameras`` dataclass (internal/cameras/cameras.py, loaded by file path from a checkout of
the reference) derives for three poses of the 1920x1080 camera ring: world_to_camera, full_projection, camera_center and the
two fields of view.  tests/test_oracle_golden.py compares b200gs.cameras.make_camera with them bit for bit.

    python tests/golden/make_golden_cameras.py <reference checkout>    -> tests/golden/cameras_1920x1080.npz
"""
import importlib.util
import math
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
POSES = (0, 5, 17)
FIELDS = ("world_to_camera", "full_projection", "camera_center", "fov_x", "fov_y")


def main(ref):
    spec = importlib.util.spec_from_file_location("ref_cameras", os.path.join(ref, "internal", "cameras", "cameras.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    from b200gs.scene import ring_pose
    W, H = 1920, 1080
    fx = 0.5 * W / math.tan(math.radians(39.6) * 0.5)
    d = {"poses": np.array(POSES, dtype=np.int64)}
    for k in POSES:
        R, T = ring_pose(k)
        cams = m.Cameras(R=R[None], T=T[None], fx=torch.tensor([fx]), fy=torch.tensor([fx]), cx=torch.tensor([W / 2.0]),
                         cy=torch.tensor([H / 2.0]), width=torch.tensor([W], dtype=torch.int32),
                         height=torch.tensor([H], dtype=torch.int32), appearance_id=torch.zeros(1, dtype=torch.int32),
                         normalized_appearance_id=torch.zeros(1), distortion_params=None, camera_type=torch.zeros(1, dtype=torch.int32))
        for name in FIELDS:
            d[f"{name}_{k}"] = getattr(cams[0], name).numpy()
    np.savez_compressed(os.path.join(HERE, "cameras_1920x1080.npz"), **d)


if __name__ == "__main__":
    main(sys.argv[1])
