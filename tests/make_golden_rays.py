"""tests/golden/rays.npz from the unmodified reference get_camera_rays (utils/ray_utils.py).  Needs a reference checkout (see make_golden.py)."""
import os, sys
import numpy as np
import torch
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from baseline import ref_runner  # noqa: E402
REF_CHECKOUT = ref_runner.reference_checkout()
if not os.path.isdir(os.path.join(REF_CHECKOUT, "nerf_sandbox")):
    sys.exit(f"no reference checkout at {REF_CHECKOUT}: set NSB_REFERENCE_SRC to a checkout of evan-wes/nerf-sandbox")
sys.path.insert(0, REF_CHECKOUT)
from nerf_sandbox.source.utils.ray_utils import get_camera_rays  # noqa: E402

rng = np.random.default_rng(77)
out = {}
def pose(r):
    c = 4.0311 * r.standard_normal(3); c /= np.linalg.norm(c) / 4.0311
    f = -c / np.linalg.norm(c); rt = np.cross(f, [0, 0, 1.0]); rt /= np.linalg.norm(rt); up = np.cross(rt, f)
    m = np.eye(4, dtype=np.float32); m[:3, 0], m[:3, 1], m[:3, 2], m[:3, 3] = rt, up, -f, c
    return m
cases = [("blender", dict(H=12, W=10, f=1111.111 / 80, conv="opengl", pc=True, ndc=False, near=2.0, px=False, c2w=pose(rng))),
         ("llff_ndc", dict(H=12, W=16, f=407.6 / 32, conv="opengl", pc=True, ndc=True, near=1.0, px=False,
                           c2w=np.array([[1, 0, 0, .1], [0, 1, 0, -.2], [0, 0, 1, .05]], dtype=np.float32))),
         ("opencv_px", dict(H=20, W=30, f=25.0, conv="opencv", pc=False, ndc=False, near=1.0, px=True, c2w=pose(rng)[:3])),
         ("p3d_ndc_px", dict(H=20, W=30, f=25.0, conv="pytorch3d", pc=True, ndc=True, near=0.5, px=True,
                             c2w=np.array([[0.98, 0.1, 0.17, .3], [-0.1, 0.99, 0.0, .1], [-0.17, -0.02, 0.98, -.1], [0, 0, 0, 1]], dtype=np.float32)))]
out["names"] = np.array([c[0] for c in cases])
for name, c in cases:
    K = np.array([[c["f"], 0, c["W"] / 2], [0, c["f"] * 1.02, c["H"] / 2], [0, 0, 1]], dtype=np.float32)
    px = rng.integers(0, [c["W"], c["H"]], size=(40, 2)).astype(np.float32) if c["px"] else None
    r = get_camera_rays(c["H"], c["W"], K, c["c2w"], device="cpu", convention=c["conv"], pixel_center=c["pc"], as_ndc=c["ndc"],
                        near_plane=c["near"], pixels_xy=px)
    out.update({f"{name}_K": K, f"{name}_c2w": c["c2w"], f"{name}_H": c["H"], f"{name}_W": c["W"], f"{name}_conv": c["conv"],
                f"{name}_pc": c["pc"], f"{name}_ndc": c["ndc"], f"{name}_near": c["near"]})
    if px is not None:
        out[f"{name}_px"] = px
    for i, t in enumerate(r):
        out[f"{name}_out{i}"] = t.numpy()
np.savez(os.path.join(HERE, "golden", "rays.npz"), **out)
print("wrote rays.npz", os.path.getsize(os.path.join(HERE, "golden", "rays.npz")))
