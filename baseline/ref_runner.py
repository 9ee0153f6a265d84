"""The reference's OWN implementation of the path, run unmodified on the host cores.

The reference package lives in ``oracle/_ref/nerf_sandbox/`` (git-ignored: its sources never enter the history).
`pip install --target oracle/_ref <reference checkout>` is refused by the reference's setup.py (:31-42 raises for any
Python other than 3.8 / 3.10), so ``vendor()`` does what that install would have done for a pure-Python package: it
copies the package tree ``nerf_sandbox/`` of a reference checkout as it is into ``oracle/_ref/``.  The checkout is the
one ``NSB_REFERENCE_SRC`` names, else BASELINE.json's ``reference_path``.  Nothing here is on the product path:
``bench.py --impl reference`` / the ``cpu_baseline`` leg time it, and the drop-in tests (tests/test_gpu_dropin.py,
tests/test_install.py) drive the reference's own ``Trainer._train_step`` through ``install()`` with it.
"""
from __future__ import annotations

import json
import os
import shutil
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def reference_checkout() -> str:
    """Root of a reference checkout (the directory holding ``nerf_sandbox/``): $NSB_REFERENCE_SRC, else
    BASELINE.json's reference_path."""
    return os.environ.get("NSB_REFERENCE_SRC") or json.load(open(os.path.join(ROOT, "BASELINE.json")))["reference_path"]


def vendor(verbose: bool = False) -> bool:
    """Copy <reference checkout>/nerf_sandbox -> oracle/_ref/nerf_sandbox when the checkout exists.  True if _ref holds
    the reference afterwards."""
    src = os.path.join(reference_checkout(), "nerf_sandbox")
    dst = os.path.join(REF_DIR, "nerf_sandbox")
    if os.path.isdir(src) and os.path.realpath(src) != os.path.realpath(dst):
        if os.path.isdir(dst):
            shutil.rmtree(dst)
        os.makedirs(REF_DIR, exist_ok=True)
        shutil.copytree(src, dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
        if verbose:
            print(f"vendored {src} -> {dst}")
    return available()


def available() -> bool:
    return os.path.isfile(os.path.join(REF_DIR, "nerf_sandbox", "source", "train", "trainer.py"))


def imageio_shim() -> None:
    """utils/render_utils.py:20 and the loaders import imageio at module scope; it is not installed here.  Stand-in: PNG
    read/write through PIL (what the Blender loader and the validation PNGs need); video export unavailable."""
    if "imageio" in sys.modules:
        return
    try:
        __import__("imageio")
    except ImportError:
        m = types.ModuleType("imageio"); m.v2 = types.ModuleType("imageio.v2")

        def _missing(*a, **k):
            raise RuntimeError("imageio is not installed: image/video export is unavailable")
        imread = imwrite = _missing
        try:
            import numpy as np
            from PIL import Image

            def imread(path, *a, **k):
                return np.array(Image.open(path))

            def imwrite(path, arr, *a, **k):
                Image.fromarray(np.asarray(arr)).save(str(path))
        except ImportError:
            pass
        m.imread = m.v2.imread = imread
        m.imwrite = m.v2.imwrite = imwrite
        m.mimwrite = m.v2.mimwrite = m.get_writer = m.v2.get_writer = _missing
        sys.modules["imageio"], sys.modules["imageio.v2"] = m, m.v2


def import_reference():
    """Put oracle/_ref on sys.path and return the reference's (trainer, render_utils) modules."""
    if not available():
        raise RuntimeError("oracle/_ref holds no reference: run __graft_entry__.build() where a reference checkout exists "
                           "(NSB_REFERENCE_SRC, else BASELINE.json's reference_path)")
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    imageio_shim()
    from nerf_sandbox.source.train import trainer as TR
    from nerf_sandbox.source.utils import render_utils as RU
    return TR, RU


def make_namespace(TR, device, nerf_c, nerf_f, pos_enc, dir_enc, *, nc=64, nf=128, near=2.0, far=6.0, use_ndc=False,
                   amp=False, global_step=1):
    """The attributes Trainer._train_step reads from ``self`` (train/trainer.py:876-1013), with the values the vanilla
    profile gives them (trainer.py:277-291, :411-416; train_nerf.py:275, 281)."""
    from types import SimpleNamespace
    return SimpleNamespace(use_ndc=use_ndc, global_step=global_step, device=device, amp=amp, nc=nc, nf=nf, det_fine=False,
                           samp_near=near, samp_far=far, pos_enc=pos_enc, dir_enc=dir_enc, nerf_c=nerf_c, nerf_f=nerf_f,
                           white_bkgd=True, sigma_activation="relu", raw_noise_std=1.0, train_mlp_chunk=0,
                           infinite_last_bin=True)


def make_cpu_step(batch_fn, *, nc=64, nf=128, threads=None, seed=0):
    """Returns (step, info): ``step()`` runs one full optimisation step of the reference on the CPU in fp32 --
    Trainer._train_step (unbound, on a namespace) + loss.backward() + torch.optim.Adam.step(), i.e. the loop body
    train/trainer.py:702-725 with amp off (what the reference does on a CPU device, trainer.py:396-397) -- on the batch
    ``batch_fn(step_index)`` returns (dict of numpy arrays with the trainer's batch keys)."""
    import torch
    TR, _ = import_reference()
    inst = sys.modules.get("nerf_sandbox_b200.install")
    if inst is not None:
        inst.uninstall()                       # this arm times the reference's OWN callables, never the rebound ones
    from nerf_sandbox.source.models.encoders import get_vanilla_nerf_encoders
    from nerf_sandbox.source.models.mlps import NeRF
    threads = int(threads or os.cpu_count() or 1)
    torch.set_num_threads(threads)
    torch.manual_seed(seed)
    pos_enc, dir_enc = get_vanilla_nerf_encoders()
    nerf_c = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu")          # trainer.py:326-341
    nerf_f = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu")
    with torch.no_grad():                      # random-init density is degenerate (SURVEY 8c): same bias as our arm
        nerf_c.sigma_out.bias.fill_(0.3); nerf_f.sigma_out.bias.fill_(0.3)
    opt = torch.optim.Adam(list(nerf_c.parameters()) + list(nerf_f.parameters()), lr=5e-4)      # trainer.py:383-386
    ns = make_namespace(TR, torch.device("cpu"), nerf_c, nerf_f, pos_enc, dir_enc, nc=nc, nf=nf)
    state = {"i": 0}

    def step():
        b = {k: torch.from_numpy(v) for k, v in batch_fn(state["i"]).items()}
        state["i"] += 1
        ns.global_step = state["i"] if state["i"] % 500 else state["i"] + 1     # skip the every-500-steps diagnostics
        opt.zero_grad(set_to_none=True)
        out = TR.Trainer._train_step(ns, b)
        out["loss"].backward()
        opt.step()
        return float(out["loss"].detach())
    return step, {"threads": torch.get_num_threads(), "torch": torch.__version__}


def make_cpu_render(rays_fn, *, nc=64, nf=128, near=2.0, far=6.0, threads=None, seed=0, eval_chunk=16384):
    """Returns (render, info): ``render()`` runs the reference's render_image_chunked (utils/render_utils.py:285-424:
    coarse pass, sample_pdf, merge, fine pass; fp32 on a CPU device) on the rays ``rays_fn()`` returns -- a dict with the
    trainer's batch keys for an H x W tile, H * W rays -- and returns the rgb image.  SURVEY 8d's eval CPU baseline."""
    import torch
    _, RU = import_reference()
    inst = sys.modules.get("nerf_sandbox_b200.install")
    if inst is not None:
        inst.uninstall()
    from nerf_sandbox.source.models.encoders import get_vanilla_nerf_encoders
    from nerf_sandbox.source.models.mlps import NeRF
    threads = int(threads or os.cpu_count() or 1)
    torch.set_num_threads(threads)
    torch.manual_seed(seed)
    pos_enc, dir_enc = get_vanilla_nerf_encoders()
    nerf_c = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu")
    nerf_f = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu")
    with torch.no_grad():
        nerf_c.sigma_out.bias.fill_(0.3); nerf_f.sigma_out.bias.fill_(0.3)
    nerf_c.eval(); nerf_f.eval()

    def render():
        r = {k: torch.from_numpy(v) for k, v in rays_fn().items()}
        n = r["rays_o_marching"].shape[0]
        H = int(round(n ** 0.5))
        while n % H:
            H -= 1
        W = n // H
        out = RU.render_image_chunked(r["rays_o_marching"], r["rays_d_marching_unit"], r["rays_d_marching_norm"], H, W, near, far,
                                      pos_enc, dir_enc, nerf_c, nerf_f, nc, nf, True, torch.device("cpu"), eval_chunk=eval_chunk,
                                      perturb=False, sigma_activation="relu", viewdirs_world_unit=r["rays_d_world_unit"],
                                      infinite_last_bin=True)
        return out["rgb"]
    return render, {"threads": torch.get_num_threads(), "torch": torch.__version__}
