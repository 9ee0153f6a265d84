"""Drop-in installation behind the reference's by-name seam.

The reference binds the hot-path callables by name at import time (train/trainer.py:46-54,
utils/render_utils.py:24-25, utils/validation_renderer.py:16-24) and its own test patches exactly that seam
(tests/unit/test_trainer.py:172).  ``install()`` rebinds those names to this package's CUDA-backed
implementations so ``scripts/train_nerf.py --vanilla`` runs unmodified on a B200."""
from __future__ import annotations

import importlib
import sys
import types

from . import encoders, mlps, rays, render, sampling

_BINDINGS = {
    "nerf_sandbox.source.train.trainer": {
        "PositionalEncoder": encoders.PositionalEncoder, "get_vanilla_nerf_encoders": encoders.get_vanilla_nerf_encoders,
        "NeRF": mlps.NeRF, "log_nerf_arch": mlps.log_nerf_arch, "volume_render_rays": render.volume_render_rays,
        "nerf_forward_pass": render.nerf_forward_pass, "sample_pdf": sampling.sample_pdf,
        "get_camera_rays": rays.get_camera_rays},
    "nerf_sandbox.source.utils.render_utils": {
        "get_camera_rays": rays.get_camera_rays, "render_pose": rays.render_pose,
        "sample_pdf": sampling.sample_pdf, "volume_render_rays": render.volume_render_rays,
        "nerf_forward_pass": render.nerf_forward_pass, "render_image_chunked": render.render_image_chunked},
    "nerf_sandbox.source.utils.validation_renderer": {"render_image_chunked": render.render_image_chunked,
                                                      "render_pose": rays.render_pose, "get_camera_rays": rays.get_camera_rays},
    "nerf_sandbox.source.data.samplers": {"get_camera_rays": rays.get_camera_rays},
    "nerf_sandbox.source.utils.ray_utils": {"get_camera_rays": rays.get_camera_rays},
    "nerf_sandbox.source.models.encoders": {
        "PositionalEncoder": encoders.PositionalEncoder, "get_vanilla_nerf_encoders": encoders.get_vanilla_nerf_encoders},
    "nerf_sandbox.source.models.mlps": {"NeRF": mlps.NeRF, "log_nerf_arch": mlps.log_nerf_arch},
    "nerf_sandbox.source.utils.sampling_utils": {"sample_pdf": sampling.sample_pdf},
}


_ORIGINALS = {}          # (module, name) -> the reference's own object, for uninstall()


def uninstall() -> None:
    """Put the reference's own callables back (e.g. to time its CPU path in the same process after a drop-in run)."""
    for (modname, n), obj in _ORIGINALS.items():
        mod = sys.modules.get(modname)
        if mod is not None:
            setattr(mod, n, obj)
    _ORIGINALS.clear()
    trainer_mod = sys.modules.get("nerf_sandbox.source.train.trainer")
    if trainer_mod is not None:
        cur = trainer_mod.Trainer._train_step
        trainer_mod.Trainer._train_step = getattr(cur, "_nsb_original", cur)


def _imageio_shim():
    """render_utils.py:20 and the loaders import imageio at module scope; when it is not installed provide a stand-in:
    PNG read/write through PIL when that is present (enough for the Blender loader and the validation PNGs), video export
    unavailable.  Image IO is outside the hot path."""
    if "imageio" in sys.modules:
        return
    try:
        importlib.import_module("imageio")
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


def _engine_for(tr):
    """Fused-step engine for a reference Trainer, or False when its configuration is not the fused kernels' (foreign models
    or encoders, non-CUDA device, mixed modes): then the reference's own _train_step keeps running on the rebound callables."""
    from .render import _is_fused_triplet
    from .trainer import VanillaTrainer
    try:
        ok = (_is_fused_triplet(tr.pos_enc, tr.dir_enc, tr.nerf_c) and _is_fused_triplet(tr.pos_enc, tr.dir_enc, tr.nerf_f)
              and tr.nerf_c.mode == tr.nerf_f.mode and str(tr.device).startswith("cuda")
              and (tr.sigma_activation or "relu").lower() in ("relu", "softplus") and int(tr.nc) >= 2 and int(tr.nf) >= 1)
        if not ok:
            return False
        return VanillaTrainer.step_engine(tr.nerf_c, tr.nerf_f, nc=tr.nc, nf=tr.nf, near=tr.samp_near, far=tr.samp_far,
                                          white_bkgd=tr.white_bkgd, raw_noise_std=tr.raw_noise_std, infinite_last_bin=tr.infinite_last_bin,
                                          det_fine=tr.det_fine, sigma_activation=tr.sigma_activation,
                                          seed=int(getattr(getattr(tr, "cfg", None), "seed", 0) or 0))
    except AttributeError:
        return False


def _fused_train_step(original):
    """Trainer._train_step (train/trainer.py:876-1013) as ONE library call (nsb_train_fwd_bwd: coarse pass, resampling, fine
    pass, loss and the whole backward), returning the same dict with an autograd `loss` -- the caller's
    `scaler.scale(loss).backward()` only scales the gradients the step already computed.  Steps on which the reference prints
    its diagnostics (step 100, every 500th: trainer.py:886-893, :937-979) run the original method."""
    from . import _hooks
    from .trainer import BATCH_KEYS

    def _train_step(self, batch):
        eng = self.__dict__.get("_nsb_engine")
        if eng is None:
            eng = self.__dict__["_nsb_engine"] = _engine_for(self)
        step = int(getattr(self, "global_step", 0) or 0)
        if eng is False or step == 100 or step % 500 == 0:
            return original(self, batch)
        eng.global_step = step                                   # Philox streams of the in-kernel draws follow the loop's step count
        B = batch["rays_o_marching"].shape[0]
        dev = batch["rays_o_marching"].device
        draws = None
        if _hooks.jitter is not None or _hooks.uniform is not None or _hooks.normal is not None:
            draws = {"U": _hooks.jitter(B, eng.nc, dev) if _hooks.jitter else None,
                     "noise_c": _hooks.normal(B * eng.nc, dev) if _hooks.normal else None,
                     "u_fine": _hooks.uniform(B, eng.nf, dev) if _hooks.uniform else None,
                     "noise_f": _hooks.normal(B * (eng.nc + eng.nf), dev) if _hooks.normal else None}
        return eng._train_step({k: batch[k] for k in BATCH_KEYS}, draws)
    _train_step._nsb_original = original
    return _train_step


def install(verbose: bool = False, mode: str | None = None, fuse_train_step: bool = True) -> dict:
    """Rebind the reference's names; returns {module: [names rebound]}.  The reference package must be importable.

    ``mode`` ("bf16" = bf16 tensor-core kernels, "fp32" = parity kernels; default: NSB_MODE, else "fp32") becomes the
    arithmetic mode of every ``NeRF`` the reference builds afterwards -- its Trainer passes no mode (train/trainer.py:326-341),
    so this is how ``train_nerf.py --vanilla`` reaches the tensor-core path.

    ``fuse_train_step`` additionally puts the fused step behind ``Trainer._train_step`` (the last row of the boundary table,
    SURVEY section 8b): the reference's loop, sampler, AMP scaler, optimiser, logging and validation run unchanged, but one
    library call does forward + backward.  False keeps the reference's own ``_train_step`` body (on the rebound callables)."""
    if mode is not None:
        mlps.set_default_mode(mode)
    _imageio_shim()
    done = {}
    for modname, names in _BINDINGS.items():
        mod = importlib.import_module(modname)
        for n, obj in names.items():
            if (modname, n) not in _ORIGINALS and hasattr(mod, n):
                _ORIGINALS[(modname, n)] = getattr(mod, n)
            setattr(mod, n, obj)
        done[modname] = sorted(names)
        if verbose:
            print(f"[nerf_sandbox_b200] {modname}: {', '.join(sorted(names))}")
    trainer_mod = importlib.import_module("nerf_sandbox.source.train.trainer")
    cur = trainer_mod.Trainer._train_step
    orig = getattr(cur, "_nsb_original", cur)
    trainer_mod.Trainer._train_step = _fused_train_step(orig) if fuse_train_step else orig
    if fuse_train_step:
        done["nerf_sandbox.source.train.trainer"] = sorted(done["nerf_sandbox.source.train.trainer"] + ["Trainer._train_step"])
    return done
