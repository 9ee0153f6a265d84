"""Device-resident pixel/ray batch sampler with the reference's interface (data/samplers.py:22-290).

The reference gathers pixels with host-side index generation, a `.cpu()` sync per batch (samplers.py:162) and a
`get_camera_rays` call; here the frames live in HBM and one kernel draws pixels (Philox), composites RGBA on white and
emits the rays -- the loop feeding `VanillaTrainer.step` never touches the host."""
from __future__ import annotations

from typing import Dict, Iterator, Optional

import numpy as np
import torch

from . import _lib
from .rays import _CONV, PoseRaysFn


class RandomPixelRaySampler:
    """Same constructor arguments and batch keys as the reference's RandomPixelRaySampler.  `scene` needs
    `.frames` (objects with .image (H,W,3|4), .K (3,3), .c2w (3|4,4)) and `.white_bkgd`."""

    def __init__(self, scene, rays_per_batch: int = 2048, device=None, white_bg_composite: Optional[bool] = None,
                 cache_images_on_device: bool = True, sample_from_single_frame: bool = False, precrop_iters: int = 0,
                 precrop_frac: float = 0.5, convention: str = "opengl", as_ndc: bool = False, near_plane: float = 1.0,
                 seed: int = 0) -> None:
        self.scene = scene
        self.B = int(rays_per_batch)
        self.device = torch.device(device) if device is not None else torch.device("cuda")
        if self.device.type != "cuda":
            raise RuntimeError("nerf_sandbox_b200 samples ray batches on CUDA devices only (no CPU fallback)")
        self.white_bkgd = scene.white_bkgd if white_bg_composite is None else bool(white_bg_composite)
        conv = (convention or "opengl").lower()
        if conv not in _CONV:
            raise ValueError(f"Unknown convention '{convention}'")
        self.convention, self.as_ndc, self.near_plane = conv, bool(as_ndc), float(near_plane)
        self.sample_from_single_frame = bool(sample_from_single_frame)
        self.precrop_iters, self.precrop_frac = int(precrop_iters), float(precrop_frac)
        self._global_step, self.seed = 0, int(seed)
        self._rng = np.random.default_rng(seed)
        imgs = [np.asarray(f.image, dtype=np.float32) for f in scene.frames]
        if any(im.shape != imgs[0].shape for im in imgs):
            raise ValueError("all frames must share one image shape")
        stack = np.stack(imgs)
        if stack.max() > 1.5:                                        # samplers.py:162-163
            stack = stack / 255.0
        self.H, self.W, self.C = int(stack.shape[1]), int(stack.shape[2]), int(stack.shape[3])
        self._imgs = torch.from_numpy(np.ascontiguousarray(stack)).to(self.device)
        Ks = np.stack([[f.K[0][0], f.K[1][1], f.K[0][2], f.K[1][2]] for f in scene.frames]).astype(np.float32)
        c2ws = np.stack([np.asarray(f.c2w, dtype=np.float32)[:3, :4].reshape(12) for f in scene.frames])
        self._Ks = torch.from_numpy(Ks).to(self.device)
        self._c2ws = torch.from_numpy(np.ascontiguousarray(c2ws)).to(self.device)
        self.F = len(imgs)

    def _current_crop_bounds(self):                                  # samplers.py:119-127
        H, W = self.H, self.W
        if self._global_step < self.precrop_iters and 0.0 < self.precrop_frac < 1.0:
            f = self.precrop_frac
            return int(H * 0.5 * (1.0 - f)), int(H * 0.5 * (1.0 + f)), int(W * 0.5 * (1.0 - f)), int(W * 0.5 * (1.0 + f))
        return 0, H, 0, W

    def next_batch(self, with_pixels: bool = False, c2ws: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """One batch of `rays_per_batch` rays.  ``c2ws`` ([F,3,4] or [F,4,4] CUDA tensor on the sampler's device) replaces the
        scene's poses for this draw; when it requires grad (and grad mode is on) the six ray outputs backpropagate into it
        through nsb_camera_rays_bwd, using the pixels and frame ids this draw made -- per-frame pose refinement (BARF-style).
        The gradient is exact for the rays themselves.  Downstream, the render path gives no gradient to the ray norms, so for
        NDC rays (``as_ndc``), whose marching norm depends on the pose, the pose gradient of a rendering loss is incomplete."""
        poses = self._c2ws
        if c2ws is not None:
            dev = self.device if self.device.index is not None else torch.device("cuda", torch.cuda.current_device())
            if not isinstance(c2ws, torch.Tensor) or c2ws.device != dev:
                raise ValueError(f"c2ws must be a tensor on {self.device}")
            if c2ws.dim() != 3 or c2ws.shape[0] != self.F or tuple(c2ws.shape[1:]) not in {(3, 4), (4, 4)}:
                raise ValueError(f"c2ws must be [{self.F},3,4] or [{self.F},4,4], got {tuple(c2ws.shape)}")
            poses = c2ws.detach()[:, :3, :4].to(torch.float32).contiguous().reshape(self.F, 12)
        grad = c2ws is not None and torch.is_grad_enabled() and c2ws.requires_grad
        h0, h1, w0, w1 = self._current_crop_bounds()
        fid = int(self._rng.integers(self.F)) if self.sample_from_single_frame else -1
        B, dev = self.B, self.device
        e = lambda k: torch.empty((B, k), device=dev, dtype=torch.float32)
        rgb = e(3)
        px = e(2) if (with_pixels or grad) else None                 # the backward needs what this draw picked
        fids = torch.empty((B,), device=dev, dtype=torch.int32) if (with_pixels or grad) else None

        def run():
            rays = (e(3), e(3), e(1), e(3), e(3), e(1))
            _lib.check(_lib.lib().nsb_sample_pixel_batch(
                _lib.ptr(self._imgs), self.F, self.H, self.W, self.C, _lib.ptr(self._Ks), _lib.ptr(poses), fid, h0, h1, w0, w1,
                int(self.white_bkgd), _CONV[self.convention], int(self.as_ndc), self.near_plane, B, self.seed, self._global_step,
                _lib.ptr(rgb), _lib.ptr(px), _lib.ptr(fids), *[_lib.ptr(t) for t in rays],
                torch.cuda.current_stream(dev).cuda_stream), "nsb_sample_pixel_batch")
            return rays

        if grad:
            ow, du, dn, om, dm, mn = PoseRaysFn.apply(c2ws, run, dict(
                H=self.H, W=self.W, Ks=self._Ks, c2ws=poses, convention=self.convention, pixel_center=True, as_ndc=self.as_ndc,
                near_plane=self.near_plane, pixels_xy=px, fids=fids))
        else:
            ow, du, dn, om, dm, mn = run()
        self._global_step += 1
        batch = {"rgb": rgb, "rays_o_world": ow, "rays_d_world_unit": du, "rays_d_world_norm": dn, "rays_o_marching": om,
                 "rays_d_marching_unit": dm, "rays_d_marching_norm": mn}                     # samplers.py:193-201
        if with_pixels:
            batch["pixels_xy"], batch["frame_ids"] = px, fids
        return batch

    def __iter__(self) -> Iterator[Dict[str, torch.Tensor]]:
        while True:
            yield self.next_batch()
