"""Render functions with the reference's signatures (utils/render_utils.py:108-424) on libnsb kernels.

``nerf_forward_pass`` recognises this package's ``NeRF`` + vanilla ``PositionalEncoder`` pair and runs
the fused path (points + encodings + MLP in the field kernels, head activations + compositing in one
warp-per-ray kernel); any other ``nerf`` callable goes through the generic composition, which still
composites with the CUDA kernel.  There is no CPU path."""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn.functional as F

from . import _hooks, _lib
from .encoders import PositionalEncoder
from .mlps import NeRF
from .sampling import sample_pdf  # noqa: F401  (re-exported like render_utils.py:24)


# --------------------------------------------------------------------------------------------------
# volume_render_rays -- utils/render_utils.py:108-167
# --------------------------------------------------------------------------------------------------
class _CompositeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rgb, sigma, z, ray_norm, flags, eps):
        L = _lib.lib()
        B, N = z.shape
        rgb_c, sig_c, z_c = _lib.f32c(rgb), _lib.f32c(sigma), _lib.f32c(z)
        rn_c = None if ray_norm is None else _lib.f32c(ray_norm).reshape(B)
        dev = z.device
        comp = torch.empty((B, 3), device=dev, dtype=torch.float32)
        w = torch.empty((B, N), device=dev, dtype=torch.float32)
        acc = torch.empty((B, 1), device=dev, dtype=torch.float32)
        depth = torch.empty((B, 1), device=dev, dtype=torch.float32)
        _lib.check(L.nsb_composite_fwd(_lib.ptr(rgb_c), _lib.ptr(sig_c), _lib.ptr(z_c), _lib.ptr(rn_c), _lib.ptr(comp),
                                       _lib.ptr(w), _lib.ptr(acc), _lib.ptr(depth), B, N, flags, eps, _lib.stream()),
                   "nsb_composite_fwd")
        ctx.save_for_backward(rgb_c, sig_c, z_c, rn_c)
        ctx.flags, ctx.eps = flags, eps
        return comp, w, acc, depth

    @staticmethod
    def backward(ctx, g_comp, g_w, g_acc, g_depth):
        rgb, sigma, z, rn = ctx.saved_tensors
        B, N = z.shape
        d_rgb, d_sig = torch.empty_like(rgb), torch.empty_like(sigma)
        zero3 = g_comp if g_comp is not None else torch.zeros((B, 3), device=z.device)
        _lib.check(_lib.lib().nsb_composite_bwd(
            _lib.ptr(rgb), _lib.ptr(sigma), _lib.ptr(z), _lib.ptr(rn), _lib.ptr(_lib.f32c(zero3)),
            _lib.ptr(_lib.f32c(g_w)), _lib.ptr(None if g_acc is None else _lib.f32c(g_acc).reshape(B)),
            _lib.ptr(None if g_depth is None else _lib.f32c(g_depth).reshape(B)), _lib.ptr(d_rgb), _lib.ptr(d_sig), B, N,
            ctx.flags, ctx.eps, _lib.stream()), "nsb_composite_bwd")
        return d_rgb, d_sig, None, None, None, None


def volume_render_rays(rgb: torch.Tensor, sigma: torch.Tensor, z_depths: torch.Tensor,
                       ray_norm: torch.Tensor | None = None, white_bkgd: bool = False, eps: float = 1e-10,
                       infinite_last_bin: bool = False):
    """Alpha compositing; returns (composite_rgb (B,3), weights (B,N), acc (B,1), depth (B,1))."""
    flags = (_lib.WHITE_BKGD if white_bkgd else 0) | (_lib.INFINITE_LAST_BIN if infinite_last_bin else 0)
    return _CompositeFn.apply(rgb, sigma, z_depths, ray_norm, flags, float(eps))


# --------------------------------------------------------------------------------------------------
# nerf_forward_pass -- utils/render_utils.py:171-283
# --------------------------------------------------------------------------------------------------
def _is_fused_triplet(pos_enc, dir_enc, nerf) -> bool:
    return (isinstance(nerf, NeRF) and nerf._vanilla and isinstance(pos_enc, PositionalEncoder)
            and isinstance(dir_enc, PositionalEncoder) and pos_enc._kernel_ok and dir_enc._kernel_ok
            and (pos_enc.num_freqs, pos_enc.include_input, pos_enc.input_dims) == (10, True, 3)
            and (dir_enc.num_freqs, dir_enc.include_input, dir_enc.input_dims) == (4, True, 3))


class _FusedPassFn(torch.autograd.Function):
    """rays + z -> (comp, weights, acc, depth); differentiable w.r.t. the NeRF parameters and the rays (rays_o, rays_d_unit,
    viewdirs) through all four outputs.  No gradient w.r.t. z or ray_norm."""

    @staticmethod
    def forward(ctx, nerf, grad_mode, rays_o, rays_d, z, rn, viewdirs, flags, noise_std, noise, seed, *params):
        L = _lib.lib()
        B, N = z.shape
        dev = z.device
        o, d = _lib.f32c(rays_o), _lib.f32c(rays_d)
        vd = None if viewdirs is None else _lib.f32c(viewdirs)
        ray_grad = [t is not None and t.requires_grad for t in (rays_o, rays_d, viewdirs)]
        need_param = grad_mode and any(p.requires_grad for p in params)     # (grad mode is off inside forward)
        need_rays = grad_mode and any(ray_grad)
        need_grad = need_param or need_rays
        packed = nerf.packed()
        wsb = L.nsb_field_workspace_bytes(B * N, nerf.mode, int(need_grad))
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev) if need_grad else nerf._ws.get(wsb, dev)
        raw = torch.empty((B * N, 4), device=dev, dtype=torch.float32)
        _lib.check(L.nsb_field_fwd_rays(_lib.ptr(o), _lib.ptr(d), _lib.ptr(z), _lib.ptr(rn), _lib.ptr(vd), _lib.ptr(packed),
                                        _lib.ptr(raw), _lib.ptr(ws), wsb, B, N, nerf.mode, int(need_grad), _lib.stream()),
                   "nsb_field_fwd_rays")
        comp = torch.empty((B, 3), device=dev, dtype=torch.float32)
        w = torch.empty((B, N), device=dev, dtype=torch.float32)
        acc = torch.empty((B, 1), device=dev, dtype=torch.float32)
        depth = torch.empty((B, 1), device=dev, dtype=torch.float32)
        _lib.check(L.nsb_composite_raw_fwd(_lib.ptr(raw), _lib.ptr(noise), noise_std, _lib.ptr(z), _lib.ptr(rn),
                                           _lib.ptr(comp), _lib.ptr(w), _lib.ptr(acc), _lib.ptr(depth), B, N, flags, seed, 0,
                                           _lib.stream()), "nsb_composite_raw_fwd")
        ctx.nerf, ctx.ws, ctx.wsb, ctx.packed = nerf, ws, wsb, packed
        ctx.saved = (raw, z, rn, noise, o, d, vd)
        ctx.cfg = (B, N, flags, noise_std, seed)
        ctx.need_param = need_param
        ctx.ray_meta = [(t.shape, t.dtype) if t is not None else None for t in (rays_o, rays_d, viewdirs)]
        ctx.set_materialize_grads(False)
        return comp, w, acc, depth

    @staticmethod
    def backward(ctx, g_comp, g_w, g_acc, g_depth):
        L = _lib.lib()
        nerf = ctx.nerf
        raw, z, rn, noise, o, d, vd = ctx.saved
        B, N, flags, noise_std, seed = ctx.cfg
        n_params = len(ctx.needs_input_grad) - 11
        want_o, want_d, want_vd = ctx.needs_input_grad[2], ctx.needs_input_grad[3], ctx.needs_input_grad[6]
        if all(g is None for g in (g_comp, g_w, g_acc, g_depth)) or not (ctx.need_param or want_o or want_d or want_vd):
            return (None,) * (11 + n_params)
        d_raw = torch.empty_like(raw)
        g_acc = None if g_acc is None else _lib.f32c(g_acc).reshape(B)
        g_depth = None if g_depth is None else _lib.f32c(g_depth).reshape(B)
        _lib.check(L.nsb_composite_raw_bwd_ex(_lib.ptr(raw), _lib.ptr(noise), noise_std, _lib.ptr(z), _lib.ptr(rn),
                                              _lib.ptr(_lib.f32c(g_comp)), _lib.ptr(_lib.f32c(g_w)), _lib.ptr(g_acc), _lib.ptr(g_depth),
                                              _lib.ptr(d_raw), B, N, flags, seed, 0, _lib.stream()), "nsb_composite_raw_bwd_ex")
        dev = raw.device
        g = torch.zeros(_lib.N_PARAMS, device=dev, dtype=torch.float32) if ctx.need_param else None
        rays = want_o or want_d or want_vd
        d_ep = torch.empty((B * N, 63), device=dev, dtype=torch.float32) if rays else None
        d_ed = torch.empty((B * N, 27), device=dev, dtype=torch.float32) if rays else None
        _lib.check(L.nsb_field_bwd_ex(_lib.ptr(d_raw), _lib.ptr(ctx.packed), _lib.ptr(g), _lib.ptr(d_ep), _lib.ptr(d_ed),
                                      _lib.ptr(ctx.ws), ctx.wsb, B * N, nerf.mode, _lib.stream()), "nsb_field_bwd_ex")
        d_o = d_d = d_vd = None
        if rays:
            d_o = torch.empty((B, 3), device=dev) if want_o else None
            # without explicit viewdirs the view-direction term belongs to rays_d (render_utils.py:218-222)
            d_d = torch.empty((B, 3), device=dev) if want_d else None
            d_vd = torch.empty((B, 3), device=dev) if want_vd else None
            _lib.check(L.nsb_encode_bwd_rays(_lib.ptr(d_ep), _lib.ptr(d_ed), _lib.ptr(o), _lib.ptr(d), _lib.ptr(z), _lib.ptr(rn),
                                             _lib.ptr(vd), _lib.ptr(d_o), _lib.ptr(d_d), _lib.ptr(d_vd), B, N, _lib.stream()),
                       "nsb_encode_bwd_rays")
        shaped = [None if (t is None or m is None) else t.reshape(m[0]).to(m[1]) for t, m in zip((d_o, d_d, d_vd), ctx.ray_meta)]
        pgrads = tuple(nerf.unflatten(g)) if g is not None else (None,) * n_params
        return (None, None, shaped[0], shaped[1], None, None, shaped[2]) + (None,) * 4 + pgrads


def nerf_forward_pass(rays_o: torch.Tensor, rays_d_unit: torch.Tensor, z_vals: torch.Tensor, *, pos_enc, dir_enc, nerf,
                      white_bkgd: bool, ray_norms: torch.Tensor | None = None,
                      viewdirs_world_unit: torch.Tensor | None = None, sigma_activation: str = "relu",
                      raw_noise_std: float = 0.0, training: bool = False, mlp_chunk: int = 0,
                      infinite_last_bin: bool = False, raw_noise: torch.Tensor | None = None, seed: int | None = None
                      ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Stateless NeRF march + composite at fixed z-samples (render_utils.py:171-283).

    ``raw_noise`` (B*N,) / ``seed`` are extra hooks: explicit N(0,1) draws replacing torch.randn at :240, or
    the Philox seed for in-kernel noise.  ``mlp_chunk`` is accepted and ignored (the kernels tile on-chip)."""
    assert rays_o.shape == rays_d_unit.shape and rays_o.shape[-1] == 3, \
        f"bad ray shapes {rays_o.shape} / {rays_d_unit.shape}"
    B, N = z_vals.shape
    if ray_norms is not None:
        assert ray_norms.shape[:1] == (B,), f"ray_norms {ray_norms.shape} must broadcast with batch {B}"
    flags = ((_lib.WHITE_BKGD if white_bkgd else 0) | (_lib.INFINITE_LAST_BIN if infinite_last_bin else 0)
             | (_lib.TRAINING if training else 0))
    act = (sigma_activation or "relu").lower()
    if _is_fused_triplet(pos_enc, dir_enc, nerf) and act in ("relu", "softplus"):
        if act == "softplus":
            flags |= _lib.SIGMA_SOFTPLUS                      # render_utils.py:243-244, fused into the compositor kernels
        z = _lib.f32c(z_vals)
        rn = None if ray_norms is None else _lib.f32c(ray_norms).reshape(B)
        use_noise = training and raw_noise_std > 0.0
        if use_noise and raw_noise is None and _hooks.normal is not None:
            raw_noise = _hooks.normal(B * N, z.device)
        noise = _lib.f32c(raw_noise).reshape(-1) if (use_noise and raw_noise is not None) else None
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if (use_noise and noise is None) else 0
        comp, w, acc, depth = _FusedPassFn.apply(nerf, torch.is_grad_enabled(), rays_o, rays_d_unit, z, rn, viewdirs_world_unit, flags,
                                                 float(raw_noise_std) if use_noise else 0.0, noise, seed, *nerf.ordered_params())
        return comp, w, acc, depth

    # ---- generic composition for foreign encoders / models (render_utils.py:209-276) ----
    rn = None if ray_norms is None else ray_norms.view(B, 1)
    z_metric = z_vals if rn is None else z_vals * rn
    pts = rays_o[:, None, :] + rays_d_unit[:, None, :] * z_metric[..., None]
    vd = F.normalize(viewdirs_world_unit if viewdirs_world_unit is not None else rays_d_unit, dim=-1)
    out = nerf(pos_enc(pts.reshape(-1, 3)), dir_enc(vd[:, None, :].expand_as(pts).reshape(-1, 3)))
    if isinstance(out, dict):
        rgb_flat, sigma_flat = torch.sigmoid(out["rgb"]), out["sigma"].reshape(-1)
    else:
        rgb_flat, sigma_flat = torch.sigmoid(out[..., :3]), out[..., 3].reshape(-1)
    if training and raw_noise_std > 0.0:
        nz = raw_noise.reshape(-1) if raw_noise is not None else torch.randn(sigma_flat.shape, device=sigma_flat.device)
        sigma_flat = sigma_flat + nz.to(sigma_flat.dtype) * float(raw_noise_std)
    sigma_flat = F.softplus(sigma_flat) if sigma_activation == "softplus" else F.relu(sigma_flat)
    return volume_render_rays(rgb_flat.reshape(B, N, 3), sigma_flat.reshape(B, N), z_vals, rn, white_bkgd, 1e-10,
                              infinite_last_bin)


# --------------------------------------------------------------------------------------------------
# render_image_chunked -- utils/render_utils.py:285-424
# --------------------------------------------------------------------------------------------------
_render_ws = {}


def render_rays(rays_o, rays_d_unit, ray_norms, viewdirs, nerf_c, nerf_f, *, near, far, nc, nf, white_bkgd,
                infinite_last_bin=False, out=None, sigma_activation="relu"):
    """One ray tile through nsb_render_rays (coarse linspace -> coarse pass -> deterministic resample ->
    fine pass).  Returns (rgb (B,3), acc (B,), depth (B,)); ``out`` may hold preallocated slices."""
    L = _lib.lib()
    B = rays_o.shape[0]
    dev = rays_o.device
    fine = nerf_f is not None and nf is not None and int(nf) > 0
    if fine and nerf_f.mode != nerf_c.mode:
        raise ValueError("coarse and fine NeRF must use the same arithmetic mode")
    nfi = int(nf) if fine else 0
    wsb = L.nsb_render_workspace_bytes(B, int(nc), nfi, nerf_c.mode)
    key = (dev, nerf_c.mode)
    ws = _render_ws.get(key)
    if ws is None or ws.numel() < wsb:
        ws = _render_ws[key] = torch.empty(wsb, dtype=torch.uint8, device=dev)
    if out is None:
        out = (torch.empty((B, 3), device=dev), torch.empty((B,), device=dev), torch.empty((B,), device=dev))
    rgb, acc, depth = out
    flags = (_lib.WHITE_BKGD if white_bkgd else 0) | (_lib.INFINITE_LAST_BIN if infinite_last_bin else 0)
    act = (sigma_activation or "relu").lower()
    if act not in ("relu", "softplus"):
        raise ValueError(f"unknown sigma_activation {sigma_activation!r}")
    if act == "softplus":
        flags |= _lib.SIGMA_SOFTPLUS
    _lib.check(L.nsb_render_rays(_lib.ptr(rays_o), _lib.ptr(rays_d_unit), _lib.ptr(ray_norms), _lib.ptr(viewdirs),
                                 _lib.ptr(nerf_c.packed()), _lib.ptr(nerf_f.packed()) if fine else None, _lib.ptr(rgb),
                                 _lib.ptr(acc), _lib.ptr(depth), _lib.ptr(ws), wsb, B, int(nc), nfi, float(near), float(far),
                                 flags, nerf_c.mode, _lib.stream()), "nsb_render_rays")
    return rgb, acc, depth


@torch.no_grad()
def render_image_chunked(rays_o: torch.Tensor, rays_d_unit: torch.Tensor, ray_norms: torch.Tensor, H: int, W: int,
                         near: float, far: float, pos_enc, dir_enc, nerf_c, nerf_f, nc_eval: int, nf_eval: int,
                         white_bkgd: bool, device: torch.device, eval_chunk: int = 8192, perturb: bool = False,
                         sigma_activation: str = "relu", *, viewdirs_world_unit: torch.Tensor | None = None,
                         infinite_last_bin: bool = False) -> dict:
    """Render an image by tiling rays into chunks; returns {"rgb": (H,W,3), "acc": (H,W,1), "depth": (H,W,1)}."""
    if perturb:
        raise NotImplementedError("eval rendering is deterministic (every caller in the reference passes perturb=False)")
    if not (_is_fused_triplet(pos_enc, dir_enc, nerf_c) and (sigma_activation or "relu").lower() in ("relu", "softplus")):
        raise NotImplementedError("render_image_chunked needs nerf_sandbox_b200 NeRF/PositionalEncoder modules (relu or softplus sigma)")
    n = H * W
    dev = torch.device(device)
    o = _lib.f32c(rays_o.reshape(n, 3).to(dev)); d = _lib.f32c(rays_d_unit.reshape(n, 3).to(dev))
    rn = _lib.f32c(ray_norms.reshape(n).to(dev))
    vd = None if viewdirs_world_unit is None else _lib.f32c(viewdirs_world_unit.reshape(n, 3).to(dev))
    rgb = torch.empty((n, 3), device=dev, dtype=torch.float32)
    acc = torch.empty((n,), device=dev, dtype=torch.float32)
    depth = torch.empty((n,), device=dev, dtype=torch.float32)
    chunk = int(eval_chunk) if eval_chunk and eval_chunk > 0 else n
    for s in range(0, n, chunk):                                                          # render_utils.py:337
        e = min(n, s + chunk)
        render_rays(o[s:e], d[s:e], rn[s:e], None if vd is None else vd[s:e], nerf_c, nerf_f, near=near, far=far,
                    nc=nc_eval, nf=nf_eval, white_bkgd=white_bkgd, infinite_last_bin=infinite_last_bin,
                    out=(rgb[s:e], acc[s:e], depth[s:e]), sigma_activation=sigma_activation)
    return {"rgb": rgb.reshape(H, W, 3), "acc": acc.reshape(H, W, 1), "depth": depth.reshape(H, W, 1)}
