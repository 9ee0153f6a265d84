"""Positional encoder with the reference's module interface (models/encoders.py:6-123), computed by the
``nsb_encode`` CUDA kernel.  The fused ray path (render.nerf_forward_pass) never materialises this
output; the module exists so that code written against the reference keeps working."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib


class _EncodeFn(torch.autograd.Function):
    """gamma(x) with its backward (nsb_encode_bwd); used only when x requires grad."""

    @staticmethod
    def forward(ctx, x, D, L, include_input, out_dim):
        xf = _lib.f32c(x).reshape(-1, D)
        out = torch.empty((xf.shape[0], out_dim), device=x.device, dtype=torch.float32)
        _lib.check(_lib.lib().nsb_encode(_lib.ptr(xf), _lib.ptr(out), xf.shape[0], D, L, int(include_input), _lib.stream()),
                   "nsb_encode")
        ctx.save_for_backward(xf)
        ctx.cfg = (D, L, include_input, out_dim, x.shape, x.dtype)
        return out.reshape(*x.shape[:-1], out_dim).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        (xf,) = ctx.saved_tensors
        D, L, include_input, out_dim, shape, dtype = ctx.cfg
        gx = torch.empty_like(xf)
        _lib.check(_lib.lib().nsb_encode_bwd(_lib.ptr(xf), _lib.ptr(_lib.f32c(g).reshape(-1, out_dim)), _lib.ptr(gx), xf.shape[0], D,
                                             L, int(include_input), _lib.stream()), "nsb_encode_bwd")
        return gx.reshape(shape).to(dtype), None, None, None, None


class PositionalEncoder(nn.Module):
    """gamma(x) = [x (optional), sin(2^k x), cos(2^k x)], k = 0..num_freqs-1 (encoders.py:11-20)."""

    def __init__(self, input_dims: int = 3, num_freqs: int = 10, include_input: bool = True, log_spaced: bool = True,
                 min_freq_log2: int | None = None, max_freq_log2: int | None = None, use_two_pi: bool = False) -> None:
        super().__init__()
        self.input_dims = int(input_dims)
        self.num_freqs = int(num_freqs)
        self.include_input = bool(include_input)
        self.use_two_pi = bool(use_two_pi)
        lo = 0 if min_freq_log2 is None else min_freq_log2
        hi = self.num_freqs - 1 if max_freq_log2 is None else max_freq_log2
        if log_spaced:
            fb = 2.0 ** torch.linspace(float(lo), float(hi), steps=self.num_freqs)          # encoders.py:61
        else:
            fb = torch.linspace(2.0 ** float(lo), 2.0 ** float(hi), steps=self.num_freqs)
        # the kernel hard-codes freq 2^k, k=0..L-1 (the only configuration the vanilla path uses)
        self._kernel_ok = bool(log_spaced and lo == 0 and hi == self.num_freqs - 1 and not self.use_two_pi)
        self.register_buffer("freq_bands", fb, persistent=False)                             # encoders.py:69
        self.out_dim = (self.input_dims if self.include_input else 0) + self.input_dims * self.num_freqs * 2

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not self._kernel_ok:
            raise NotImplementedError("nerf_sandbox_b200 encodes with freq_bands = 2^k, k=0..L-1, no 2*pi (vanilla path)")
        if x.shape[-1] != self.input_dims:
            raise RuntimeError(f"expected last dim {self.input_dims}, got {tuple(x.shape)}")
        if torch.is_grad_enabled() and x.requires_grad:
            return _EncodeFn.apply(x, self.input_dims, self.num_freqs, self.include_input, self.out_dim)
        xf = _lib.f32c(x).reshape(-1, self.input_dims)
        out = torch.empty((xf.shape[0], self.out_dim), device=x.device, dtype=torch.float32)
        _lib.check(_lib.lib().nsb_encode(_lib.ptr(xf), _lib.ptr(out), xf.shape[0], self.input_dims, self.num_freqs,
                                         int(self.include_input), _lib.stream()), "nsb_encode")
        return out.reshape(*x.shape[:-1], self.out_dim).to(x.dtype)


def get_vanilla_nerf_encoders():
    """(pos, dir) encoders with the NeRF defaults Lx=10 -> 63, Ld=4 -> 27 (encoders.py:108-123)."""
    return (PositionalEncoder(input_dims=3, num_freqs=10, include_input=True, log_spaced=True, use_two_pi=False),
            PositionalEncoder(input_dims=3, num_freqs=4, include_input=True, log_spaced=True, use_two_pi=False))
