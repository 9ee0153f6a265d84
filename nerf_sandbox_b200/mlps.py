"""NeRF MLP with the reference's module interface (models/mlps.py:35-314); forward and backward run in
libnsb (fp32 parity mode or bf16 mode, both on tcgen05).  Parameters live in nn.Linear modules so ``state_dict``
keeps the reference's keys/shapes (SURVEY section 5), but their storage is one flat fp32 buffer in
state_dict order: the kernels, the gradient all-reduce and the fused Adam step all see a single array."""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import _lib


def log_nerf_arch(nerf, pos_enc=None, dir_enc=None, logger=print, name="NeRF"):
    """Same table as models/mlps.py:10-33."""
    epd = getattr(nerf, "enc_pos_dim", None) or getattr(pos_enc, "out_dim", None)
    edd = getattr(nerf, "enc_dir_dim", None) or getattr(dir_enc, "out_dim", None)
    skip = getattr(nerf, "skip_pos", None)
    logger(f"[{name}] enc_pos_dim={epd} enc_dir_dim={edd} hidden_dim={getattr(nerf, 'hidden_dim', None)} "
           f"n_layers={getattr(nerf, 'n_layers', None)} skip_pos={skip}  # 0-based index")
    logger(f"[{name}] Trunk layers (idx  in_features → out_features):")
    for idx, layer in enumerate(nerf.mlp):
        mark = "  <-- SKIP (concat γ(x) into INPUT)" if (skip is not None and idx == skip) else ""
        logger(f"  [{idx:02d}] {layer.in_features} → {layer.out_features}{mark}")
    for attr in ["feature", "sigma_out", "color_fc", "color_out"]:
        head = getattr(nerf, attr, None)
        if head is not None and hasattr(head, "in_features"):
            logger(f"[{name}] {attr}: {head.in_features} → {head.out_features}")


# Arithmetic mode of NeRF modules built without an explicit ``mode=`` -- which is how the reference's Trainer builds them
# (train/trainer.py:326-341 passes no such argument).  install(mode=...) / set_default_mode() / NSB_MODE select it:
# "bf16" = bf16 tensor-core kernels, "fp32" = parity kernels (fp32 activations, split-operand tensor-core GEMMs).
import os as _os
_DEFAULT_MODE = _os.environ.get("NSB_MODE", "fp32").lower()


def set_default_mode(mode: str) -> str:
    """Mode used by ``NeRF(...)`` when the caller passes none; returns the previous default."""
    global _DEFAULT_MODE
    mode = str(mode).lower()
    if mode not in ("fp32", "bf16"):
        raise ValueError(f"mode must be 'fp32' or 'bf16', got {mode!r}")
    prev, _DEFAULT_MODE = _DEFAULT_MODE, mode
    return prev


def get_default_mode() -> str:
    return _DEFAULT_MODE


class _Workspace:
    """Grow-only device scratch owned by PyTorch (the library never allocates)."""

    def __init__(self):
        self.buf = None

    def get(self, nbytes: int, device) -> torch.Tensor:
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        return self.buf


class _FieldEncFn(torch.autograd.Function):
    """NeRF.forward on materialised encodings; grads w.r.t. the parameters and the two encodings."""

    @staticmethod
    def forward(ctx, nerf, grad_mode, enc_pos, enc_dir, *params):
        L = _lib.lib()
        ep, ed = _lib.f32c(enc_pos), _lib.f32c(enc_dir)
        Q = ep.shape[0]
        need_grad = grad_mode and (enc_pos.requires_grad or enc_dir.requires_grad
                                   or any(p.requires_grad for p in params))     # (grad mode is off inside forward)
        packed = nerf.packed()
        wsb = L.nsb_field_workspace_bytes(Q, nerf.mode, int(need_grad))
        ws = (torch.empty(wsb, dtype=torch.uint8, device=ep.device) if need_grad else nerf._ws.get(wsb, ep.device))
        raw = torch.empty((Q, 4), device=ep.device, dtype=torch.float32)
        _lib.check(L.nsb_field_fwd_enc(_lib.ptr(ep), _lib.ptr(ed), _lib.ptr(packed), _lib.ptr(raw), _lib.ptr(ws), wsb, Q,
                                       nerf.mode, int(need_grad), _lib.stream()), "nsb_field_fwd_enc")
        ctx.nerf, ctx.ws, ctx.wsb, ctx.Q, ctx.packed = nerf, ws, wsb, Q, packed
        ctx.enc_dtypes = (enc_pos.dtype, enc_dir.dtype)
        return raw

    @staticmethod
    def backward(ctx, d_raw):
        nerf = ctx.nerf
        dev = d_raw.device
        need_param = any(ctx.needs_input_grad[4:])
        g = torch.zeros(_lib.N_PARAMS, device=dev, dtype=torch.float32) if need_param else None
        d_ep = torch.empty((ctx.Q, nerf.enc_pos_dim), device=dev, dtype=torch.float32) if ctx.needs_input_grad[2] else None
        d_ed = torch.empty((ctx.Q, nerf.enc_dir_dim), device=dev, dtype=torch.float32) if ctx.needs_input_grad[3] else None
        if g is None and d_ep is None and d_ed is None:
            return (None,) * len(ctx.needs_input_grad)
        _lib.check(_lib.lib().nsb_field_bwd_ex(_lib.ptr(_lib.f32c(d_raw)), _lib.ptr(ctx.packed), _lib.ptr(g), _lib.ptr(d_ep),
                                               _lib.ptr(d_ed), _lib.ptr(ctx.ws), ctx.wsb, ctx.Q, nerf.mode, _lib.stream()),
                   "nsb_field_bwd_ex")
        pgrads = tuple(nerf.unflatten(g)) if g is not None else (None,) * (len(ctx.needs_input_grad) - 4)
        return (None, None, None if d_ep is None else d_ep.to(ctx.enc_dtypes[0]),
                None if d_ed is None else d_ed.to(ctx.enc_dtypes[1])) + pgrads


class NeRF(nn.Module):
    """8x256 trunk with the skip concat at the input of layer ``skip_pos``, raw [r,g,b,sigma] output
    (models/mlps.py:41-134, :192-278).  ``mode``: "fp32" (parity) or "bf16"; None = the package default
    (set_default_mode / install(mode=...) / NSB_MODE), so the reference's own constructor call selects it."""

    def __init__(self, enc_pos_dim: int, enc_dir_dim: int, n_layers: int = 8, hidden_dim: int = 256, skip_pos: int = 4,
                 near: float = 2.0, far: float = 6.0, initial_acc_opacity: float | None = None,
                 sigma_activation: str = "softplus", mode: str | None = None) -> None:
        super().__init__()
        self.enc_pos_dim, self.enc_dir_dim = enc_pos_dim, enc_dir_dim
        self.n_layers, self.hidden_dim, self.skip_pos = n_layers, hidden_dim, skip_pos
        layers, in_dim = [], enc_pos_dim
        for idx in range(n_layers):                                               # mlps.py:94-102
            layers.append(nn.Linear(in_dim + (enc_pos_dim if idx == skip_pos else 0), hidden_dim))
            in_dim = hidden_dim
        self.mlp = nn.ModuleList(layers)
        self.feature = nn.Linear(hidden_dim, hidden_dim)                          # :107
        self.sigma_out = nn.Linear(hidden_dim, 1)                                 # :110
        self.color_fc = nn.Linear(hidden_dim + enc_dir_dim, hidden_dim // 2)      # :116
        self.color_out = nn.Linear(hidden_dim // 2, 3)                            # :117
        if initial_acc_opacity is not None:                                       # :120-131
            p = float(max(1e-6, min(0.99, initial_acc_opacity)))
            sigma_star = -math.log(1.0 - p) / float(max(1e-8, far - near))
            bias = math.log(math.expm1(sigma_star)) if (sigma_activation or "softplus").lower() == "softplus" else sigma_star
            with torch.no_grad():
                self.sigma_out.bias.fill_(bias)
                self.color_out.bias.zero_()
                self.color_out.weight.mul_(0.1)
        for m in self.mlp:                                                        # :178-190
            nn.init.kaiming_uniform_(m.weight, nonlinearity="relu"); nn.init.zeros_(m.bias)
        nn.init.kaiming_uniform_(self.feature.weight, nonlinearity="linear"); nn.init.zeros_(self.feature.bias)
        nn.init.kaiming_uniform_(self.color_fc.weight, nonlinearity="relu"); nn.init.zeros_(self.color_fc.bias)
        if mode is None:
            mode = _DEFAULT_MODE
        if mode not in ("fp32", "bf16"):
            raise ValueError(f"mode must be 'fp32' or 'bf16', got {mode!r}")
        self.mode = {"fp32": _lib.MODE_FP32, "bf16": _lib.MODE_BF16}[mode]
        self._vanilla = (enc_pos_dim, enc_dir_dim, n_layers, hidden_dim, skip_pos) == (63, 27, 8, 256, 4)
        self._flat = None
        self._packed = None
        self._packed_version = -1
        self._ws = _Workspace()

    # ---- flat parameter storage ------------------------------------------------------------------
    def ordered_params(self):
        """Parameters in state_dict order (the flat layout of include/nsb.h)."""
        return [p for _, p in self.named_parameters()]

    def flat_params(self) -> torch.Tensor:
        """One contiguous fp32 buffer aliasing every parameter; rebuilt after .to()/.cuda()."""
        ps = self.ordered_params()
        ok = self._flat is not None and self._flat.device == ps[0].device
        if ok:
            off = 0
            for p in ps:
                if p.data.data_ptr() != self._flat.data_ptr() + 4 * off:
                    ok = False
                    break
                off += p.numel()
        if not ok:
            flat = torch.cat([p.data.detach().reshape(-1).to(torch.float32) for p in ps]).contiguous()
            off = 0
            for p in ps:
                p.data = flat[off:off + p.numel()].view(p.shape)
                off += p.numel()
            self._flat, self._packed_version = flat, -1
        return self._flat

    def storage_key(self):
        """Cheap identity of everything a captured CUDA graph bakes in for this net: the flat parameter buffer (first and last
        parameter still alias it -- .to() / load into new tensors breaks that) and the packed-weights buffer."""
        ps = self._param_ends if getattr(self, "_param_ends", None) else None
        if ps is None:
            allp = self.ordered_params()
            ps = self._param_ends = (allp[0], allp[-1], sum(p.numel() for p in allp[:-1]))
        f, pk = self._flat, self._packed
        if f is None or pk is None or ps[0].data.data_ptr() != f.data_ptr() or ps[1].data.data_ptr() != f.data_ptr() + 4 * ps[2]:
            self.flat_params(); self.packed(for_inference=False)
            f, pk = self._flat, self._packed
        return (f.data_ptr(), pk.data_ptr())

    def unflatten(self, flat: torch.Tensor):
        out, off = [], 0
        for p in self.ordered_params():
            out.append(flat[off:off + p.numel()].view(p.shape)); off += p.numel()
        return out

    def packed(self, force: bool = False, for_inference: bool = True) -> torch.Tensor:
        """Kernel-format weights (nsb_pack_weights), refreshed when any parameter changed in place.  A training loop re-packs
        only the training images after each optimiser step (``repack``) and marks the inference-only fp16 images stale; they
        are refreshed here the next time anything but the trainer asks (``for_inference=True``, the default)."""
        if not self._vanilla:
            raise NotImplementedError("libnsb kernels are specialised to NeRF(63,27,8,256,skip_pos=4)")
        flat = self.flat_params()
        if not flat.is_cuda:
            raise RuntimeError("nerf_sandbox_b200 has no CPU path: move the model to a CUDA device")
        L = _lib.lib()
        if self._packed is None or self._packed.device != flat.device:
            self._packed = torch.empty(L.nsb_packed_weights_bytes(), dtype=torch.uint8, device=flat.device)
            self._packed_version = -1
        version = sum(p._version for p in self.ordered_params())     # in-place updates (optimizer, load_state_dict)
        if force or self._packed_version != version or (for_inference and getattr(self, "_infer_stale", False)):
            _lib.check(L.nsb_pack_weights(_lib.ptr(flat), _lib.ptr(self._packed), self.mode, _lib.stream()), "nsb_pack_weights")
            self._packed_version = version
            self._infer_stale = False
        return self._packed

    @staticmethod
    def repack(nets) -> None:
        """Re-pack several nets with one call (nsb_pack_weights_batch: a single launch in tensor-core mode); what the
        trainer does after every optimiser step."""
        import ctypes as C
        nets = list(nets)
        bufs = [n.packed() if n._packed is None else n._packed for n in nets]
        arr = lambda ts: (C.c_void_p * len(ts))(*[_lib.ptr(t) for t in ts])
        _lib.check(_lib.lib().nsb_pack_weights_batch(arr([n.flat_params() for n in nets]), arr(bufs), len(nets),
                                                     nets[0].mode | _lib.PACK_TRAIN_ONLY, _lib.stream()), "nsb_pack_weights_batch")
        for n in nets:
            n._packed_version = sum(p._version for p in n.ordered_params())
            n._infer_stale = True                  # the fp16 inference images are refreshed by the next packed() for inference

    # ---- forward ------------------------------------------------------------------------------------
    def forward(self, enc_pos: torch.Tensor, enc_dir: torch.Tensor) -> torch.Tensor:
        if self._debug_active():
            self._debug_decrement_once_per_forward()
        if enc_pos.shape[-1] != self.enc_pos_dim or enc_dir.shape[-1] != self.enc_dir_dim:
            raise RuntimeError(f"feature dims ({enc_pos.shape[-1]}, {enc_dir.shape[-1]}) do not match "
                               f"({self.enc_pos_dim}, {self.enc_dir_dim})")              # nn.Linear would raise the same
        lead = enc_pos.shape[:-1]
        raw = _FieldEncFn.apply(self, torch.is_grad_enabled(), enc_pos.reshape(-1, self.enc_pos_dim),
                                enc_dir.reshape(-1, self.enc_dir_dim),
                                *self.ordered_params())
        return raw.reshape(*lead, 4).to(enc_pos.dtype)

    # ---- debug helpers kept for Trainer.__init__ (train/trainer.py:367-380; mlps.py:282-314) ----------
    def enable_debug(self, steps: int = 5, logger=print):
        self._debug_steps_remaining, self._debug_logger = int(steps), logger

    def _debug_active(self) -> bool:
        return getattr(self, "_debug_steps_remaining", 0) > 0

    def _debug_log(self, msg: str):
        (getattr(self, "_debug_logger", None) or print)(msg)

    def _debug_decrement_once_per_forward(self):
        if self._debug_active():
            self._debug_steps_remaining -= 1

    def _debug_dump_arch_once(self):
        self._debug_log(f"[NeRF] enc_pos_dim={self.enc_pos_dim} enc_dir_dim={self.enc_dir_dim} "
                        f"hidden_dim={self.hidden_dim} n_layers={self.n_layers} skip_pos={self.skip_pos}")
        for idx, layer in enumerate(self.mlp):
            self._debug_log(f"  mlp[{idx}]: {layer.in_features} → {layer.out_features}"
                            f"{'  <-- SKIP input concat' if idx == self.skip_pos else ''}")
        for n in ("feature", "sigma_out", "color_fc", "color_out"):
            m = getattr(self, n)
            self._debug_log(f"  {n}: {m.in_features} → {m.out_features}")
