"""The vanilla train step (train/trainer.py:876-1013 + :717-725) on libnsb.

``VanillaTrainer`` owns what the reference ``Trainer`` owns for the hot path -- encoders, coarse/fine
NeRF, Adam state -- and exposes

* ``_train_step(batch)``: the reference's method contract (dict with an autograd ``loss``; the caller runs
  ``loss.backward()`` and any torch optimizer over ``parameters()``), implemented as ONE library call that
  computes forward and backward together, and
* ``step(batch)``: the fast path -- forward+backward, optional gradient all-reduce, fused Adam and weight
  re-pack as three library calls on the current stream, capturable in a CUDA graph.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .dist import PeerGrads, allreduce_grads, world_info
from .encoders import get_vanilla_nerf_encoders
from .mlps import NeRF

BATCH_KEYS = ("rays_o_marching", "rays_d_marching_unit", "rays_d_marching_norm", "rays_d_world_unit", "rgb")


def mse2psnr(mse: torch.Tensor) -> torch.Tensor:                       # trainer.py:77-78
    return -10.0 * torch.log10(mse.clamp_min(1e-10))


class _FusedStepFn(torch.autograd.Function):
    """loss = mse(comp_c)+mse(comp_f); forward already ran the backward kernels, so ``backward`` only scales.  The ray tensors
    (rays_o_marching, rays_d_marching_unit, rays_d_world_unit) are explicit inputs: when one requires grad the step also
    computes the loss's gradient w.r.t. them (nsb_train_fwd_bwd_ex)."""

    @staticmethod
    def forward(ctx, tr, batch, draws, grad_mode, rays_o, rays_d, viewdirs, *params):
        # gradients go to a buffer of this call's own (never the trainer's shared / peer-visible buffers): a later
        # _train_step(), step() or step_graph() before loss.backward() cannot change what backward() returns
        want = [grad_mode and t.requires_grad for t in (rays_o, rays_d, viewdirs)]
        ray_grads = None
        grads = torch.empty(2 * _lib.N_PARAMS, device=tr.device, dtype=torch.float32)
        if any(want):
            ray_grads = tuple(torch.empty((t.shape[0], 3), device=tr.device, dtype=torch.float32) if w else None
                              for t, w in zip((rays_o, rays_d, viewdirs), want))
            if not any(p.requires_grad for p in params):
                grads = None                                     # frozen field: no weight-gradient kernel runs
        scal, comp_c, comp_f = tr._fwd_bwd(batch, draws, grad_scale=1.0, grads=grads, ray_grads=ray_grads)
        ctx.tr = tr
        ctx.ray_grads = ray_grads
        ctx.ray_meta = [(t.shape, t.dtype) for t in (rays_o, rays_d, viewdirs)]
        ctx.save_for_backward(grads)
        ctx.mark_non_differentiable(comp_c, comp_f)
        return scal[0].clone(), scal[1].clone(), comp_c, comp_f

    @staticmethod
    def backward(ctx, g_loss, g_psnr, g_cc, g_cf):
        tr = ctx.tr
        (grads,) = ctx.saved_tensors
        n = _lib.N_PARAMS
        if grads is None:
            pg = (None,) * (len(ctx.needs_input_grad) - 7)
        else:
            pg = tuple(tr.nerf_c.unflatten(grads[:n] * g_loss)) + tuple(tr.nerf_f.unflatten(grads[n:] * g_loss))
        rg = (None, None, None) if ctx.ray_grads is None else tuple(
            None if g is None else (g * g_loss).reshape(m[0]).to(m[1]) for g, m in zip(ctx.ray_grads, ctx.ray_meta))
        return (None, None, None, None) + rg + pg


class VanillaTrainer:
    def __init__(self, device="cuda", *, rays_per_batch=1024, nc=64, nf=128, near=2.0, far=6.0, white_bkgd=True,
                 raw_noise_std=1.0, infinite_last_bin=True, det_fine=False, lr=5e-4, betas=(0.9, 0.999), eps=1e-8,
                 mode="fp32", seed=0, sigma_bias=None, process_group=None, allreduce="auto", lr_scheduler="none",
                 lr_scheduler_params=None, grad_clip_norm=0.0, sigma_activation="relu"):
        # hard-coded vanilla settings of the reference: trainer.py:277-291, :411-416; train_nerf.py:275,281
        self.device = torch.device(device)
        self.nc, self.nf, self.samp_near, self.samp_far = int(nc), int(nf), float(near), float(far)
        self.white_bkgd, self.raw_noise_std = bool(white_bkgd), float(raw_noise_std)
        self.infinite_last_bin, self.det_fine = bool(infinite_last_bin), bool(det_fine)
        self.sigma_activation = (sigma_activation or "relu").lower()      # vanilla: relu (trainer.py:277-291); softplus is fused too
        if self.sigma_activation not in ("relu", "softplus"):
            raise ValueError(f"unknown sigma_activation {sigma_activation!r}")
        self.rays_per_batch = int(rays_per_batch)
        self.lr, self.betas, self.eps = float(lr), betas, float(eps)
        # make_scheduler (train/trainer.py:81-90): "none"/"constant" or "cosine" = CosineAnnealingLR(T_max, eta_min)
        name = (lr_scheduler or "none").lower()
        if name not in ("none", "constant", "cosine"):
            raise ValueError(f"unknown lr_scheduler {lr_scheduler!r}")
        sp = lr_scheduler_params or {}
        self.lr_T_max = int(sp["T_max"]) if name == "cosine" else 0
        self.lr_eta_min = float(sp.get("eta_min", 0.0)) if name == "cosine" else 0.0
        self.grad_clip_norm = float(grad_clip_norm or 0.0)          # trainer.py:719-721 (0 = off, the reference default)
        self.mode = {"fp32": _lib.MODE_FP32, "bf16": _lib.MODE_BF16}[mode]
        self.seed, self.global_step, self.adam_t = int(seed), 0, 0
        self.pg = process_group
        # init draws come from a forked RNG: neither the caller's CPU generator nor this device's CUDA generator is reseeded
        with torch.random.fork_rng(devices=[self.device] if self.device.type == "cuda" else []):
            torch.manual_seed(seed)
            self.pos_enc, self.dir_enc = get_vanilla_nerf_encoders()
            self.nerf_c = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation=self.sigma_activation, mode=mode)      # trainer.py:326-341
            self.nerf_f = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation=self.sigma_activation, mode=mode)
        if sigma_bias is not None:
            with torch.no_grad():
                self.nerf_c.sigma_out.bias.fill_(sigma_bias); self.nerf_f.sigma_out.bias.fill_(sigma_bias)
        for m in (self.pos_enc, self.dir_enc, self.nerf_c, self.nerf_f):
            m.to(self.device)
        n = _lib.N_PARAMS
        z = lambda: torch.zeros(n, device=self.device, dtype=torch.float32)
        # multi-GPU: "p2p" = gradient buffers in symmetric memory, all-reduce fused into the Adam kernel over peer loads
        # (nsb_adam_allreduce_step); "nccl" = one NCCL sum-allreduce + the plain Adam kernel; "auto" = p2p when the process
        # group spans several CUDA ranks and symmetric memory can be set up, else nccl
        self.peer = None
        world = world_info(process_group)[1]
        if allreduce not in ("auto", "p2p", "nccl"):
            raise ValueError("allreduce must be 'auto', 'p2p' or 'nccl'")
        if world > 1 and self.grad_clip_norm > 0:
            if allreduce == "p2p":
                raise ValueError("grad_clip_norm needs the norm of the reduced gradient before Adam: use allreduce='nccl'")
            allreduce = "nccl"
        if world > 1 and allreduce in ("auto", "p2p") and self.device.type == "cuda":
            try:
                self.peer = PeerGrads(2 * n, self.device, process_group)
            except Exception as exc:                                   # no symmetric memory on this system / torch build
                if allreduce == "p2p":
                    raise
                import warnings
                warnings.warn(f"symmetric-memory gradient buffers unavailable ({exc!r}); using the NCCL all-reduce")
        # the exchange epoch of a step IS its Adam step count t (one counter on every path: step(), step_graph(), resume)
        if self.peer is not None:
            self.grads_all = self.peer.buffer(1)
        else:
            self.grads_all = torch.zeros(2 * n, device=self.device, dtype=torch.float32)   # one buffer -> one all-reduce
        self.grads_c, self.grads_f = self.grads_all[:n], self.grads_all[n:]
        self.m_c, self.v_c, self.m_f, self.v_f = z(), z(), z(), z()
        self._scal8 = torch.zeros(8, device=self.device, dtype=torch.float32)     # [loss, psnr, mse_c, mse_f, |g|^2, spare x3]
        self.scalars = self._scal8[:4]
        self._ws = None
        self._graphs = None
        self._graph_key = None
        self.nerf_c.packed(); self.nerf_f.packed()

    @classmethod
    def step_engine(cls, nerf_c, nerf_f, *, nc, nf, near, far, white_bkgd=True, raw_noise_std=1.0, infinite_last_bin=True,
                    det_fine=False, sigma_activation="relu", seed=0):
        """A trainer shell around EXISTING modules (no optimiser state): what `install(fuse_train_step=True)` puts behind the
        reference's `Trainer._train_step` -- only `_train_step` / `_fwd_bwd` may be used on it."""
        if nerf_c.mode != nerf_f.mode:
            raise ValueError("coarse and fine NeRF must use the same arithmetic mode")
        self = cls.__new__(cls)
        self.device = nerf_c.flat_params().device
        self.nc, self.nf, self.samp_near, self.samp_far = int(nc), int(nf), float(near), float(far)
        self.white_bkgd, self.raw_noise_std = bool(white_bkgd), float(raw_noise_std)
        self.infinite_last_bin, self.det_fine = bool(infinite_last_bin), bool(det_fine)
        self.sigma_activation = (sigma_activation or "relu").lower()
        self.mode, self.seed, self.global_step, self.adam_t = nerf_c.mode, int(seed), 0, 0
        self.nerf_c, self.nerf_f, self.peer, self.pg = nerf_c, nerf_f, None, None
        self._scal8 = torch.zeros(8, device=self.device, dtype=torch.float32)
        self.scalars = self._scal8[:4]
        self.grads_all = self.grads_c = self.grads_f = None            # _FusedStepFn brings its own gradient buffer
        self._ws = self._graphs = self._graph_key = None
        return self

    def current_lr(self, sched_steps=None) -> float:
        """Learning rate after `sched_steps` scheduler steps (default: now) -- closed form of CosineAnnealingLR."""
        t = self.adam_t if sched_steps is None else int(sched_steps)
        if self.lr_T_max <= 0:
            return self.lr
        import math
        return self.lr_eta_min + (self.lr - self.lr_eta_min) * (1.0 + math.cos(math.pi * t / self.lr_T_max)) * 0.5

    # ---- helpers ---------------------------------------------------------------------------------------
    def parameters(self):
        return list(self.nerf_c.parameters()) + list(self.nerf_f.parameters())     # trainer.py:383-386

    def _flags(self):
        return ((_lib.WHITE_BKGD if self.white_bkgd else 0) | (_lib.INFINITE_LAST_BIN if self.infinite_last_bin else 0)
                | (_lib.SIGMA_SOFTPLUS if self.sigma_activation == "softplus" else 0))

    def _workspace(self, B, ray_grads=False):
        need = _lib.lib().nsb_train_workspace_bytes_ex(B, self.nc, self.nf, self.mode, int(ray_grads))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            self._graphs = None                    # captured graphs hold the old workspace address: recapture on next use
        return self._ws, need

    def _fwd_bwd(self, batch, draws=None, grad_scale=1.0, grads=None, ray_grads=None):
        """nsb_train_fwd_bwd: fills `grads` (default: this step's self.grads_c/grads_f) and self.scalars; returns
        (scalars, comp_c, comp_f).  ray_grads = (d_rays_o, d_rays_d, d_viewdirs) [B,3] fp32 outputs, each optional: then
        nsb_train_fwd_bwd_ex, and `grads` may be None (a frozen field)."""
        L = _lib.lib()
        o, d, rn, vd, tgt = (_lib.f32c(batch[k]) for k in BATCH_KEYS)
        B = o.shape[0]
        ws, wsb = self._workspace(B, ray_grads is not None)
        comp_c = torch.empty((B, 3), device=self.device); comp_f = torch.empty((B, 3), device=self.device)
        draws = draws or {}
        g = lambda k: None if draws.get(k) is None else _lib.f32c(draws[k])
        n = _lib.N_PARAMS
        if ray_grads is not None:
            grads_c, grads_f = (None, None) if grads is None else (grads[:n], grads[n:])
        else:
            grads_c, grads_f = (self.grads_c, self.grads_f) if grads is None else (grads[:n], grads[n:])
        args = (_lib.ptr(o), _lib.ptr(d), _lib.ptr(rn.reshape(B)), _lib.ptr(vd), _lib.ptr(tgt),
                _lib.ptr(self.nerf_c.packed(for_inference=False)), _lib.ptr(self.nerf_f.packed(for_inference=False)), _lib.ptr(grads_c),
                _lib.ptr(grads_f), _lib.ptr(self.scalars), _lib.ptr(comp_c), _lib.ptr(comp_f), _lib.ptr(ws), wsb, B, self.nc, self.nf,
                self.samp_near, self.samp_far, self.raw_noise_std, self._flags(), int(self.det_fine), self.mode,
                float(grad_scale), self.seed, self.global_step, _lib.ptr(g("U")), _lib.ptr(g("u_fine")),
                _lib.ptr(g("noise_c")), _lib.ptr(g("noise_f")))
        if ray_grads is None:
            _lib.check(L.nsb_train_fwd_bwd(*args, _lib.stream()), "nsb_train_fwd_bwd")
        else:
            _lib.check(L.nsb_train_fwd_bwd_ex(*args, *[_lib.ptr(t) for t in ray_grads], _lib.stream()), "nsb_train_fwd_bwd_ex")
        return self.scalars, comp_c, comp_f

    # ---- reference-compatible step ---------------------------------------------------------------------
    def _train_step(self, batch, draws=None) -> dict:
        """Same contract as Trainer._train_step (trainer.py:876-1013): ``loss`` carries autograd history to the
        48 parameters, so ``loss.backward(); torch.optim.Adam(...).step()`` works unchanged.

        When ``rays_o_marching``, ``rays_d_marching_unit`` or ``rays_d_world_unit`` requires grad (and grad mode is on), the
        loss also backpropagates into them -- e.g. to poses through ``RandomPixelRaySampler.next_batch(c2ws=...)`` or
        ``get_camera_rays``.  The ray norms and z samples get no gradient.  For world-space rays that loses nothing under a
        rigid pose update (|R d_cam| does not depend on R); for NDC rays the marching norm depends on the pose, so their pose
        gradient is incomplete.  When no NeRF parameter requires grad, only the ray gradients are computed."""
        loss, psnr, comp_c, comp_f = _FusedStepFn.apply(self, batch, draws, torch.is_grad_enabled(), batch["rays_o_marching"],
                                                        batch["rays_d_marching_unit"], batch["rays_d_world_unit"],
                                                        *self.nerf_c.ordered_params(), *self.nerf_f.ordered_params())
        return {"loss": loss, "psnr": psnr.detach(), "comp_f": comp_f.detach(), "comp_c": comp_c.detach()}

    # ---- fast path ---------------------------------------------------------------------------------------
    def step(self, batch, draws=None):
        """forward + backward (+ all-reduce) + Adam + re-pack.  Returns the device scalars tensor
        [loss, psnr, mse_c, mse_f] of this rank's shard (no host sync)."""
        L = _lib.lib()
        n = _lib.N_PARAMS
        epoch = self.adam_t + 1                               # exchange epoch == Adam's t of this step (same as step_graph)
        if self.peer is not None:                             # this step's gradient buffer (double-buffered by epoch parity)
            self.grads_all = self.peer.buffer(epoch)
            self.grads_c, self.grads_f = self.grads_all[:n], self.grads_all[n:]
        self._fwd_bwd(batch, draws, grad_scale=1.0)
        lr = self.current_lr()                                # sched.step() follows opt.step(): t-1 scheduler steps so far
        self.adam_t += 1
        self.global_step += 1
        if self.peer is not None:
            # all-reduce + Adam in one kernel per net: peer loads over NVLink, no NCCL call on the step path
            pr = self.peer
            arr = lambda ts: (C.c_void_p * len(ts))(*[_lib.ptr(t) for t in ts])
            red_mc, red, lsync = pr.two_phase()
            _lib.check(L.nsb_adam_allreduce_step(arr([self.nerf_c.flat_params(), self.nerf_f.flat_params()]), arr([self.m_c, self.m_f]),
                                                 arr([self.v_c, self.v_f]), 2, pr.pointers(epoch), pr.multicast(epoch), red_mc, _lib.ptr(red),
                                                 _lib.ptr(lsync), pr.flag_array, pr.rank, pr.world,
                                                 epoch, n, lr, self.betas[0], self.betas[1], self.eps, self.adam_t,
                                                 1.0 / pr.world, _lib.ptr(self.scalars), _lib.stream()), "nsb_adam_allreduce_step")
            NeRF.repack((self.nerf_c, self.nerf_f))
            return self.scalars
        world = allreduce_grads(self.grads_all, self.pg)     # ONE sum-allreduce of 2 x 595,844 fp32 over NCCL/NVLink
        guard = self.scalars
        if world > 1:                                         # the skip decision must be common: any rank's bad loss skips all
            guard = self.scalars[:1].clone()
            torch.distributed.all_reduce(guard, op=torch.distributed.ReduceOp.SUM, group=self.pg)     # inf/nan propagate
        if self.grad_clip_norm > 0:                           # clip_grad_norm_ over both nets (trainer.py:719-721)
            _lib.check(L.nsb_grad_clip(_lib.ptr(self.grads_all), 2 * n, self.grad_clip_norm, 1.0 / world, _lib.ptr(self._scal8[4:]),
                                       _lib.stream()), "nsb_grad_clip")
        for nerf, g, m, v in ((self.nerf_c, self.grads_c, self.m_c, self.v_c), (self.nerf_f, self.grads_f, self.m_f, self.v_f)):
            flat = nerf.flat_params()
            _lib.check(L.nsb_adam_step(_lib.ptr(flat), _lib.ptr(g), _lib.ptr(m), _lib.ptr(v), _lib.N_PARAMS, lr,
                                       self.betas[0], self.betas[1], self.eps, self.adam_t, 1.0 / world, _lib.ptr(guard), _lib.stream()),
                       "nsb_adam_step")
        NeRF.repack((self.nerf_c, self.nerf_f))
        return self.scalars

    # ---- fast path, CUDA-graph replay ------------------------------------------------------------------------
    def _launch_train_step(self, parity: int):
        """nsb_train_step on the static batch buffers: the whole step with the step count in device memory."""
        L = _lib.lib()
        n = _lib.N_PARAMS
        st = self._static
        B = st["rays_o_marching"].shape[0]
        ws, wsb = self._workspace(B)
        arr = lambda ts: (C.c_void_p * len(ts))(*[_lib.ptr(t) for t in ts])
        if self.peer is not None:
            grads, pg, pf, rank, world = self.peer.buffer(parity), self.peer.pointers(parity), self.peer.flag_array, self.peer.rank, self.peer.world
            mc = self.peer.multicast(parity)
            red_mc, red, lsync = self.peer.two_phase()
        else:
            grads, pg, pf, rank, world, mc = self.grads_all, None, None, 0, 1, None
            red_mc = red = lsync = None
        _lib.check(L.nsb_train_step(
            _lib.ptr(st["rays_o_marching"]), _lib.ptr(st["rays_d_marching_unit"]), _lib.ptr(st["rays_d_marching_norm"].reshape(B)),
            _lib.ptr(st["rays_d_world_unit"]), _lib.ptr(st["rgb"]), arr([self.nerf_c.flat_params(), self.nerf_f.flat_params()]),
            arr([self.m_c, self.m_f]), arr([self.v_c, self.v_f]), arr([self.nerf_c.packed(for_inference=False), self.nerf_f.packed(for_inference=False)]), _lib.ptr(grads),
            _lib.ptr(self._scal8), _lib.ptr(self._static_comp[0]), _lib.ptr(self._static_comp[1]), _lib.ptr(ws), wsb, B, self.nc,
            self.nf, self.samp_near, self.samp_far, self.raw_noise_std, self._flags(), int(self.det_fine), self.mode, self.seed,
            self.lr, self.lr_eta_min, self.lr_T_max, self.betas[0], self.betas[1], self.eps, self.grad_clip_norm,
            _lib.ptr(self._step_dev), pg, mc, red_mc, _lib.ptr(red), _lib.ptr(lsync), pf, rank,
            world, _lib.stream()),
            "nsb_train_step")

    def step_graph(self, batch):
        """`step()` as ONE CUDA-graph replay (train/trainer.py:702-729 without per-step host work).  The batch is copied
        into static device buffers (host tensors: an H2D copy; pinned memory makes it asynchronous); random draws and the
        Adam bias corrections follow a step counter in device memory.  With several GPUs this needs the peer-memory
        gradient exchange (`allreduce='p2p'`): NCCL calls are not part of the captured step.  Returns the device
        scalars tensor [loss, psnr, mse_c, mse_f] (no host sync)."""
        if world_info(self.pg)[1] > 1 and self.peer is None:
            raise RuntimeError("step_graph needs the peer-memory gradient exchange (allreduce='p2p') on several GPUs")
        if self.adam_t != self.global_step:
            raise RuntimeError("step_graph derives Philox streams and Adam's t from one counter: adam_t must equal global_step")
        B = batch["rays_o_marching"].shape[0]
        # everything whose ADDRESS a captured graph bakes in: a re-flattened / moved parameter buffer, re-allocated packed
        # weights or a grown workspace (see _workspace) force a recapture instead of a replay into freed memory
        key = (B, self.nerf_c.storage_key(), self.nerf_f.storage_key(), self.nc, self.nf)
        if self._graphs is None or self._graph_key != key:
            self._static = {k: torch.empty(tuple(batch[k].shape), dtype=torch.float32, device=self.device) for k in BATCH_KEYS}
            self._static_comp = (torch.empty((B, 3), device=self.device), torch.empty((B, 3), device=self.device))
            self._step_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
            for k in BATCH_KEYS:
                self._static[k].copy_(batch[k])
            # eager warm-up of every kernel on the path, into a PRIVATE gradient buffer: the symmetric buffers may still be
            # read by peers finishing the previous step (no state change, no cross-rank traffic)
            self._fwd_bwd(self._static, grads=torch.empty(2 * _lib.N_PARAMS, device=self.device, dtype=torch.float32))
            self._workspace(B)                               # (sized before capture: growing it later invalidates the graphs)
            torch.cuda.synchronize(self.device)
            self._graphs, self._graph_launches = [], 0
            for parity in ((0, 1) if self.peer is not None else (0,)):
                g = torch.cuda.CUDAGraph()
                before = _lib.launch_count()
                with torch.cuda.graph(g):
                    self._launch_train_step(parity)
                self._graph_launches = _lib.launch_count() - before
                self._graphs.append(g)
            self._graph_key = key
            self._step_host = -1
        if self._step_host != self.adam_t:                   # (re)synchronise the device counter with the host's step count
            self._step_dev.fill_(self.adam_t)
            self._step_host = self.adam_t
        for k in BATCH_KEYS:
            self._static[k].copy_(batch[k], non_blocking=True)
        self.adam_t += 1; self.global_step += 1; self._step_host += 1
        self._graphs[self.adam_t & 1 if self.peer is not None else 0].replay()
        self.nerf_c._infer_stale = self.nerf_f._infer_stale = True      # the graph re-packs the training images only
        return self.scalars

    def check_peers(self):
        """Raise if a peer-memory gradient exchange timed out (nsb_peer_status; synchronises the device).  Call it wherever
        the step's scalars are read on the host."""
        if self.peer is None:
            return
        code = C.c_int(0)
        _lib.check(_lib.lib().nsb_peer_status(C.byref(code)), "nsb_peer_status")
        if code.value:
            raise RuntimeError(f"rank {self.peer.rank}: gradient exchange timed out waiting for rank {code.value - 1} "
                               f"(NSB_PEER_TIMEOUT_S); the update of that step was skipped -- replicas may have diverged")

    # ---- checkpoint: the reference's format (trainer.py:596-645) ----------------------------------------------
    def _adam_param_group(self):
        g = torch.optim.Adam([torch.zeros(1)], lr=self.lr, betas=tuple(self.betas), eps=self.eps).state_dict()["param_groups"][0]
        g = dict(g); g["lr"] = self.current_lr(); g["initial_lr"] = self.lr; g["params"] = list(range(48))
        return g

    def state_dict(self):
        """{step, nerf_c, nerf_f, opt, sched} as Trainer.save_checkpoint writes them: ``opt`` is a torch.optim.Adam
        state_dict over list(nerf_c.parameters()) + list(nerf_f.parameters()) (trainer.py:383-386), so checkpoints move
        between the reference trainer and this one in both directions.  Tensors are copies, not live views."""
        state = {}
        if self.adam_t > 0:
            ms = self.nerf_c.unflatten(self.m_c) + self.nerf_f.unflatten(self.m_f)
            vs = self.nerf_c.unflatten(self.v_c) + self.nerf_f.unflatten(self.v_f)
            for i, (m, v) in enumerate(zip(ms, vs)):
                state[i] = {"step": torch.tensor(float(self.adam_t)), "exp_avg": m.clone(), "exp_avg_sq": v.clone()}
        sched = None
        if self.lr_T_max > 0:
            sched = {"T_max": self.lr_T_max, "eta_min": self.lr_eta_min, "base_lrs": [self.lr], "last_epoch": self.adam_t,
                     "_step_count": self.adam_t + 1, "_last_lr": [self.current_lr()]}
        clone = lambda sd: {k: v.detach().clone() for k, v in sd.items()}
        return {"step": self.global_step, "nerf_c": clone(self.nerf_c.state_dict()), "nerf_f": clone(self.nerf_f.state_dict()),
                "opt": {"state": state, "param_groups": [self._adam_param_group()]}, "scaler": None, "sched": sched}

    def load_state_dict(self, sd):
        """Accepts what state_dict() writes, a reference checkpoint (torch Adam ``opt``, possibly None) and this package's
        round-1 format ({"t", "m_c", ...})."""
        self.global_step = int(sd.get("step", 0))
        self.nerf_c.load_state_dict(sd["nerf_c"]); self.nerf_f.load_state_dict(sd["nerf_f"])
        opt = sd.get("opt")
        for buf in (self.m_c, self.v_c, self.m_f, self.v_f):
            buf.zero_()
        if opt is None:
            self.adam_t = 0
        elif "state" in opt:                                   # torch.optim.Adam.state_dict()
            st = opt["state"]
            self.adam_t = int(float(st[0]["step"])) if len(st) else 0
            if len(st) not in (0, 48):
                raise ValueError(f"optimizer state holds {len(st)} parameters, expected 48 (coarse + fine NeRF)")
            ms = self.nerf_c.unflatten(self.m_c) + self.nerf_f.unflatten(self.m_f)
            vs = self.nerf_c.unflatten(self.v_c) + self.nerf_f.unflatten(self.v_f)
            for i in range(len(st)):
                ms[i].copy_(st[i]["exp_avg"]); vs[i].copy_(st[i]["exp_avg_sq"])
        else:                                                  # round-1 format
            self.adam_t = int(opt["t"])
            for k in ("m_c", "v_c", "m_f", "v_f"):
                getattr(self, k).copy_(opt[k])
        if self.peer is not None:
            # the flag blocks may hold epochs beyond the restored step count: zero them between two barriers so no rank
            # sees a stale "peer has arrived" for an epoch that has not happened yet
            torch.cuda.synchronize(self.device)
            torch.distributed.barrier(self.pg)
            self.peer.flags.zero_()
            torch.cuda.synchronize(self.device)
            torch.distributed.barrier(self.pg)
        self._step_host = -1                                   # step_graph re-synchronises the device counter
        self.nerf_c.packed(force=True); self.nerf_f.packed(force=True)
