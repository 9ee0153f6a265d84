#!/usr/bin/env python
"""bench.py -- headline benchmark of the vanilla-NeRF ray-march path (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode fp32|bf16] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one optimisation step of `train_nerf.py --vanilla` (train/trainer.py:702-729): stratified
coarse sampling, coarse pass, sample_pdf + merge, fine pass, loss, backward, Adam -- over one batch of
1024 synthetic Blender-shaped rays per GPU.  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the last of the K timed steps produced (rank 0) as float32 .npy files, so that two
builds run with the same arguments -- hence the same seeded batches, weights and draws -- can be compared array by array.
Repeated runs of one build are not bitwise identical: the backward sums with fp32 atomics, and Adam's early steps
(~lr * sign(g)) amplify that where a gradient is near zero.  Two bf16 runs of the defaults on one B200 (1000 W limit)
differed by about 6e-5 relative in the loss and up to about 6e-3 in single weights of magnitude <= 0.31 (about 1e-3 at
the 99th percentile): profiles/r3_dump_repeatability.json.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RAYS, NC, NF = 1024, 64, 128
H = W = 800
FX = 0.5 * W / np.tan(0.5 * 0.6911112)            # camera_angle_x of the Blender scenes -> 1111.11
FLOP_TRAIN_PER_POINT = 3_489_024                   # SURVEY 8d: fwd 1,186,816 + dgrad 1,115,392 + wgrad 1,186,816
FLOP_FWD_PER_POINT = 1_186_816
POINTS_PER_RAY = NC + (NC + NF)


def blender_rays(rng, n, step):
    """Synthetic Blender-shape batch: one random pose on the r=4.0311 sphere looking at the origin, `n`
    random pixels of an 800x800 pinhole image (precrop to the central 50% for the first 500 steps,
    samplers.py:119-127), targets U(0,1) composited on white.  Keys as trainer.py:880-884."""
    th, ph = rng.uniform(0, 2 * np.pi), rng.uniform(np.deg2rad(-60), np.deg2rad(10))
    c = 4.0311 * np.array([np.cos(ph) * np.cos(th), np.cos(ph) * np.sin(th), -np.sin(ph)])
    fwd = -c / np.linalg.norm(c); right = np.cross(fwd, [0, 0, 1.0]); right /= np.linalg.norm(right); up = np.cross(right, fwd)
    R = np.stack([right, up, -fwd], 1)                                   # OpenGL camera: looks down -z
    lo, hi = (W // 4, 3 * W // 4) if step < 500 else (0, W)
    px = rng.integers(lo, hi, size=(n, 2))
    d_cam = np.stack([(px[:, 0] + 0.5 - W / 2) / FX, -(px[:, 1] + 0.5 - H / 2) / FX, -np.ones(n)], -1)
    d = d_cam @ R.T
    nrm = np.linalg.norm(d, axis=-1, keepdims=True)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    return dict(rays_o_marching=f32(np.broadcast_to(c, (n, 3))), rays_d_marching_unit=f32(d / nrm), rays_d_marching_norm=f32(nrm),
                rays_d_world_unit=f32(d / nrm), rgb=f32(rng.uniform(0, 1, (n, 3))))


def frame_rays(rng):
    th = rng.uniform(0, 2 * np.pi)
    b = blender_rays(np.random.default_rng(1), 1, 1000)
    c = b["rays_o_marching"][0].astype(np.float64)
    fwd = -c / np.linalg.norm(c); right = np.cross(fwd, [0, 0, 1.0]); right /= np.linalg.norm(right); up = np.cross(right, fwd)
    R = np.stack([right, up, -fwd], 1)
    jj, ii = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    d_cam = np.stack([(ii + 0.5 - W / 2) / FX, -(jj + 0.5 - H / 2) / FX, -np.ones_like(ii, dtype=np.float64)], -1).reshape(-1, 3)
    d = d_cam @ R.T
    nrm = np.linalg.norm(d, axis=-1, keepdims=True)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    return f32(np.broadcast_to(c, d.shape)), f32(d / nrm), f32(nrm[:, 0])


def llff_ndc_rays(rng, n):
    """BASELINE configs[3] batch: LLFF fern shape (504x378 = 4032x3024 / 8, f = 3260 / 8), forward-facing NDC marching rays
    (utils/ray_utils.py:92-126: o, d warped to the near plane, z in [0,1], ray_norms = |d_ndc|), world-space view directions."""
    Hh, Ww, f = 378, 504, 407.6
    px = np.stack([rng.integers(0, Ww, n), rng.integers(0, Hh, n)], -1).astype(np.float64) + 0.5
    d = np.stack([(px[:, 0] - Ww / 2) / f, -(px[:, 1] - Hh / 2) / f, -np.ones(n)], -1)        # OpenGL camera, c2w ~ identity + shift
    o = np.broadcast_to(np.array([0.05, -0.03, 0.02]), d.shape)
    near = 1.0
    t = -(near + o[:, 2]) / d[:, 2]
    o = o + t[:, None] * d
    o0 = -f / (Ww / 2) * o[:, 0] / o[:, 2]; o1 = -f / (Hh / 2) * o[:, 1] / o[:, 2]; o2 = 1.0 + 2.0 * near / o[:, 2]
    d0 = -f / (Ww / 2) * (d[:, 0] / d[:, 2] - o[:, 0] / o[:, 2]); d1 = -f / (Hh / 2) * (d[:, 1] / d[:, 2] - o[:, 1] / o[:, 2])
    d2 = -2.0 * near / o[:, 2]
    on, dn = np.stack([o0, o1, o2], -1), np.stack([d0, d1, d2], -1)
    nrm = np.linalg.norm(dn, axis=-1, keepdims=True)
    dw = d / np.linalg.norm(d, axis=-1, keepdims=True)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    return dict(rays_o_marching=f32(on), rays_d_marching_unit=f32(dn / nrm), rays_d_marching_norm=f32(nrm), rays_d_world_unit=f32(dw),
                rgb=f32(rng.uniform(0, 1, (n, 3))))


def dropin_rays_per_s(mode, dev, batches, steps=20, fuse=True):
    """rays/s of the loop body train/trainer.py:702-725 executed by the REFERENCE'S code (oracle/_ref) on this package's
    kernels: install(mode) rebinds its by-name imports, then its unbound Trainer._train_step, autograd backward and
    torch.optim.Adam run unmodified (amp off: the arithmetic mode is the kernels')."""
    import torch
    from baseline import ref_runner
    from nerf_sandbox_b200.install import install, uninstall
    TR, _ = ref_runner.import_reference()
    install(mode=mode, fuse_train_step=fuse)
    try:
        return _dropin_timed(TR, ref_runner, mode, dev, batches, steps)
    finally:
        uninstall()                                   # the CPU baseline leg below times the reference's OWN callables


def _dropin_timed(TR, ref_runner, mode, dev, batches, steps):
    import torch
    with torch.random.fork_rng(devices=[dev]):
        torch.manual_seed(0)
        pos_enc, dir_enc = TR.get_vanilla_nerf_encoders()
        nc_, nf_ = TR.NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu").to(dev), TR.NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu").to(dev)
    with torch.no_grad():
        nc_.sigma_out.bias.fill_(0.3); nf_.sigma_out.bias.fill_(0.3)
    opt = torch.optim.Adam(list(nc_.parameters()) + list(nf_.parameters()), lr=5e-4)
    ns = ref_runner.make_namespace(TR, dev, nc_, nf_, pos_enc.to(dev), dir_enc.to(dev), nc=NC, nf=NF)

    def step(b):
        opt.zero_grad(set_to_none=True)
        out = TR.Trainer._train_step(ns, b)
        out["loss"].backward()
        opt.step()
        return out["loss"]
    for i in range(3):
        step(batches[i % len(batches)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loss = step(batches[i % len(batches)])
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    fused = hasattr(TR.Trainer._train_step, "_nsb_original")
    return {"path": "reference loop body (Trainer._train_step + loss.backward() + torch.optim.Adam) after nerf_sandbox_b200.install(mode); "
                    + ("_train_step = the fused step (install default)" if fused else "the reference's own _train_step body on the rebound callables"),
            "mode": mode,
            "ms_per_step": ms, "train_rays_per_s": RAYS / (ms * 1e-3), "steps": steps, "loss_after": float(loss.detach())}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nme, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def host_threads():
    """Threads the CPU arm uses: every host core, set explicitly (torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_step_fn(rays_per_step):
    """One full optimisation step (fwd+bwd+Adam) of the path on the host cores, on `rays_per_step` rays of the bench
    workload.  Preferred: the reference's OWN code from oracle/_ref (unbound Trainer._train_step + backward + torch Adam,
    fp32, amp off as the reference runs on a CPU device) -> kind "reference".  Only when oracle/_ref is absent: the numpy
    oracle port -> kind "port".  Returns (step callable, kind, threads actually used, description)."""
    threads = host_threads()
    rng = np.random.default_rng(0)
    from baseline import ref_runner
    if ref_runner.available():
        step, info = ref_runner.make_cpu_step(lambda i: blender_rays(rng, rays_per_step, i), nc=NC, nf=NF, threads=threads)
        return step, "reference", info["threads"], (f"reference Trainer._train_step + backward + torch.optim.Adam (oracle/_ref, unmodified), "
                                                    f"torch {info['torch']} CPU fp32, torch threads={info['threads']}")
    from threadpoolctl import threadpool_limits
    from oracle import nerf_oracle as O
    threadpool_limits(limits=threads)
    st = dict(pc=O.init_params(rng, 0.3), pf=O.init_params(rng, 0.3), t=0)
    st["Pc"], st["Pf"] = O.flatten_params(st["pc"]), O.flatten_params(st["pf"])
    st["m"] = [np.zeros_like(st["Pc"]) for _ in range(4)]

    def step():
        B = rays_per_step
        batch = blender_rays(rng, B, st["t"])
        out = O.train_step(st["pc"], st["pf"], batch, near=2.0, far=6.0, nc=NC, nf=NF, U=rng.uniform(0, 1, (B, NC)).astype(np.float32),
                           u_fine=rng.uniform(0, 1, (B, NF)).astype(np.float32), noise_c=rng.standard_normal(B * NC).astype(np.float32),
                           noise_f=rng.standard_normal(B * (NC + NF)).astype(np.float32))
        st["t"] += 1
        st["Pc"], st["m"][0], st["m"][1] = O.adam_step(st["Pc"], O.flatten_params(out["grads_c"]), st["m"][0], st["m"][1], st["t"])
        st["Pf"], st["m"][2], st["m"][3] = O.adam_step(st["Pf"], O.flatten_params(out["grads_f"]), st["m"][2], st["m"][3], st["t"])
        st["pc"], st["pf"] = O.unflatten_params(st["Pc"]), O.unflatten_params(st["Pf"])
        return float(out["loss"])
    return step, "port", threads, f"numpy fp32 oracle port (oracle/_ref absent), BLAS threads={threads}"


def dump_outputs(out_dir, tr):
    """The step's scalars [loss, psnr, mse_c, mse_f] and the parameters it updated in place (2 x 595,844 fp32, 4.8 MB)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"scalars": tr.scalars, "params_coarse": tr.nerf_c.flat_params(), "params_fine": tr.nerf_f.flat_params()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


WORKLOAD = ("vanilla NeRF Blender-shape training 800x800 white bkgd precrop, 1024 rays/step/GPU, 64 coarse + 128 fine, "
            "8x256 MLP x2 fwd+bwd+Adam, random-init (BASELINE configs[1])")


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the step on the host cores -- always the bench workload
    (1024 rays/step), every host thread, rank 0 only (the CPU arm does not depend on the number of GPUs)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step, kind, threads, what = cpu_reference_step_fn(RAYS)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = RAYS * args.steps / dt
    sample = f"{args.steps} full steps (fwd+bwd+Adam) of {RAYS} rays x (64+192) samples after {args.warmup} warm-up: {what}"
    print(json.dumps({
        "impl": "reference", "metric": "train_rays_per_s", "value": v, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rays_per_step_per_gpu": RAYS, "host_threads": threads},
        "cpu_baseline": {"value": v, "unit": "rays/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of each training loop (headline, end to end, repeats, LLFF-NDC, drop-in); the field "
                         "roofline times a fixed 10 launch sets and the CPU baseline a fixed 4 steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("NSB_BENCH_MODE", "bf16"), choices=["fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-frame", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true")
    ap.add_argument("--no-dropin", action="store_true")
    ap.add_argument("--graph", type=int, default=1, help="capture the step in a CUDA graph (N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import nerf_sandbox_b200 as nsb
    from nerf_sandbox_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W_ = max(args.warmup, 3)
    K = args.steps

    tr = nsb.VanillaTrainer(dev, rays_per_batch=RAYS, nc=NC, nf=NF, near=2.0, far=6.0, mode=args.mode, seed=0, sigma_bias=0.3,
                            allreduce=os.environ.get("NSB_ALLREDUCE", "auto"))
    exchange = ("all-reduce fused into the Adam kernel over NVLink peer loads (nsb_adam_allreduce_step)" if tr.peer is not None
                else ("NCCL all-reduce" if world > 1 else "no exchange (single GPU)"))
    rng = np.random.default_rng(1000 + rank)
    pool_n = 8
    host = [{k: torch.from_numpy(v).pin_memory() for k, v in blender_rays(rng, RAYS, s).items()} for s in range(pool_n)]
    devb = [{k: v.to(dev) for k, v in b.items()} for b in host]
    h2d = sum(v.numel() * 4 for v in host[0].values())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms, op=None):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=op or dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing ("value") --------------------------------------------------------------
    clk = ClockSampler(local) if rank == 0 else None      # samples through warm-up + both timed regions (all under load)
    # the step is one CUDA-graph replay (VanillaTrainer.step_graph = nsb_train_step captured once; step count, Philox streams
    # and Adam bias corrections live in device memory) unless NSB_BENCH_GRAPH=0 or the gradient exchange goes through NCCL
    use_graph = os.environ.get("NSB_BENCH_GRAPH", "1") != "0" and (world == 1 or tr.peer is not None)
    do_step = tr.step_graph if use_graph else tr.step
    for i in range(W_):
        do_step(devb[i % pool_n])
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        do_step(devb[i % pool_n])
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if use_graph:
        launches = K * tr._graph_launches                              # kernels of ours inside one replayed graph x steps
    else:
        launches = _lib.launch_count() - l0 + (K if world > 1 and tr.peer is None else 0)      # + one NCCL all-reduce kernel per step
    loss_dev = float(tr.scalars[0])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr)
    # ---- end to end: pinned host batch -> H2D -> step -> D2H loss, every step ---------------------------
    # one pinned host buffer per batch, [o | d | norm | viewdir | rgb] field-major, so a step is ONE H2D copy
    keys = ("rays_o_marching", "rays_d_marching_unit", "rays_d_marching_norm", "rays_d_world_unit", "rgb")
    hpack = [torch.cat([b[k].reshape(-1) for k in keys]).pin_memory() for b in host]
    dpack = torch.empty_like(hpack[0], device=dev)
    offs = np.cumsum([0] + [host[0][k].numel() for k in keys])
    stage = {k: dpack[offs[i]:offs[i + 1]].view(host[0][k].shape) for i, k in enumerate(keys)}
    # every step: one H2D copy of the batch from pinned memory, the step, one D2H copy of [loss, psnr, mse_c, mse_f] into
    # pinned memory.  The host consumes step k's scalars while step k+1 runs (what a training loop that logs every step
    # does): it waits on the copy event of the PREVIOUS step, so the GPU never idles on the read-back; every step's result
    # is read inside the timed region, the last one before the closing event.
    pin = [torch.empty(4, dtype=torch.float32).pin_memory() for _ in range(2)]
    evs = [torch.cuda.Event(), torch.cuda.Event()]
    def e2e_loop(n):
        loss = None
        for i in range(n):
            dpack.copy_(hpack[i % pool_n], non_blocking=True)
            pin[i & 1].copy_(do_step(stage), non_blocking=True)
            evs[i & 1].record()
            if i > 0:
                evs[(i - 1) & 1].synchronize()
                loss = pin[(i - 1) & 1].clone()
        evs[(n - 1) & 1].synchronize()
        return pin[(n - 1) & 1].clone()
    e2e_loop(3)
    barrier()
    e0.record()
    loss_host = e2e_loop(K)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    # spread: four more blocks of K steps, same bracketing (the line's value stays the first block)
    # (after the end-to-end block: sustained load lowers the clocks under the power cap, see the values)
    repeats = [ms_total / K]
    for _ in range(4):
        barrier()
        e0.record()
        for i in range(K):
            do_step(devb[i % pool_n])
        e1.record()
        barrier()
        repeats.append(max_over_ranks(e0.elapsed_time(e1)) / K)

    clocks = clk.stop() if clk else None

    # ---- roofline of the dominant kernel family (encoder+MLP fwd+bwd of the fine pass), timed alone ------
    L = _lib.lib()
    Q = RAYS * (NC + NF)
    b0 = devb[0]
    z = torch.sort(torch.rand((RAYS, NC + NF), device=dev) * 4 + 2, -1).values.contiguous()
    wsb = L.nsb_field_workspace_bytes(Q, tr.mode, 1)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    raw = torch.empty((Q, 4), device=dev); d_raw = torch.randn((Q, 4), device=dev) * 1e-3
    gbuf = torch.zeros(_lib.N_PARAMS, device=dev)
    st = _lib.stream()

    def field():
        _lib.check(L.nsb_field_fwd_rays(_lib.ptr(b0["rays_o_marching"]), _lib.ptr(b0["rays_d_marching_unit"]), _lib.ptr(z),
                                        _lib.ptr(b0["rays_d_marching_norm"].reshape(-1)), _lib.ptr(b0["rays_d_world_unit"]),
                                        _lib.ptr(tr.nerf_f.packed()), _lib.ptr(raw), _lib.ptr(ws), wsb, RAYS, NC + NF, tr.mode, 1, st))
        _lib.check(L.nsb_field_bwd(_lib.ptr(d_raw), _lib.ptr(tr.nerf_f.packed()), _lib.ptr(gbuf), _lib.ptr(ws), wsb, Q, tr.mode, st))
    for _ in range(3):
        field()
    torch.cuda.synchronize()
    reps = 10
    e0.record()
    for _ in range(reps):
        field()
    e1.record(); torch.cuda.synchronize()
    ms_field = e0.elapsed_time(e1) / reps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    ach_tf = Q * FLOP_TRAIN_PER_POINT / (ms_field * 1e-3) / 1e12
    traffic = None
    try:      # DRAM bytes of this launch set from the committed ncu --set full captures (bf16 mode only)
        if args.mode == "bf16":
            traffic = int(json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["field_fwd_bwd_fine_bytes"])
    except Exception:
        pass
    roofline = {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf, "traffic": traffic,
                "kernel": f"field fwd+bwd ({args.mode}) on the fine pass, {Q} points, {ms_field:.3f} ms/launch-set",
                "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst; kernel timed alone)" if peaks else "fallback 1590 (B200_PROFILING.md)"}
    if traffic:      # the same launch set against the HBM roof: the backward half of it is bandwidth-bound (stash round trip)
        hbm_peak = float(peaks.get("hbm_gbs", 6452.5)) if peaks else 6452.5
        roofline["hbm"] = {"achieved": traffic / (ms_field * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                           "frac": traffic / (ms_field * 1e-3) / 1e9 / hbm_peak}

    # ---- secondary metric: 800x800 eval frame (configs[2]), pixel rows split over the N ranks + one all-gather ----------
    extra = {"repeat_ms_per_step": [round(x, 5) for x in repeats]}
    if not args.no_frame:
        from nerf_sandbox_b200.dist import render_image_sharded
        o, d, rn = (torch.from_numpy(a).to(dev) for a in frame_rays(rng))
        chunk = 65536
        full = args.mode == "bf16"
        Hf = H if full else 164                                              # fp32 mode: a bounded band of rows, extrapolated
        nrays = Hf * W
        tim = {}
        def frame():
            return render_image_sharded(o[:nrays], d[:nrays], rn[:nrays], Hf, W, 2.0, 6.0, tr.nerf_c, tr.nerf_f, NC, NF, True, eval_chunk=chunk,
                                        viewdirs_world_unit=d[:nrays], timings=tim)
        frame(); barrier()
        e0.record(); img = frame(); e1.record(); barrier()
        ms_frame = max_over_ranks(e0.elapsed_time(e1)) * (H * W / nrays)
        ms_comp = max_over_ranks(tim["compute"][0].elapsed_time(tim["compute"][1])) * (H * W / nrays)
        # the all-gather as seen by the LAST rank to arrive (min over ranks): on the others the interval is mostly waiting for it
        ms_gather = max_over_ranks(tim["gather"][0].elapsed_time(tim["gather"][1]), dist.ReduceOp.MIN if world > 1 else None)
        ms_comp_min = max_over_ranks(tim["compute"][0].elapsed_time(tim["compute"][1]), dist.ReduceOp.MIN if world > 1 else None) * (H * W / nrays)
        extra.update({"render_800x800_frames_per_s": 1e3 / ms_frame, "render_ms_per_frame": ms_frame, "render_rays_timed": nrays,
                      "render_eval_chunk": chunk, "render_n_gpus": world, "render_ms_compute_max_rank": ms_comp, "render_ms_compute_min_rank": ms_comp_min,
                      "render_ms_allgather": ms_gather if world > 1 else 0.0,
                      "render_mlp_tflops": H * W * POINTS_PER_RAY * FLOP_FWD_PER_POINT / (ms_frame * 1e-3) / 1e12,
                      "render_checksum": float(img["rgb"].double().mean())})
        del o, d, rn, img

    # ---- BASELINE configs[3]: LLFF fern-shape NDC training, ray-sharded 8,192 rays/GPU, same exchange as the headline ------
    if not args.no_cfg4 and args.mode == "bf16":
        B4 = 8192
        rng4 = np.random.default_rng(2000 + rank)
        tr4 = nsb.VanillaTrainer(dev, rays_per_batch=B4, nc=NC, nf=NF, near=0.0, far=1.0, mode=args.mode, seed=0, sigma_bias=2.0,
                                 allreduce=os.environ.get("NSB_ALLREDUCE", "auto"))
        pool4 = [{k: torch.from_numpy(v).to(dev) for k, v in llff_ndc_rays(rng4, B4).items()} for _ in range(4)]
        step4 = tr4.step_graph if use_graph else tr4.step
        for i in range(3):
            step4(pool4[i % 4])
        barrier()
        e0.record()
        for i in range(K):
            step4(pool4[i % 4])
        e1.record()
        barrier()
        ms4 = max_over_ranks(e0.elapsed_time(e1)) / K
        extra["cfg4"] = {"workload": "LLFF fern-shape NDC (504x378, f=407.6, z in [0,1]) training, 8192 rays/step/GPU, 64+128 (BASELINE configs[3])",
                         "rays_per_step_per_gpu": B4, "n_gpus": world, "ms_per_step": ms4, "train_rays_per_s": world * B4 / (ms4 * 1e-3),
                         "steps": K, "loss_after": float(tr4.scalars[0]),
                         "mlp_tflops_per_gpu": B4 * POINTS_PER_RAY * FLOP_TRAIN_PER_POINT / (ms4 * 1e-3) / 1e12}
        tr4.check_peers()
        del tr4, pool4
        torch.cuda.empty_cache()

    # ---- the drop-in seam: the REFERENCE'S OWN Trainer._train_step + backward + torch Adam after install(mode) (N=1) -------
    if rank == 0 and world == 1 and not args.no_dropin:
        try:      # install()'s default (Trainer._train_step = the fused step) and the reference's own _train_step body
            extra["dropin"] = dropin_rays_per_s(args.mode, dev, devb, steps=K)
            extra["dropin_reference_body"] = dropin_rays_per_s(args.mode, dev, devb, steps=K, fuse=False)
        except Exception as exc:                      # oracle/_ref absent, ...: report, do not fail the bench
            extra["dropin"] = {"unavailable": repr(exc)[:200]}

    # ---- CPU baseline (rank 0, N=1 only): the oracle port on the host cores, bounded sample ---------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        stepf, kind, threads, what = cpu_reference_step_fn(RAYS)
        stepf()
        t0 = time.perf_counter(); n = 0
        while n < 4:
            stepf(); n += 1
        dt = time.perf_counter() - t0
        cpu = {"value": RAYS * n / dt, "unit": "rays/s", "cores": threads, "kind": kind,
               "sample": f"{n} full steps (fwd+bwd+Adam) of {RAYS} rays x (64+192) samples after 1 warm-up: {what}"}
        # SURVEY 8d's eval baseline: the reference's render_image_chunked on a tile of the frame, extrapolated to 800x800
        if kind == "reference" and not args.no_frame:
            try:
                from baseline import ref_runner
                tile = 64 * 64
                rr = np.random.default_rng(7)
                render, info = ref_runner.make_cpu_render(lambda: blender_rays(rr, tile, 1000), nc=NC, nf=NF, threads=threads)
                render()
                t0 = time.perf_counter(); render(); dt = time.perf_counter() - t0
                extra["render_cpu_baseline"] = {"rays_per_s": tile / dt, "frames_per_s_extrapolated": tile / dt / (H * W), "cores": info["threads"],
                                                "kind": "reference", "sample": f"render_image_chunked (oracle/_ref, unmodified) on a {tile}-ray tile, "
                                                f"64 + 128 samples, fp32 CPU, second of two calls"}
            except Exception as exc:
                extra["render_cpu_baseline"] = {"unavailable": repr(exc)[:200]}

    if rank == 0:
        ws_gb = L.nsb_train_workspace_bytes(RAYS, NC, NF, tr.mode) / 1e9
        print(json.dumps({
            "metric": "train_rays_per_s", "value": world * RAYS * K / (ms_total * 1e-3), "unit": "rays/s", "n_gpus": world, "steps": K,
            "warmup": W_, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.mode == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "rays_per_step_per_gpu": RAYS, "parallelism": f"ray-sharded dp{world}, {exchange} of 2x595,844 fp32 grads",
                       "mode": args.mode, "step": "one CUDA-graph replay (nsb_train_step)" if use_graph else "eager launches",
                       "l2": f"no flush: per-step working set {ws_gb:.2f} GB exceeds the 126 MB L2"},
            "clocks": clocks,
            "e2e": {"value": world * RAYS * K / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16,
                    "ms_per_step": ms_e2e / K},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "extra": extra,
            "loss_after": loss_dev, "loss_e2e_last": float(loss_host[0]),
        }))
    tr.check_peers()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
