"""Cost of input gradients on the fused NeRF path, and a short iNeRF pose-recovery demo.

    python scripts/perf_input_grads.py [out.json]        (default: profiles/r3_input_grads.json)

1. CUDA-event time of the backward of nerf_forward_pass (field + compositor + ray chain) at 196,608 and 1,572,864 points
   (B = 1024 / 8192 rays x 192 samples) in both arithmetic modes, three ways: parameters only, parameters + rays, rays only
   (frozen field).  Median of 10 timed backward calls per configuration after 3 warm-up calls; every call has its own
   forward (untimed), so the stash it reads is the size a user's backward reads (far above the 126 MB L2).
2. field_dinput_kernel's kernel time from torch.profiler (a separate run of 5 backward calls), and its rate against HBM:
   1280 B read (the dY_0, dY_4, dY_9 tile images) + 360 B written per point.
3. iNeRF: the analytic scene of tests/test_gpu_fullsize.py trained 600 steps in bf16, then a camera pose perturbed by 2 deg
   and 5 cm recovered with Adam on an se(3) increment (rays built in torch from the pose, frozen coarse field, 2048 random
   pixels of a 64 x 64 view per iteration, 300 iterations), against two targets: the analytic scene's image, and the trained
   field's own render at the true pose (which separates the pose gradient from the field's error on that view).
The card's name and power limit are read in the same run."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import nerf_sandbox_b200 as nsb                                      # noqa: E402
from nerf_sandbox_b200 import render                                # noqa: E402
from oracle import nerf_oracle as O                                 # noqa: E402

DEV = "cuda"
HBM_BPS = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def make_inputs(B, N, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    o = torch.randn(B, 3, device=DEV, generator=g)
    o = 4.0 * o / o.norm(dim=-1, keepdim=True)
    d = torch.nn.functional.normalize(-o + 0.35 * torch.randn(B, 3, device=DEV, generator=g), dim=-1)
    z = torch.sort(2.0 + 4.0 * torch.rand(B, N, device=DEV, generator=g), -1).values
    rn = 1.0 + 0.1 * torch.rand(B, device=DEV, generator=g)
    G = [torch.randn(s, device=DEV, generator=g) for s in ((B, 3), (B, N), (B, 1), (B, 1))]
    return o, d, z, rn, G


def fused_loss(net, o, d, z, rn, G):
    pe, de = nsb.get_vanilla_nerf_encoders()
    outs = render.nerf_forward_pass(o, d, z, pos_enc=pe, dir_enc=de, nerf=net, white_bkgd=True, ray_norms=rn, viewdirs_world_unit=d)
    return sum((x * gg).sum() for x, gg in zip(outs, G))


def time_backward(net, B, N, params, rays, reps=10, warm=3):
    o, d, z, rn, G = make_inputs(B, N)
    for q in net.parameters():
        q.requires_grad_(params)
    o.requires_grad_(rays); d.requires_grad_(rays)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for i in range(warm + reps):
        net.zero_grad(set_to_none=True)
        o.grad = d.grad = None
        loss = fused_loss(net, o, d, z, rn, G)
        torch.cuda.synchronize()
        e0.record()
        loss.backward()
        e1.record()
        torch.cuda.synchronize()
        if i >= warm:
            ts.append(e0.elapsed_time(e1))
    for q in net.parameters():
        q.requires_grad_(True)
    return float(np.median(ts))


def dinput_kernel_ms(net, B, N, calls=5):
    o, d, z, rn, G = make_inputs(B, N)
    o.requires_grad_(True); d.requires_grad_(True)
    fused_loss(net, o, d, z, rn, G).backward()                       # warm
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fused_loss(net, o, d, z, rn, G).backward()
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "field_dinput_kernel" in ev.key:
            total_us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total")
            return total_us / 1e3 / ev.count
    return None


# ---------------------------------------------------------------------------------------------------- iNeRF demo
def rodrigues(w):
    th = w.norm() + 1e-12
    k = w / th
    K = torch.zeros(3, 3, device=w.device, dtype=w.dtype)
    K[0, 1], K[0, 2], K[1, 0], K[1, 2], K[2, 0], K[2, 1] = -k[2], k[1], k[2], -k[0], -k[1], k[0]
    return torch.eye(3, device=w.device, dtype=w.dtype) + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


def look_at(eye):
    fwd = -eye / eye.norm()
    right = torch.nn.functional.normalize(torch.linalg.cross(fwd, torch.tensor([0.0, 0.0, 1.0], device=eye.device)), dim=0)
    up = torch.linalg.cross(right, fwd)
    return torch.stack([right, up, -fwd], dim=1)                    # OpenGL camera: x right, y up, looking down -z


def pose_rays(R, t, H=64, W=64, focal=60.0):
    ys, xs = torch.meshgrid(torch.arange(H, device=DEV, dtype=torch.float32), torch.arange(W, device=DEV, dtype=torch.float32),
                            indexing="ij")
    dirs = torch.stack([(xs + 0.5 - W / 2) / focal, -(ys + 0.5 - H / 2) / focal, -torch.ones_like(xs)], -1).reshape(-1, 3)
    d = torch.nn.functional.normalize(dirs @ R.T, dim=-1)
    return t.expand_as(d), d


def inerf_demo(steps_train=600, iters=300, lr=5e-4):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_fullsize import scene_batches
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    pool = [{k: T(v) for k, v in b.items()} for b in scene_batches(32, 1024, 1000)]
    tr = nsb.VanillaTrainer(DEV, mode="bf16", seed=0, sigma_bias=0.4, lr_scheduler="cosine",
                            lr_scheduler_params={"T_max": steps_train, "eta_min": 5e-5})
    for i in range(steps_train):
        tr.step_graph(pool[i % len(pool)])
    torch.cuda.synchronize()
    net = tr.nerf_c
    for q in net.parameters():
        q.requires_grad_(False)
    eye = torch.tensor([2.6, -2.4, 1.9], device=DEV)
    eye = 4.0 * eye / eye.norm()
    R_true = look_at(eye)
    o_t, d_t = pose_rays(R_true, eye)
    from test_gpu_fullsize import scene_gt
    pe, de = nsb.get_vanilla_nerf_encoders()
    Nz = 128
    z_all = torch.linspace(2.0, 6.0, Nz, device=DEV)
    targets = {"analytic_scene": T(scene_gt(o_t.cpu().numpy(), d_t.cpu().numpy(), np.ones(o_t.shape[0], np.float32)))}
    with torch.no_grad():      # the trained field's own render at the true pose: isolates the pose gradient from the field's error
        targets["field_render"] = render.nerf_forward_pass(o_t, d_t, z_all.expand(o_t.shape[0], Nz), pos_enc=pe, dir_enc=de,
                                                           nerf=net, white_bkgd=True)[0]
    out = {"train_steps_bf16": steps_train, "iters": iters, "rays_per_iter": 2048, "samples": Nz, "adam_lr": lr}
    for name, target in targets.items():
        out[name] = recover_pose(net, target, R_true, eye, iters, lr, pe, de, z_all)
    return out


def recover_pose(net, target, R_true, eye, iters, lr, pe, de, z_all):
    Nz = z_all.numel()
    # perturbed start: 2 degrees about a random axis, 5 cm along a random direction
    rng = np.random.default_rng(3)
    ax = torch.tensor(rng.standard_normal(3), dtype=torch.float32, device=DEV); ax = ax / ax.norm()
    tv = torch.tensor(rng.standard_normal(3), dtype=torch.float32, device=DEV); tv = tv / tv.norm()
    R0 = rodrigues(ax * math.radians(2.0)) @ R_true
    t0 = eye + 0.05 * tv
    xi = torch.zeros(6, device=DEV, requires_grad=True)              # se(3) increment: rotation (3), translation (3)
    opt = torch.optim.Adam([xi], lr=lr)

    def errors(R, t):
        cos = ((torch.trace(R.T @ R_true) - 1) / 2).clamp(-1, 1)
        return math.degrees(float(torch.arccos(cos))), float((t - eye).norm())

    g = torch.Generator(device=DEV).manual_seed(0)
    hist = []
    for it in range(iters):
        R = rodrigues(xi[:3]) @ R0
        t = t0 + xi[3:]
        o, d = pose_rays(R, t)
        sel = torch.randperm(o.shape[0], device=DEV, generator=g)[:2048]
        comp = render.nerf_forward_pass(o[sel], d[sel], z_all.expand(sel.numel(), Nz), pos_enc=pe, dir_enc=de, nerf=net,
                                        white_bkgd=True)[0]
        loss = ((comp - target[sel]) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        if it % 50 == 0 or it == iters - 1:
            with torch.no_grad():
                rot_e, tr_e = errors(rodrigues(xi[:3]) @ R0, t0 + xi[3:])
            hist.append({"iter": it, "loss": float(loss.detach()), "rot_err_deg": rot_e, "trans_err_m": tr_e})
    return {"history": hist, "loss_fell": hist[-1]["loss"] < hist[0]["loss"],
            "pose_error_fell": hist[-1]["rot_err_deg"] < hist[0]["rot_err_deg"] and hist[-1]["trans_err_m"] < hist[0]["trans_err_m"]}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_input_grads.json")
    res = {"card": card(), "backward_ms": {}, "field_dinput_kernel": {}}
    for mode in ("fp32", "bf16"):
        net = nsb.NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu", mode=mode).to(DEV)
        for B in (1024, 8192):
            N = 192
            key = f"{mode}_{B * N}"
            r = {way: time_backward(net, B, N, params, rays)
                 for way, params, rays in (("params", True, False), ("params+rays", True, True), ("rays_frozen", False, True))}
            res["backward_ms"][key] = r
            print(key, r, flush=True)
            if mode == "bf16":
                ms = dinput_kernel_ms(net, B, N)
                res["field_dinput_kernel"][key] = {"ms": ms, "bytes": B * N * (1280 + 360),
                                                   "GBps": None if ms is None else B * N * 1640 / ms / 1e6,
                                                   "share_of_7.7TBps": None if ms is None else B * N * 1640 / (ms * 1e-3) / HBM_BPS}
                print(key, res["field_dinput_kernel"][key], flush=True)
        del net
        torch.cuda.empty_cache()
    res["inerf"] = inerf_demo()
    print(json.dumps(res["inerf"]), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
