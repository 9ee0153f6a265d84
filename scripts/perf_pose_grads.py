"""Cost of pose gradients, and a BARF-style joint refinement of field and poses on the fused path.

    python scripts/perf_pose_grads.py [out.json]        (default: profiles/r4_pose_grads.json)

(a) nsb_camera_rays_bwd kernel time (torch.profiler, both launches, mean of 50 calls) at 1,024 and 8,192 rays drawn from 8
    frames, and on a full 800 x 800 grid of one frame (640,000 rays), with upstream gradients on all six outputs (56 B per ray).
(b) VanillaTrainer._train_step + loss.backward() at 1,024 and 8,192 rays (64 + 128 samples) in both modes: parameter gradients
    only, parameters + ray gradients, and ray gradients of a frozen field.  CUDA events, median of 10 calls after 3 warm-ups.
(c) BARF-style run: 8 views (64 x 64) of the analytic scene of tests/test_gpu_fullsize.py with poses perturbed by 3 deg and
    10 cm; a bf16 field trained from scratch with RandomPixelRaySampler(c2ws=refined poses), the fused _train_step and torch
    Adam on the NeRF parameters and a per-frame se(3) increment, against the same training on the perturbed poses held fixed.
    Reports pose errors before / after and the PSNR of two held-out views rendered at their true poses.  No pass bar.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
import nerf_sandbox_b200 as nsb                                      # noqa: E402
from nerf_sandbox_b200 import _lib                                  # noqa: E402
from nerf_sandbox_b200 import rays as R                             # noqa: E402
from oracle import nerf_oracle as O                                 # noqa: E402

DEV = "cuda"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


# ---------------------------------------------------------------------------------------------------- (a)
def rays_bwd_kernel_us(n, F, grid=None, calls=50):
    g = torch.Generator(device=DEV).manual_seed(n)
    H, W = grid if grid else (400, 600)
    Ks = torch.tensor([[500.0, 500.0, W / 2, H / 2]] * F, device=DEV)
    c2ws = torch.eye(4, device=DEV)[:3].reshape(1, 12).repeat(F, 1).contiguous()
    px = None if grid else torch.stack([torch.randint(0, W, (n,), device=DEV, generator=g),
                                        torch.randint(0, H, (n,), device=DEV, generator=g)], -1).float()
    fids = None if grid else torch.randint(0, F, (n,), device=DEV, generator=g, dtype=torch.int32)
    G = [torch.randn((n, k), device=DEV, generator=g) for k in (3, 3, 1, 3, 3, 1)]
    call = lambda: R.camera_rays_backward(H, W, Ks, c2ws, G, convention="opengl", pixel_center=True, as_ndc=False, near_plane=1.0,
                                          pixels_xy=px, fids=fids)
    for _ in range(5):
        call()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            call()
        torch.cuda.synchronize()
    us = {}
    for ev in prof.key_averages():
        if "camera_rays_bwd" in ev.key:
            us[ev.key.split("(")[0].split("::")[-1]] = (getattr(ev, "device_time_total", None) or ev.cuda_time_total) / calls
    return {"rays": n, "frames": F, "kernel_us": us, "total_us": sum(us.values()), "upstream_bytes": 56 * n}


# ---------------------------------------------------------------------------------------------------- (b)
def step_ms(tr, B, how, reps=10, warm=3):
    rng = np.random.default_rng(B)
    r = O.synthetic_rays(rng, B)
    rays_grad = how != "params"
    for q in tr.parameters():
        q.requires_grad_(how != "rays_frozen")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for i in range(warm + reps):
        batch = {k: torch.tensor(v, device=DEV, requires_grad=rays_grad and k in ("rays_o_marching", "rays_d_marching_unit",
                                                                                   "rays_d_world_unit")) for k, v in r.items()}
        for q in tr.parameters():
            q.grad = None
        torch.cuda.synchronize()
        e0.record()
        tr._train_step(batch)["loss"].backward()
        e1.record()
        torch.cuda.synchronize()
        if i >= warm:
            ts.append(e0.elapsed_time(e1))
    for q in tr.parameters():
        q.requires_grad_(True)
    return float(np.median(ts))


# ---------------------------------------------------------------------------------------------------- (c)
def rodrigues(w):
    th = w.norm() + 1e-12
    k = w / th
    K = torch.zeros(3, 3, device=w.device, dtype=w.dtype)
    K[0, 1], K[0, 2], K[1, 0], K[1, 2], K[2, 0], K[2, 1] = -k[2], k[1], k[2], -k[0], -k[1], k[0]
    return torch.eye(3, device=w.device, dtype=w.dtype) + torch.sin(th) * K + (1 - torch.cos(th)) * (K @ K)


def look_at(eye):
    fwd = -eye / np.linalg.norm(eye)
    right = np.cross(fwd, [0.0, 0.0, 1.0]); right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    c2w = np.eye(4, dtype=np.float32)
    c2w[:3, 0], c2w[:3, 1], c2w[:3, 2], c2w[:3, 3] = right, up, -fwd, eye
    return c2w


class _Frame:
    def __init__(self, image, K, c2w):
        self.image, self.K, self.c2w = image, K, c2w


class _Scene:
    def __init__(self, frames):
        self.frames, self.white_bkgd = frames, True


def view_image(K, c2w, H=64, W=64):
    from test_gpu_fullsize import scene_gt
    with torch.no_grad():
        o, d, nrm = (t.cpu().numpy() for t in nsb.get_camera_rays(H, W, K, c2w, pixel_center=True)[:3])
    return scene_gt(o, d, nrm).reshape(H, W, 3)            # z is scaled by the ray norm, as the sampler's batches are


def held_out_psnr(tr, views, K):
    out = []
    for c2w, img in views:
        with torch.no_grad():
            o, d, nrm = nsb.get_camera_rays(64, 64, K, c2w, pixel_center=True)[:3]
            rgb = nsb.render_rays(o, d, nrm.reshape(-1), d, tr.nerf_c, tr.nerf_f, near=2.0, far=6.0, nc=64, nf=128, white_bkgd=True)[0]
        mse = float(((rgb.clamp(0, 1) - torch.tensor(img.reshape(-1, 3), device=DEV)) ** 2).mean())
        out.append(-10 * math.log10(max(mse, 1e-10)))
    return out


def pose_errors(c2ws, true):
    rot, tr = [], []
    for a, b in zip(c2ws, true):
        Rab = a[:3, :3].T @ b[:3, :3]
        rot.append(math.degrees(math.acos(max(-1.0, min(1.0, (np.trace(Rab) - 1) / 2)))))
        tr.append(float(np.linalg.norm(a[:3, 3] - b[:3, 3])))
    return {"rot_deg_mean": float(np.mean(rot)), "rot_deg_max": float(np.max(rot)), "trans_m_mean": float(np.mean(tr)),
            "trans_m_max": float(np.max(tr))}


def barf(steps=3000, refine=True, lr_pose=1e-3):
    rng = np.random.default_rng(7)
    K = np.array([[60.0, 0, 32.0], [0, 60.0, 32.0], [0, 0, 1]], np.float32)
    eyes = []
    for i in range(10):
        az, el = 2 * math.pi * i / 10 + 0.2, 0.35 + 0.25 * math.sin(3 * i)
        eyes.append(4.0 * np.array([math.cos(az) * math.cos(el), math.sin(az) * math.cos(el), math.sin(el)]))
    true = [look_at(e) for e in eyes]
    train_ids, held_ids = list(range(0, 10)), [1, 6]
    train_ids = [i for i in train_ids if i not in held_ids]
    perturbed = []
    for i in train_ids:
        ax = rng.standard_normal(3); ax /= np.linalg.norm(ax)
        tv = rng.standard_normal(3); tv /= np.linalg.norm(tv)
        p = true[i].copy()
        p[:3, :3] = rodrigues(torch.tensor(ax * math.radians(3.0))).numpy() @ true[i][:3, :3]
        p[:3, 3] += 0.10 * tv
        perturbed.append(p)
    scene = _Scene([_Frame(view_image(K, true[i]), K, perturbed[j]) for j, i in enumerate(train_ids)])
    held = [(true[i], view_image(K, true[i])) for i in held_ids]
    s = nsb.RandomPixelRaySampler(scene, rays_per_batch=1024, device=DEV, seed=1)
    tr = nsb.VanillaTrainer(DEV, mode="bf16", seed=0, sigma_bias=0.4)
    P0 = torch.tensor(np.stack(perturbed)[:, :3, :4], device=DEV)
    xi = torch.zeros((len(train_ids), 6), device=DEV, requires_grad=refine)
    opt = torch.optim.Adam(tr.parameters(), lr=5e-4)
    opt_pose = torch.optim.Adam([xi], lr=lr_pose) if refine else None
    hist = []
    for it in range(steps):
        c2ws = torch.stack([torch.cat([rodrigues(xi[f, :3]) @ P0[f, :, :3], (P0[f, :, 3] + xi[f, 3:])[:, None]], 1)
                            for f in range(len(train_ids))]) if refine else P0
        batch = s.next_batch(c2ws=c2ws)
        loss = tr._train_step(batch)["loss"]
        opt.zero_grad()
        if opt_pose:
            opt_pose.zero_grad()
        loss.backward()
        opt.step()                                               # (the fused step re-packs changed weights itself)
        if opt_pose:
            opt_pose.step()
        if it % 500 == 0 or it == steps - 1:
            hist.append({"iter": it, "loss": float(loss.detach())})
    with torch.no_grad():
        final = torch.stack([torch.cat([rodrigues(xi[f, :3]) @ P0[f, :, :3], (P0[f, :, 3] + xi[f, 3:])[:, None]], 1)
                             for f in range(len(train_ids))]).cpu().numpy()
    true_t = [true[i] for i in train_ids]
    return {"refine_poses": refine, "steps": steps, "rays_per_step": 1024, "pose_lr": lr_pose if refine else None,
            "pose_error_before": pose_errors(np.stack(perturbed), true_t), "pose_error_after": pose_errors(final, true_t),
            "held_out_psnr_db": held_out_psnr(tr, held, K), "loss_history": hist}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r4_pose_grads.json")
    res = {"card": card(), "camera_rays_bwd": [], "train_step_ms": {}}
    for n, F, grid in ((1024, 8, None), (8192, 8, None), (640000, 1, (800, 800))):
        r = rays_bwd_kernel_us(n, F, grid)
        res["camera_rays_bwd"].append(r)
        print(r, flush=True)
    for mode in ("fp32", "bf16"):
        tr = nsb.VanillaTrainer(DEV, mode=mode, sigma_bias=0.4)
        for B in (1024, 8192):
            r = {how: step_ms(tr, B, how) for how in ("params", "params+rays", "rays_frozen")}
            r["ray_grads_overhead"] = r["params+rays"] / r["params"] - 1.0
            res["train_step_ms"][f"{mode}_{B}"] = r
            print(mode, B, r, flush=True)
        del tr
        torch.cuda.empty_cache()
    res["barf"] = {"joint": barf(refine=True), "fixed_perturbed_poses": barf(refine=False)}
    print(json.dumps(res["barf"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
