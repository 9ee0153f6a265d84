"""Parity against the oracle AT THE SIZES bench.py runs (BASELINE.json configs[1], [2], [3]) with explicit draws:

* a 1024-ray, 64+128 train step (configs[1]): loss / composites / every gradient, fp32 mode at the fp32 bar, bf16 mode at
  the bf16 bar;
* an 8,192-ray LLFF-shaped NDC step (configs[3]): the oracle evaluates the batch in eight 1024-ray pieces (loss and
  gradients of a mean-squared error are sums over rays, so the pieces add up exactly -- that keeps the CPU side at
  seconds and a few GB), the GPU runs ONE 8,192-ray step;
* one 65,536-ray eval tile of an 800x800 pose (configs[2], eval_chunk = 65,536): the GPU renders the whole tile in one
  nsb_render_rays call; the oracle renders every 16th ray of it (rays are independent: each checked pixel was produced by
  the full-size launch);
* a TRAINED scene (analytic density/colour field, ground truth by 512-sample quadrature): PSNR on held-out rays of the bf16
  tensor-core mode against the fp32 mode -- same weights rendered in both modes (|dPSNR| <= 0.05 dB, north_star's bar) and
  the two modes trained from the same init on the same batches and Philox draws.
"""
import os

import numpy as np
import pytest
import torch

from oracle import nerf_oracle as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
KEYS = ("rays_o_marching", "rays_d_marching_unit", "rays_d_marching_norm", "rays_d_world_unit", "rgb")


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def N(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope="module")
def nsb():
    import nerf_sandbox_b200 as m
    return m


def _draws(rng, B, nc, nf):
    return dict(U=rng.uniform(0, 1, (B, nc)).astype(np.float32), u_fine=rng.uniform(0, 1, (B, nf)).astype(np.float32),
                noise_c=rng.standard_normal(B * nc).astype(np.float32), noise_f=rng.standard_normal(B * (nc + nf)).astype(np.float32))


def _oracle_step_in_pieces(pc, pf, batch, draws, *, near, far, nc, nf, piece=1024):
    """O.train_step over ray pieces; returns the whole-batch loss, psnr, composites and gradients."""
    B = batch["rgb"].shape[0]
    tot = dict(loss=0.0, mse_f=0.0, comp_c=[], comp_f=[], z_all=[], gc=None, gf=None)
    for s in range(0, B, piece):
        e = min(B, s + piece)
        b = {k: v[s:e] for k, v in batch.items()}
        d = dict(U=draws["U"][s:e], u_fine=draws["u_fine"][s:e], noise_c=draws["noise_c"][s * nc:e * nc],
                 noise_f=draws["noise_f"][s * (nc + nf):e * (nc + nf)])
        r = O.train_step(pc, pf, b, near=near, far=far, nc=nc, nf=nf, **d)
        w = (e - s) / B                                                   # mean over the whole batch = weighted mean of the pieces
        tot["loss"] += w * float(r["loss"])
        tot["mse_f"] += w * 10.0 ** (-float(r["psnr"]) / 10.0)              # psnr = -10 log10(mse_f), trainer.py:77-78
        tot["comp_c"].append(r["comp_c"]); tot["comp_f"].append(r["comp_f"]); tot["z_all"].append(r["z_all"])
        gc, gf = O.flatten_params(r["grads_c"]).astype(np.float64) * w, O.flatten_params(r["grads_f"]).astype(np.float64) * w
        tot["gc"] = gc if tot["gc"] is None else tot["gc"] + gc
        tot["gf"] = gf if tot["gf"] is None else tot["gf"] + gf
    return dict(loss=tot["loss"], psnr=-10 * np.log10(max(tot["mse_f"], 1e-10)), comp_c=np.concatenate(tot["comp_c"]),
                comp_f=np.concatenate(tot["comp_f"]), z_all=np.concatenate(tot["z_all"]), grads_c=tot["gc"], grads_f=tot["gf"])


def _check_step(nsb, batch, draws, *, near, far, nc, nf, sigma_bias, modes):
    ref = None
    for mode in modes:
        tr = nsb.VanillaTrainer(DEV, rays_per_batch=batch["rgb"].shape[0], nc=nc, nf=nf, near=near, far=far, mode=mode, seed=5,
                                sigma_bias=sigma_bias)
        if ref is None:            # both modes start from the same seed -> same weights: one oracle run serves both
            pc = {k: N(v) for k, v in tr.nerf_c.state_dict().items()}; pf = {k: N(v) for k, v in tr.nerf_f.state_dict().items()}
            ref = _oracle_step_in_pieces(pc, pf, batch, draws, near=near, far=far, nc=nc, nf=nf)
        out = tr._train_step({k: T(v) for k, v in batch.items()}, {k: T(v) for k, v in draws.items()})
        out["loss"].backward()
        loss = float(out["loss"].detach())
        gc = N(torch.cat([q.grad.reshape(-1) for q in tr.nerf_c.parameters()])).astype(np.float64)
        gf = N(torch.cat([q.grad.reshape(-1) for q in tr.nerf_f.parameters()])).astype(np.float64)
        rel = lambda a, b: float(np.linalg.norm(a - b) / np.linalg.norm(b))
        if mode == "fp32":
            assert abs(loss - ref["loss"]) <= 1e-4 * ref["loss"], (loss, ref["loss"])
            assert abs(float(out["psnr"]) - ref["psnr"]) <= 1e-3
            np.testing.assert_allclose(N(out["comp_c"]), ref["comp_c"], rtol=1e-4, atol=1e-6)          # north_star: 1e-4 relative
            # The fine composite of the CHAINED step sits behind sample_pdf, whose inverse CDF divides by bin masses as small as
            # 2e-5 (empty bins hold only the two +1e-5 terms): a 1-ulp difference in a coarse weight moves a fine sample by
            # ~1e-4 of a bin, i.e. the chain amplifies fp32 rounding noise to ~1e-4 on a few rays per thousand (the reference
            # against itself in another summation order does the same).  So: the bar on >= 99% of the chained values and a loose
            # cap on the rest, and the strict bar on the fine pass fed with the ORACLE'S sample positions.
            err = np.abs(N(out["comp_f"]) - ref["comp_f"]) - (1e-4 * np.abs(ref["comp_f"]) + 1e-6)
            assert (err <= 0).mean() >= 0.99 and err.max() <= 1e-3, ((err <= 0).mean(), err.max())
            comp_f2, _, _, _ = nsb.nerf_forward_pass(T(batch["rays_o_marching"]), T(batch["rays_d_marching_unit"]), T(ref["z_all"]),
                                                     pos_enc=tr.pos_enc, dir_enc=tr.dir_enc, nerf=tr.nerf_f, white_bkgd=True,
                                                     ray_norms=T(batch["rays_d_marching_norm"]), viewdirs_world_unit=T(batch["rays_d_world_unit"]),
                                                     sigma_activation="relu", raw_noise_std=1.0, training=True, infinite_last_bin=True,
                                                     raw_noise=T(draws["noise_f"]))
            np.testing.assert_allclose(N(comp_f2), ref["comp_f"], rtol=1e-4, atol=1e-6)
            # gradients: fp32 summation-order noise over 10^5..10^6 points (measured against an fp64 oracle run in round 1: 5e-3)
            assert rel(gc, ref["grads_c"]) <= 5e-3 and rel(gf, ref["grads_f"]) <= 2e-2, (rel(gc, ref["grads_c"]), rel(gf, ref["grads_f"]))
        else:
            # bars = ~10x what scripts/tc_precision.py measures at this size (profiles/r2_tc_precision.json: loss 1.5e-4,
            # composite 52.7 dB, gradient cosine 0.99996, |g| ratio 1.0005) -- the training kernels compute in bf16
            assert abs(loss - ref["loss"]) <= 2e-3 * ref["loss"], (loss, ref["loss"])
            assert float(np.abs(N(out["comp_f"]) - ref["comp_f"]).max()) <= 4e-2
            mse = float(np.mean((N(out["comp_f"]) - ref["comp_f"]) ** 2))
            assert -10 * np.log10(max(mse, 1e-12)) >= 48.0                                               # bf16 vs reference render
            cos = lambda a, b: float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)))
            assert cos(gc, ref["grads_c"]) >= 0.9995 and cos(gf, ref["grads_f"]) >= 0.9995, (cos(gc, ref["grads_c"]), cos(gf, ref["grads_f"]))
            # (|g| ratio: 1.0005 on the Blender-shaped batch, 1.012 on the NDC batch whose sigma bias saturates more samples)
            assert abs(np.linalg.norm(gf) / np.linalg.norm(ref["grads_f"]) - 1) <= 3e-2


def test_train_step_1024_rays_matches_oracle(nsb):
    """BASELINE configs[1]: 1024 rays, 64 coarse + 128 fine, both modes."""
    rng = np.random.default_rng(101)
    batch = O.synthetic_rays(rng, 1024)
    _check_step(nsb, batch, _draws(rng, 1024, 64, 128), near=2.0, far=6.0, nc=64, nf=128, sigma_bias=0.4, modes=("fp32", "bf16"))


def llff_ndc_batch(rng, B):
    """BASELINE configs[3] shape: LLFF fern 504x378 (f = 3260/8), NDC marching rays (z in [0,1]), world-space viewdirs."""
    H, W, f = 378, 504, 407.6
    K = np.array([[f, 0, W / 2], [0, f, H / 2], [0, 0, 1]], dtype=np.float32)
    c2w = np.array([[1, 0, 0, 0.05], [0, 1, 0, -0.03], [0, 0, 1, 0.02]], dtype=np.float32)
    px = np.stack([rng.integers(0, W, B), rng.integers(0, H, B)], -1).astype(np.float32)
    r = O.camera_rays(H, W, K, c2w, pixel_center=True, as_ndc=True, near_plane=1.0, pixels_xy=px)
    return dict(rays_o_marching=r[3], rays_d_marching_unit=r[4], rays_d_marching_norm=r[5], rays_d_world_unit=r[1],
                rgb=rng.uniform(0, 1, (B, 3)).astype(np.float32))


def test_train_step_8192_ndc_rays_matches_oracle(nsb):
    """BASELINE configs[3]: 8,192 NDC rays per GPU in one step."""
    rng = np.random.default_rng(102)
    batch = llff_ndc_batch(rng, 8192)
    _check_step(nsb, batch, _draws(rng, 8192, 64, 128), near=0.0, far=1.0, nc=64, nf=128, sigma_bias=2.0, modes=("fp32", "bf16"))


def test_eval_tile_65536_rays_matches_oracle(nsb):
    """BASELINE configs[2]: one eval_chunk = 65,536 tile (rows 359..440) of an 800x800 Blender-shaped pose."""
    H = W = 800
    fx = 0.5 * W / np.tan(0.5 * 0.6911112)
    K = np.array([[fx, 0, W / 2], [0, fx, H / 2], [0, 0, 1]], dtype=np.float32)
    th, ph = 0.9, 0.5
    c = 4.0311 * np.array([np.cos(ph) * np.cos(th), np.cos(ph) * np.sin(th), np.sin(ph)])
    f = -c / np.linalg.norm(c); r = np.cross(f, [0, 0, 1.0]); r /= np.linalg.norm(r); u = np.cross(r, f)
    c2w = np.stack([r, u, -f, c], 1).astype(np.float32)
    rays = O.camera_rays(H, W, K, c2w, pixel_center=True)
    s0 = 359 * W
    sl = slice(s0, s0 + 65536)
    o, d, rn = rays[0][sl], rays[1][sl], rays[2][sl]
    sub = np.arange(0, 65536, 16)
    for mode, tol in (("fp32", None), ("bf16", 5e-3)):
        tr = nsb.VanillaTrainer(DEV, mode=mode, seed=7, sigma_bias=1.0)
        rgb, acc, depth = nsb.render_rays(T(o), T(d), T(rn).reshape(-1), T(d), tr.nerf_c, tr.nerf_f, near=2.0, far=6.0, nc=64, nf=128,
                                          white_bkgd=True)
        if mode == "fp32":
            pc = {k: N(v) for k, v in tr.nerf_c.state_dict().items()}; pf = {k: N(v) for k, v in tr.nerf_f.state_dict().items()}
            ref = O.render_rays_eval(pc, pf, o[sub], d[sub], rn[sub], d[sub], near=2.0, far=6.0, nc=64, nf=128)
            assert 0.05 < float(ref["acc"].mean()) < 0.999                       # a non-degenerate frame (SURVEY 8c caveat)
            np.testing.assert_allclose(N(rgb)[sub], ref["rgb"], rtol=1e-4, atol=2e-6)
            np.testing.assert_allclose(N(acc)[sub], ref["acc"].reshape(-1), rtol=1e-4, atol=2e-6)
            # depth = sum(w z) / (acc + 1e-10): where acc ~ 0 it is a ratio of rounding noise, so the bar applies to acc * depth
            np.testing.assert_allclose(N(depth)[sub] * N(acc)[sub], ref["depth"].reshape(-1) * ref["acc"].reshape(-1), rtol=2e-4, atol=2e-5)
        else:            # the inference kernel computes on fp16 operands: measured 79 dB against the fp32 render
            assert float(np.abs(N(rgb)[sub] - ref["rgb"]).max()) <= tol
            mse = float(np.mean((N(rgb)[sub] - ref["rgb"]) ** 2))
            assert -10 * np.log10(max(mse, 1e-12)) >= 65.0


# ---------------------------------------------------------------------------------------------------- trained scene
def scene_gt(o, d, rn, near=2.0, far=6.0, n=512):
    """Analytic scene: two Gaussian density blobs with position-dependent colour on a white background, integrated with the
    oracle's compositor over n uniform samples."""
    z = np.broadcast_to(np.linspace(near, far, n, dtype=np.float32), (o.shape[0], n))
    pts = o[:, None, :] + d[:, None, :] * (z * rn.reshape(-1, 1))[..., None]
    c1, c2 = np.array([0.5, 0.2, 0.0], np.float32), np.array([-0.6, -0.3, 0.3], np.float32)
    sig = 9.0 * np.exp(-((pts - c1) ** 2).sum(-1) / (2 * 0.55 ** 2)) + 7.0 * np.exp(-((pts - c2) ** 2).sum(-1) / (2 * 0.4 ** 2))
    rgb = 0.5 + 0.45 * np.sin(2.5 * pts + np.array([0.0, 2.0, 4.0], np.float32))
    comp = O.volume_render_rays(rgb.astype(np.float32), sig.astype(np.float32), z.astype(np.float32), rn.reshape(-1, 1), white_bkgd=True)[0]
    return comp.astype(np.float32)


def scene_batches(n_batches, rays, seed0):
    out = []
    for s in range(n_batches):
        r = O.synthetic_rays(np.random.default_rng(seed0 + s), rays)
        r["rgb"] = scene_gt(r["rays_o_marching"], r["rays_d_marching_unit"], r["rays_d_marching_norm"])
        out.append(r)
    return out


def train_and_eval(nsb, steps, n_pool=32, rays=1024, held=4096):
    pool = [{k: T(v) for k, v in b.items()} for b in scene_batches(n_pool, rays, 1000)]
    hb = scene_batches(1, held, 5000)[0]
    args = (T(hb["rays_o_marching"]), T(hb["rays_d_marching_unit"]), T(hb["rays_d_marching_norm"]).reshape(-1), T(hb["rays_d_world_unit"]))
    gt = T(hb["rgb"])
    psnr = lambda rgb: float(-10 * torch.log10(((rgb.clamp(0, 1) - gt) ** 2).mean()))
    res, trainers = {}, {}
    for mode in ("fp32", "bf16"):
        tr = nsb.VanillaTrainer(DEV, mode=mode, seed=0, sigma_bias=0.4, lr_scheduler="cosine", lr_scheduler_params={"T_max": steps, "eta_min": 5e-5})
        for i in range(steps):
            tr.step_graph(pool[i % n_pool])
        torch.cuda.synchronize()
        trainers[mode] = tr
        res[f"trained_{mode}_rendered_{mode}"] = psnr(nsb.render_rays(*args, tr.nerf_c, tr.nerf_f, near=2.0, far=6.0, nc=64, nf=128, white_bkgd=True)[0])
    # the bf16-trained weights rendered by the fp32 kernels (identical inputs, two arithmetic modes)
    pair = []
    for src in (trainers["bf16"].nerf_c, trainers["bf16"].nerf_f):
        m = nsb.NeRF(63, 27, mode="fp32").to(DEV); m.load_state_dict(src.state_dict()); pair.append(m)
    res["trained_bf16_rendered_fp32"] = psnr(nsb.render_rays(*args, pair[0], pair[1], near=2.0, far=6.0, nc=64, nf=128, white_bkgd=True)[0])
    res["steps"] = steps
    return res


def test_trained_scene_psnr_delta_bf16_vs_fp32(nsb):
    steps = int(os.environ.get("NSB_TEST_TRAIN_STEPS", "600"))
    res = train_and_eval(nsb, steps)
    print("trained-scene PSNR (dB):", res)
    assert res["trained_bf16_rendered_bf16"] > 20.0, res                          # the scene is actually learnt
    # north_star's bf16 bar on identical inputs: the same trained weights rendered in the two modes
    assert abs(res["trained_bf16_rendered_bf16"] - res["trained_bf16_rendered_fp32"]) <= 0.05, res
    # and training IN bf16 reaches the quality of training in fp32 (same init, batches and draws).  The two trajectories differ
    # only by arithmetic and diverge chaotically -- each mode also differs from ITSELF run to run (fp32 atomics order): measured
    # end points over six runs, fp32 33.32 .. 33.52 dB (FFMA and tensor-core GEMMs), bf16 33.23 .. 33.45 dB -- so the bar is half
    # a dB either way, not a sign.
    assert abs(res["trained_bf16_rendered_bf16"] - res["trained_fp32_rendered_fp32"]) <= 0.5, res
