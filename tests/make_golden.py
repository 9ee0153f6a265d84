"""Generate tests/golden/*.npz by running the UNMODIFIED reference (evan-wes/nerf-sandbox)
on seeded inputs.  Needs a checkout of the reference (NSB_REFERENCE_SRC, else BASELINE.json's reference_path); the
fixtures it writes are committed and are what pins oracle/nerf_oracle.py.

    python tests/make_golden.py            # rewrites tests/golden/

Weights are drawn with numpy's PCG64 (stable across versions) through
oracle.init_params and loaded into the reference NeRF with load_state_dict, so a
fixture only has to carry the seed, not 2.4 MB of weights.  Random draws inside
the reference (torch.rand_like / torch.rand / torch.randn at trainer.py:907,
sampling_utils.py:48, render_utils.py:240) are replaced by explicit tensors stored
in the fixture, so the oracle and the CUDA path can consume identical numbers.
"""
import os
import sys
import types
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from baseline import ref_runner  # noqa: E402
REF_CHECKOUT = ref_runner.reference_checkout()
if not os.path.isdir(os.path.join(REF_CHECKOUT, "nerf_sandbox")):
    sys.exit(f"no reference checkout at {REF_CHECKOUT}: set NSB_REFERENCE_SRC to a checkout of evan-wes/nerf-sandbox")
sys.path.insert(0, REF_CHECKOUT)

# imageio is not installed and is imported at module scope by render_utils.py:20
_shim = types.ModuleType("imageio"); _shim.v2 = types.ModuleType("imageio.v2")
_shim.imread = _shim.imwrite = _shim.mimwrite = lambda *a, **k: None
_shim.v2.imread = _shim.v2.imwrite = lambda *a, **k: None
sys.modules.setdefault("imageio", _shim); sys.modules.setdefault("imageio.v2", _shim.v2)

from nerf_sandbox.source.models.encoders import get_vanilla_nerf_encoders  # noqa: E402
from nerf_sandbox.source.models.mlps import NeRF  # noqa: E402
from nerf_sandbox.source.utils.sampling_utils import sample_pdf  # noqa: E402
from nerf_sandbox.source.utils import render_utils as RU  # noqa: E402
from nerf_sandbox.source.train import trainer as TR  # noqa: E402

from oracle import nerf_oracle as O  # noqa: E402

OUT = os.path.join(HERE, "golden")
os.makedirs(OUT, exist_ok=True)
torch.set_num_threads(8)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
N = lambda t: t.detach().cpu().numpy()


def ref_nerf(seed, sigma_bias=None):
    p = O.init_params(np.random.default_rng(seed), sigma_bias=sigma_bias)
    net = NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu")
    net.load_state_dict({k: T(v) for k, v in p.items()})
    return net, p


class Draws:
    """Replace torch.rand_like / rand / randn by a queue of explicit tensors."""
    def __init__(self, rand_like=(), rand=(), randn=()):
        self.q = dict(rand_like=list(rand_like), rand=list(rand), randn=list(randn))
    def __enter__(self):
        self.orig = (torch.rand_like, torch.rand, torch.randn)
        torch.rand_like = lambda x, *a, **k: T(self.q["rand_like"].pop(0)).reshape(x.shape)
        torch.rand = lambda *s, **k: T(self.q["rand"].pop(0)).reshape(*s)
        torch.randn = lambda s, *a, **k: T(self.q["randn"].pop(0)).reshape(tuple(s))
        return self
    def __exit__(self, *e):
        torch.rand_like, torch.rand, torch.randn = self.orig


def grad_probe(net, idx):
    flat = torch.cat([p.grad.reshape(-1) for p in net.parameters()])
    norms = np.array([float(p.grad.norm()) for p in net.parameters()], dtype=np.float64)
    return N(flat)[idx], norms


def remove_relu_knife_edges(x, p, pos_enc, enc_dir, rel=2e-6):
    """A pre-activation of a ReLU layer whose magnitude is below the fp32 rounding error of its own dot product (|pre| < rel * sum|terms|)
    has no defined sign for an fp32 implementation: the reference, an FFMA GEMM and a tensor-core GEMM may each land on either
    side, and the ReLU mask flips the gradient of everything upstream (the first version of this fixture had one: layer 6,
    point 158, unit 29, pre = 3.6e-7 against sum|terms| = 8.5).  Such points are moved (scaled by 0.97, no random draw, so
    the fixtures generated after this one are unchanged) until none is left; checked in float64 with the fixture's weights."""
    x = x.copy()
    for _ in range(100):
        e = N(pos_enc(T(x))).astype(np.float64)
        h = e
        bad = np.zeros(len(x), dtype=bool)
        for l in range(8):
            W = p[f"mlp.{l}.weight"].astype(np.float64); b = p[f"mlp.{l}.bias"].astype(np.float64)
            if l == 4:
                h = np.concatenate([h, e], -1)
            pre = h @ W.T + b
            scale = np.abs(h) @ np.abs(W).T + np.abs(b)
            bad |= (np.abs(pre) < rel * scale).any(-1)
            h = np.maximum(pre, 0)
        feat = h @ p["feature.weight"].astype(np.float64).T + p["feature.bias"].astype(np.float64)
        hc = np.concatenate([feat, np.broadcast_to(enc_dir.astype(np.float64), (len(x), enc_dir.shape[-1]))], -1)
        Wc = p["color_fc.weight"].astype(np.float64); bc = p["color_fc.bias"].astype(np.float64)
        bad |= (np.abs(hc @ Wc.T + bc) < rel * (np.abs(hc) @ np.abs(Wc).T + np.abs(bc))).any(-1)
        if not bad.any():
            return x
        x[bad] *= np.float32(0.97)
    raise RuntimeError("could not remove the ReLU knife edges")


def main():
    rng = np.random.default_rng(1234)
    pos_enc, dir_enc = get_vanilla_nerf_encoders()

    # ---- encoder (a1)
    x = rng.uniform(-6, 6, size=(96, 3)).astype(np.float32)
    x[0] = 0.0; x[1] = [6.0, -6.0, 4.0311]
    d = rng.standard_normal((96, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=-1, keepdims=True)
    np.savez(os.path.join(OUT, "encoder.npz"), x=x, d=d, enc_pos=N(pos_enc(T(x))), enc_dir=N(dir_enc(T(d))))

    # ---- MLP forward + parameter grads (a2/a3)
    net, p = ref_nerf(7, sigma_bias=0.3)
    xm = rng.uniform(-5, 5, (160, 3)).astype(np.float32)
    ed = N(dir_enc(T(d[:1].repeat(160, 0))))
    xm = remove_relu_knife_edges(xm, p, pos_enc, ed[0])
    ep = N(pos_enc(T(xm)))
    d_out = rng.standard_normal((160, 4)).astype(np.float32)
    out = net(T(ep), T(ed)); out.backward(T(d_out))
    idx = rng.integers(0, O.N_PARAMS, size=4096)
    gs, gn = grad_probe(net, idx)
    np.savez(os.path.join(OUT, "mlp.npz"), seed=7, sigma_bias=0.3, enc_pos=ep, enc_dir=ed, out=N(out),
             d_out=d_out, grad_idx=idx, grad_samples=gs, grad_norms=gn)

    # ---- compositor (a5), author's recipe compare_nerf_repos.py:638-653 + edge rows
    Bc, Nn = 96, 64
    z = np.sort(rng.uniform(2, 6, (Bc, Nn)).astype(np.float32), -1); z[:8] = np.linspace(2, 6, Nn, dtype=np.float32)
    rgb = (1 / (1 + np.exp(-rng.standard_normal((Bc, Nn, 3))))).astype(np.float32)
    sig = np.maximum(0.2 * rng.standard_normal((Bc, Nn)), 0).astype(np.float32)
    sig[8:16] *= 40.0                      # dense rays: acc -> 1, sdt hits the 60 clamp
    sig[16:20] = 0.0                       # empty rays
    sig[20:24] = 5000.0                    # sigma*delta > 60 everywhere
    sig[24, ::2] = -1.0                    # negative sigma (API allows it) -> clamp_min mask
    z[25, 10:20] = z[25, 10]               # repeated samples -> zero deltas
    rn = rng.uniform(1.0, 1.12, (Bc, 1)).astype(np.float32)
    comp_cases = {}
    for tag, white, inf_last, use_rn in [("a", True, True, True), ("b", False, False, True), ("c", True, False, False)]:
        trgb, tsig = T(rgb).requires_grad_(), T(sig).requires_grad_()
        c, w, a, dep = RU.volume_render_rays(trgb, tsig, T(z), T(rn) if use_rn else None, white, 1e-10, inf_last)
        g_c = rng.standard_normal((Bc, 3)).astype(np.float32); g_w = rng.standard_normal((Bc, Nn)).astype(np.float32)
        g_a = rng.standard_normal((Bc, 1)).astype(np.float32); g_d = rng.standard_normal((Bc, 1)).astype(np.float32)
        # (i) only comp grad (the trainer's case), (ii) all four outputs
        gi = torch.autograd.grad((c * T(g_c)).sum(), [trgb, tsig], retain_graph=True)
        gii = torch.autograd.grad((c * T(g_c)).sum() + (w * T(g_w)).sum() + (a * T(g_a)).sum() + (dep * T(g_d)).sum(),
                                  [trgb, tsig])
        comp_cases.update({f"{tag}_comp": N(c), f"{tag}_w": N(w), f"{tag}_acc": N(a), f"{tag}_depth": N(dep),
                           f"{tag}_g_c": g_c, f"{tag}_g_w": g_w, f"{tag}_g_a": g_a, f"{tag}_g_d": g_d,
                           f"{tag}_drgb_i": N(gi[0]), f"{tag}_dsig_i": N(gi[1]),
                           f"{tag}_drgb_ii": N(gii[0]), f"{tag}_dsig_ii": N(gii[1])})
    np.savez(os.path.join(OUT, "compositor.npz"), z=z, rgb=rgb, sigma=sig, ray_norm=rn, **comp_cases)

    # ---- sample_pdf (a8): author's recipe compare_nerf_repos.py:439-447 + variants
    r0 = np.random.default_rng(0)
    edges = np.sort(r0.uniform(0, 1, (8, 64)).astype(np.float32), -1)
    wts = r0.uniform(0, 1, (8, 63)).astype(np.float32)
    pdf = {"edges": edges, "w_edges": wts}
    pdf["out_edges_det64"] = N(sample_pdf(T(edges), T(wts), 64, deterministic=True))
    zc = O.stratified_z(2.0, 6.0, 64, rng.uniform(0, 1, (40, 64)).astype(np.float32))
    w_c = rng.uniform(0, 1, (40, 64)).astype(np.float32) ** 8          # peaky weights
    w_c[0] = 0.0; w_c[1, 30] = 1.0; w_c[1, :30] = 0; w_c[1, 31:] = 0   # flat / single spike
    bins_mid, wb = O.interval_bins(zc, w_c)
    u = rng.uniform(0, 1, (40, 128)).astype(np.float32); u[2, :4] = [0.0, 1.0 - 2 ** -24, 0.5, 1e-7]
    with Draws(rand=[u]):
        pdf["out_mid_rand128"] = N(sample_pdf(T(bins_mid), T(wb), 128, deterministic=False))
    pdf["out_mid_det128"] = N(sample_pdf(T(bins_mid), T(wb), 128, deterministic=True))
    pdf["out_mid_det1"] = N(sample_pdf(T(bins_mid), T(wb), 1, deterministic=True))
    # the CDF the reference built (for the bit-exact index test) and its indices
    wt = (T(wb) + 1e-5).clamp_min(0); cdf = torch.cumsum(wt / wt.sum(-1, keepdim=True), -1)
    cdf = torch.cat([torch.zeros(40, 1), cdf], -1)
    pdf["cdf_mid"] = N(cdf); pdf["inds_mid_rand128"] = N(torch.searchsorted(cdf, T(u), right=True))
    ul = torch.linspace(0, 1, 128).expand(40, -1).contiguous()
    pdf["inds_mid_det128"] = N(torch.searchsorted(cdf, ul, right=True))
    m1_b = rng.uniform(2, 6, (5, 1)).astype(np.float32); m1_w = rng.uniform(0, 1, (5, 1)).astype(np.float32)
    pdf["m1_bins"], pdf["m1_w"] = m1_b, m1_w
    pdf["out_m1_det8"] = N(sample_pdf(T(m1_b), T(m1_w), 8, deterministic=True))
    pdf.update(zc=zc, w_c=w_c, bins_mid=bins_mid, wb=wb, u=u)
    np.savez(os.path.join(OUT, "sample_pdf.npz"), **pdf)

    # ---- stratified sampler + merge (a6, a9): inline code of trainer.py:901-908, :981
    strat = {}
    for i, (near, far, nc) in enumerate([(2.0, 6.0, 64), (0.0, 1.0, 64), (2.0, 6.0, 32), (0.0, 1.0, 128),
                                         (2.0, 6.0, 256), (0.5, 3.25, 7)]):
        U = rng.uniform(0, 1, (12, nc)).astype(np.float32)
        t = torch.linspace(0.0, 1.0, steps=nc, dtype=torch.float32)
        zt = (near * (1.0 - t) + far * t).expand(12, nc).contiguous()
        mids = 0.5 * (zt[:, 1:] + zt[:, :-1])
        lower = torch.cat([zt[:, :1], mids], -1); upper = torch.cat([mids, zt[:, -1:]], -1)
        zj = torch.sort(lower + (upper - lower) * T(U), -1).values
        strat.update({f"near{i}": near, f"far{i}": far, f"nc{i}": nc, f"U{i}": U, f"z{i}": N(zj), f"zlin{i}": N(zt[0])})
    strat["n_cases"] = 6
    zf = pdf["out_mid_rand128"]
    strat["merge_zc"], strat["merge_zf"] = zc, zf
    strat["merge_out"] = N(torch.sort(torch.cat([T(zc), T(zf)], -1), -1).values)
    np.savez(os.path.join(OUT, "sampler.npz"), **strat)

    # ---- nerf_forward_pass (a4): training noise, NDC-like (viewdirs != marching dirs), None variants
    net, p = ref_nerf(11, sigma_bias=0.5)
    rays = O.synthetic_rays(np.random.default_rng(5), 24)
    zz = O.stratified_z(2.0, 6.0, 64, rng.uniform(0, 1, (24, 64)).astype(np.float32))
    noise = rng.standard_normal(24 * 64).astype(np.float32)
    vd = rng.standard_normal((24, 3)).astype(np.float32) * 3.0      # un-normalised on purpose (:219 normalises)
    fp = {"seed": 11, "sigma_bias": 0.5, "z": zz, "noise": noise, "viewdirs": vd, **rays}
    for tag, kw in [("train", dict(ray_norms=T(rays["rays_d_marching_norm"]), viewdirs_world_unit=T(vd),
                                   raw_noise_std=1.0, training=True, infinite_last_bin=True, white_bkgd=True)),
                    ("eval", dict(ray_norms=T(rays["rays_d_marching_norm"]), viewdirs_world_unit=T(vd),
                                  raw_noise_std=0.0, training=False, infinite_last_bin=False, white_bkgd=False)),
                    ("bare", dict(ray_norms=None, viewdirs_world_unit=None, raw_noise_std=0.0, training=False,
                                  infinite_last_bin=True, white_bkgd=True, mlp_chunk=100))]:
        with Draws(randn=[noise]):
            c, w, a, dep = RU.nerf_forward_pass(T(rays["rays_o_marching"]), T(rays["rays_d_marching_unit"]), T(zz),
                                                pos_enc=pos_enc, dir_enc=dir_enc, nerf=net, sigma_activation="relu", **kw)
        fp.update({f"{tag}_comp": N(c), f"{tag}_w": N(w), f"{tag}_acc": N(a), f"{tag}_depth": N(dep)})
    np.savez(os.path.join(OUT, "forward_pass.npz"), **fp)

    # ---- full train step (trainer.py:876-1013) + backward, B=48, 64+128
    B, nc, nf = 48, 64, 128
    net_c, pc = ref_nerf(21, sigma_bias=0.4); net_f, pf = ref_nerf(22, sigma_bias=0.4)
    rays = O.synthetic_rays(np.random.default_rng(9), B)
    U = rng.uniform(0, 1, (B, nc)).astype(np.float32); uf = rng.uniform(0, 1, (B, nf)).astype(np.float32)
    n_c = rng.standard_normal(B * nc).astype(np.float32); n_f = rng.standard_normal(B * (nc + nf)).astype(np.float32)
    ns = SimpleNamespace(use_ndc=False, global_step=1, device=torch.device("cpu"), amp=False, nc=nc, nf=nf,
                         det_fine=False, samp_near=2.0, samp_far=6.0, pos_enc=pos_enc, dir_enc=dir_enc,
                         nerf_c=net_c, nerf_f=net_f, white_bkgd=True, sigma_activation="relu", raw_noise_std=1.0,
                         train_mlp_chunk=0, infinite_last_bin=True)
    with Draws(rand_like=[U], rand=[uf], randn=[n_c, n_f]):
        out = TR.Trainer._train_step(ns, {k: T(v) for k, v in rays.items()})
    out["loss"].backward()
    idx = rng.integers(0, O.N_PARAMS, size=4096)
    gsc, gnc = grad_probe(net_c, idx); gsf, gnf = grad_probe(net_f, idx)
    # one Adam step over both nets, trainer.py:383-386 (lr 5e-4, default betas/eps)
    opt = torch.optim.Adam(list(net_c.parameters()) + list(net_f.parameters()), lr=5e-4)
    opt.step()
    pc1 = N(torch.cat([q.reshape(-1) for q in net_c.parameters()]))[idx]
    pf1 = N(torch.cat([q.reshape(-1) for q in net_f.parameters()]))[idx]
    np.savez(os.path.join(OUT, "train_step.npz"), seed_c=21, seed_f=22, sigma_bias=0.4, B=B, nc=nc, nf=nf,
             U=U, u_fine=uf, noise_c=n_c, noise_f=n_f, loss=float(out["loss"]), psnr=float(out["psnr"]),
             comp_c=N(out["comp_c"]), comp_f=N(out["comp_f"]), grad_idx=idx,
             grad_samples_c=gsc, grad_norms_c=gnc, grad_samples_f=gsf, grad_norms_f=gnf,
             adam_c=pc1, adam_f=pf1, **rays)

    # ---- eval frame tile (render_utils.py:286-424), ragged last chunk, H*W=6*9=54, chunk 20
    H, W = 6, 9
    net_c, _ = ref_nerf(31, sigma_bias=1.0); net_f, _ = ref_nerf(32, sigma_bias=1.0)
    rays = O.synthetic_rays(np.random.default_rng(13), H * W)
    ev = {"seed_c": 31, "seed_f": 32, "sigma_bias": 1.0, "H": H, "W": W, **rays}
    for tag, ilb, nfe in [("fine", False, 128), ("fine_inf", True, 128), ("coarse_only", False, 0)]:
        r = RU.render_image_chunked(T(rays["rays_o_marching"]), T(rays["rays_d_marching_unit"]),
                                    T(rays["rays_d_marching_norm"]), H, W, 2.0, 6.0, pos_enc, dir_enc, net_c, net_f,
                                    64, nfe, True, torch.device("cpu"), eval_chunk=20, perturb=False,
                                    sigma_activation="relu", viewdirs_world_unit=T(rays["rays_d_world_unit"]),
                                    infinite_last_bin=ilb)
        ev.update({f"{tag}_rgb": N(r["rgb"]), f"{tag}_acc": N(r["acc"]), f"{tag}_depth": N(r["depth"])})
    np.savez(os.path.join(OUT, "eval_tile.npz"), **ev)
    tot = sum(os.path.getsize(os.path.join(OUT, f)) for f in os.listdir(OUT))
    print("golden written:", sorted(os.listdir(OUT)), f"{tot/1e6:.2f} MB")


if __name__ == "__main__":
    main()
