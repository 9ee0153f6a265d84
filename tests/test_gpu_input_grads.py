"""Gradients w.r.t. the inputs of the field and of the fused ray path: rays, encodings, and the weights / opacity / depth
outputs of the compositor.

The reference computes all of them by autograd (utils/render_utils.py:108-283, models/mlps.py:192-278,
models/encoders.py:73-106).  This file restates that composition in float64 torch; the CPU tests pin the restatement to the
oracle (itself pinned to the reference goldens), and the GPU tests compare both arithmetic modes against it:
  * fp32 mode: encoding gradients within 1e-4 relative L2 and ray gradients within 1e-3, or within twice the distance of the
    same composition run in float32 on the CPU, whichever is larger (the 2^9 top frequency amplifies fp32 phase error, and ReLU
    masks of near-zero pre-activations flip between float32 and float64: measured 1.06e-4 for d gamma(x) at 4096 points);
  * bf16 mode: the per-point input gradients carry the error of bf16 arithmetic itself -- bf16 activations, weights and dY
    images shift ReLU masks and every layer of the chain -- measured on a B200 at cosine 0.988-0.989 and relative L2 0.15 against
    float64 for both the encodings and the rays, which a float64 emulation of the same bf16 roundings reproduces to four
    digits (relative L2 0.1506 vs 0.1506).  So bf16 is held to that emulation (relative L2 <= 1e-2) and to cosine >= 0.98 /
    relative L2 <= 0.2 against float64;
  * parameter gradients of the combined loss: 5e-3 relative L2 in fp32 mode; bf16 mode measured 0.04-0.08 on this loss (the
    depth term divides by the opacity), held to 0.12."""
import numpy as np
import pytest
import torch

from oracle import nerf_oracle as O

DEV = "cuda"
F64 = torch.float64


# ------------------------------------------------------------------------------------------------ float64 restatement
def encode(x, L):
    """encoders.py:88-106: [x | sin(2^k x) k-major | cos(2^k x)]."""
    fb = 2.0 ** torch.arange(L, dtype=x.dtype, device=x.device)
    xb = x[..., None, :] * fb[:, None]
    enc = torch.cat([torch.sin(xb), torch.cos(xb)], dim=-2).reshape(*x.shape[:-1], -1)
    return torch.cat([x, enc], dim=-1)


def mlp(p, ep, ed):
    """mlps.py:221-278 (skip concat [h, gamma(x)] at layer 4, h first)."""
    h = ep
    for i in range(8):
        if i == 4:
            h = torch.cat([h, ep], dim=-1)
        h = torch.relu(h @ p[f"mlp.{i}.weight"].T + p[f"mlp.{i}.bias"])
    sigma = h @ p["sigma_out.weight"].T + p["sigma_out.bias"]
    feat = h @ p["feature.weight"].T + p["feature.bias"]
    c = torch.relu(torch.cat([feat, ed], dim=-1) @ p["color_fc.weight"].T + p["color_fc.bias"])
    return torch.cat([c @ p["color_out.weight"].T + p["color_out.bias"], sigma], dim=-1)


def composite(rgb, sigma, z, rn, white, eps=1e-10, inf_last=False):
    """render_utils.py:108-167."""
    B = z.shape[0]
    last = torch.full((B, 1), 1e10 if inf_last else 0.0, dtype=z.dtype, device=z.device)
    deltas = torch.cat([z[:, 1:] - z[:, :-1], last], dim=-1)
    if rn is not None:
        deltas = deltas * rn.reshape(B, 1)
    alphas = 1.0 - torch.exp(-torch.clamp(sigma * deltas, 0.0, 60.0))
    shifted = torch.cat([torch.ones((B, 1), dtype=z.dtype, device=z.device), 1.0 - alphas + eps], dim=-1)
    w = torch.nan_to_num(torch.cumprod(shifted, dim=-1)[:, :-1] * alphas, 0.0, 0.0, 0.0)
    acc = torch.clamp(w.sum(-1, keepdim=True), 0.0, 1.0)
    depth = (w * z).sum(-1, keepdim=True) / (acc + eps)
    c = (w[..., None] * rgb).sum(-2)
    if white:
        c = c + (1.0 - acc)
    return torch.clamp(torch.nan_to_num(c, 0.0, 1.0, 0.0), 0.0, 1.0), w, acc, depth


def forward_pass(p, o, d, z, rn, vd, white, noise=None, noise_std=0.0, inf_last=False):
    """render_utils.py:209-276 with relu sigma."""
    B, N = z.shape
    zm = z if rn is None else z * rn.reshape(B, 1)
    pts = o[:, None, :] + d[:, None, :] * zm[..., None]
    v = torch.nn.functional.normalize(vd if vd is not None else d, dim=-1)
    raw = mlp(p, encode(pts.reshape(-1, 3), 10), encode(v[:, None, :].expand_as(pts).reshape(-1, 3), 4))
    sig = raw[:, 3]
    if noise is not None:
        sig = sig + noise * noise_std
    return composite(torch.sigmoid(raw[:, :3]).reshape(B, N, 3), torch.relu(sig).reshape(B, N), z, rn, white, 1e-10, inf_last)


def params_t(p, dtype=F64, device="cpu", grad=False):
    return {k: torch.tensor(v, dtype=dtype, device=device, requires_grad=grad) for k, v in p.items()}


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def cosine(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float(a @ b / max(np.linalg.norm(a) * np.linalg.norm(b), 1e-30))


def N_(t):
    return t.detach().double().cpu().numpy()


def make_case(seed, B, N, ray_norm=True, viewdirs=True):
    rng = np.random.default_rng(seed)
    r = O.synthetic_rays(rng, B)
    z = np.sort(rng.uniform(2.0, 6.0, size=(B, N)), axis=-1).astype(np.float32)
    vd = r["rays_d_world_unit"] + 0.05 * rng.standard_normal((B, 3)).astype(np.float32) if viewdirs else None
    return dict(o=r["rays_o_marching"], d=r["rays_d_marching_unit"], z=z,
                rn=r["rays_d_marching_norm"].reshape(B) if ray_norm else None, vd=vd,
                noise=rng.standard_normal(B * N).astype(np.float32),
                G=[rng.standard_normal(s).astype(np.float32) for s in ((B, 3), (B, N), (B, 1), (B, 1))])


def loss_of(outs, G):
    return sum((o * g).sum() for o, g in zip(outs, G))


# ------------------------------------------------------------------------------------------------ CPU: pin the restatement
def test_restatement_matches_oracle_mlp():
    rng = np.random.default_rng(3)
    p = O.init_params(rng, sigma_bias=0.5)
    ep = O.positional_encode(rng.uniform(-1.5, 1.5, (512, 3)).astype(np.float32), 10)
    ed = O.positional_encode(O._normalize(rng.standard_normal((512, 3)).astype(np.float32)), 4)
    want, caches = O.mlp_forward(p, ep, ed, keep=True)
    d_out = rng.standard_normal((512, 4)).astype(np.float32)
    pt = params_t(p, grad=True)
    raw = mlp(pt, torch.tensor(ep, dtype=F64), torch.tensor(ed, dtype=F64))
    assert rel_l2(N_(raw), want) < 1e-6
    (raw * torch.tensor(d_out, dtype=F64)).sum().backward()
    g = O.mlp_backward(p, caches, d_out)
    # over the whole flat gradient: single small tensors (sigma_out.weight) carry the oracle's own float32 rounding at ~1e-6
    got = np.concatenate([N_(pt[k].grad).ravel() for k, _ in O.PARAM_SHAPES])
    assert rel_l2(got, O.flatten_params(g)) < 1e-6


@pytest.mark.parametrize("white,inf_last", [(False, False), (True, True)])
def test_restatement_matches_oracle_compositor(white, inf_last):
    rng = np.random.default_rng(5)
    B, Nn = 64, 48
    rgb = rng.uniform(0, 1, (B, Nn, 3)).astype(np.float32)
    sigma = rng.uniform(0, 3, (B, Nn)).astype(np.float32)
    z = np.sort(rng.uniform(2, 6, (B, Nn)), -1).astype(np.float32)
    rn = rng.uniform(1, 1.1, B).astype(np.float32)
    gs = [rng.standard_normal(s).astype(np.float32) for s in ((B, 3), (B, Nn), (B, 1), (B, 1))]
    *outs_o, cache = O.volume_render_rays(rgb, sigma, z, rn, white, 1e-10, inf_last, keep=True)
    want_rgb, want_sig = O.volume_render_backward(cache, gs[0], gs[1], gs[2], gs[3])
    rt, st = torch.tensor(rgb, dtype=F64, requires_grad=True), torch.tensor(sigma, dtype=F64, requires_grad=True)
    outs = composite(rt, st, torch.tensor(z, dtype=F64), torch.tensor(rn, dtype=F64), white, 1e-10, inf_last)
    for a, b in zip(outs, outs_o):
        assert rel_l2(N_(a), b) < 1e-6
    loss_of(outs, [torch.tensor(g, dtype=F64) for g in gs]).backward()
    assert rel_l2(N_(rt.grad), want_rgb) < 1e-6
    assert rel_l2(N_(st.grad), want_sig) < 1e-6


def test_restatement_matches_oracle_encoder():
    x = np.random.default_rng(7).uniform(-4, 4, (256, 3)).astype(np.float32)
    assert rel_l2(N_(encode(torch.tensor(x, dtype=F64), 10)), O.positional_encode(x, 10)) < 1e-6


# ------------------------------------------------------------------------------------------------ GPU
def load_nerf(seed, mode):
    import nerf_sandbox_b200 as nsb
    p = O.init_params(np.random.default_rng(int(seed)), sigma_bias=0.1)
    net = nsb.NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu", mode=mode).to(DEV)
    net.load_state_dict({k: torch.tensor(v, device=DEV) for k, v in p.items()})
    return net, p


def run_fused(net, case, training, white, inf_last, rays_grad=True, vd=True):
    from nerf_sandbox_b200 import render
    import nerf_sandbox_b200 as nsb
    pe, de = nsb.get_vanilla_nerf_encoders()
    t = {k: torch.tensor(case[k], device=DEV, requires_grad=rays_grad and k in ("o", "d", "vd"))
         for k in ("o", "d", "vd") if case[k] is not None}
    outs = render.nerf_forward_pass(t["o"], t["d"], torch.tensor(case["z"], device=DEV), pos_enc=pe, dir_enc=de, nerf=net,
                                    white_bkgd=white, ray_norms=None if case["rn"] is None else torch.tensor(case["rn"], device=DEV),
                                    viewdirs_world_unit=t.get("vd") if vd else None, raw_noise_std=1.0 if training else 0.0,
                                    training=training, raw_noise=torch.tensor(case["noise"], device=DEV) if training else None,
                                    infinite_last_bin=inf_last)
    return t, outs


def reference_grads(p, case, training, white, inf_last, dtype, device):
    pt = params_t(p, dtype, device, grad=True)
    t = {k: torch.tensor(case[k], dtype=dtype, device=device, requires_grad=True) for k in ("o", "d", "vd") if case[k] is not None}
    rn = None if case["rn"] is None else torch.tensor(case["rn"], dtype=dtype, device=device)
    outs = forward_pass(pt, t["o"], t["d"], torch.tensor(case["z"], dtype=dtype, device=device), rn, t.get("vd"), white,
                        torch.tensor(case["noise"], dtype=dtype, device=device) if training else None, 1.0, inf_last)
    loss_of(outs, [torch.tensor(g, dtype=dtype, device=device) for g in case["G"]]).backward()
    flat = torch.cat([pt[k].grad.reshape(-1) for k, _ in O.PARAM_SHAPES])
    return {k: N_(v.grad) for k, v in t.items()}, N_(flat), [N_(o) for o in outs]


_REF_CACHE = {}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,Nn,training,white,inf_last", [(1024, 64, False, False, False), (1024, 192, True, True, True)])
def test_fused_pass_input_grads(mode, B, Nn, training, white, inf_last):
    net, p = load_nerf(11, mode)
    case = make_case(100 + Nn, B, Nn, viewdirs=Nn == 64)           # N = 192: the view-direction term goes to rays_d
    t, outs = run_fused(net, case, training, white, inf_last)
    loss_of(outs, [torch.tensor(g, device=DEV) for g in case["G"]]).backward()
    got = {k: N_(v.grad) for k, v in t.items()}
    flat = N_(torch.cat([q.grad.reshape(-1) for q in net.ordered_params()]))
    key = (B, Nn, training, white, inf_last)
    if key not in _REF_CACHE:
        _REF_CACHE[key] = (reference_grads(p, case, training, white, inf_last, F64, DEV),
                           reference_grads(p, case, training, white, inf_last, torch.float32, "cpu"))
    (ref, ref_flat, _), (ref32, _, _) = _REF_CACHE[key]
    assert rel_l2(flat, ref_flat) < (5e-3 if mode == "fp32" else 0.12), rel_l2(flat, ref_flat)
    for k in got:
        if mode == "fp32":
            bar = max(1e-3, 2.0 * rel_l2(ref32[k], ref[k]))
            assert rel_l2(got[k], ref[k]) <= bar, (k, rel_l2(got[k], ref[k]), bar)
        else:
            assert cosine(got[k], ref[k]) >= 0.98 and rel_l2(got[k], ref[k]) <= 0.2, (k, cosine(got[k], ref[k]), rel_l2(got[k], ref[k]))


def bf16_encoding_grads(p, ep, ed, d_out):
    """d gamma(x), d gamma(d) of mlp() with the roundings of the bf16 field kernels: weights, layer inputs and every dY image in
    bf16, fp32-grade accumulation (float64 here)."""
    bf = lambda t: t.to(torch.bfloat16).to(F64)
    W = {k: bf(v) if k.endswith("weight") else v for k, v in p.items()}
    epb, edb = bf(ep), bf(ed)
    h, pre = epb, []
    for i in range(8):
        if i == 4:
            h = torch.cat([h, epb], -1)
        pre.append(h @ W[f"mlp.{i}.weight"].T + W[f"mlp.{i}.bias"])
        h = bf(torch.relu(pre[-1]))
    feat = bf(h @ W["feature.weight"].T + W["feature.bias"])
    cz = torch.cat([feat, edb], -1) @ W["color_fc.weight"].T + W["color_fc.bias"]
    dc = bf((d_out[:, :3] @ p["color_out.weight"]) * (cz > 0))
    dfeat = bf((dc @ W["color_fc.weight"])[:, :256])
    dy = {7: bf((dfeat @ W["feature.weight"] + d_out[:, 3:4] @ p["sigma_out.weight"]) * (pre[7] > 0))}
    for i in range(7, 0, -1):
        dy[i - 1] = bf((dy[i] @ W[f"mlp.{i}.weight"])[:, :256] * (pre[i - 1] > 0))
    return dy[0] @ W["mlp.0.weight"] + dy[4] @ W["mlp.4.weight"][:, 256:], dc @ W["color_fc.weight"][:, 256:]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_nerf_module_encoding_grads(mode):
    import nerf_sandbox_b200 as nsb
    net, p = load_nerf(12, mode)
    rng = np.random.default_rng(21)
    Q = 4096
    x = rng.uniform(-1.5, 1.5, (Q, 3)).astype(np.float32)
    v = O._normalize(rng.standard_normal((Q, 3)).astype(np.float32))
    pe, de = nsb.get_vanilla_nerf_encoders()
    xt = torch.tensor(x, device=DEV, requires_grad=True)
    vt = torch.tensor(v, device=DEV, requires_grad=True)
    ep, ed = pe(xt), de(vt)
    ep.retain_grad(); ed.retain_grad()
    d_out = rng.standard_normal((Q, 4)).astype(np.float32)
    (net(ep, ed) * torch.tensor(d_out, device=DEV)).sum().backward()
    pt = params_t(p, F64, DEV)
    xr = torch.tensor(x, dtype=F64, device=DEV, requires_grad=True)
    vr = torch.tensor(v, dtype=F64, device=DEV, requires_grad=True)
    epr, edr = encode(xr, 10), encode(vr, 4)
    epr.retain_grad(); edr.retain_grad()
    (mlp(pt, epr, edr) * torch.tensor(d_out, dtype=F64, device=DEV)).sum().backward()
    # the same composition in float32 on the CPU: its distance is the float32 floor of this comparison
    p32 = params_t(p, torch.float32)
    x32 = torch.tensor(x, requires_grad=True)
    v32 = torch.tensor(v, requires_grad=True)
    ep32, ed32 = encode(x32, 10), encode(v32, 4)
    ep32.retain_grad(); ed32.retain_grad()
    (mlp(p32, ep32, ed32) * torch.tensor(d_out)).sum().backward()
    pairs = ((ep.grad, epr.grad, ep32.grad), (ed.grad, edr.grad, ed32.grad), (xt.grad, xr.grad, x32.grad), (vt.grad, vr.grad, v32.grad))
    for got, want, f32 in pairs:
        g, w = N_(got), N_(want)
        if mode == "fp32":
            bar = max(1e-4, 2.0 * rel_l2(N_(f32), w))
            assert rel_l2(g, w) <= bar, (rel_l2(g, w), bar)
        else:
            assert cosine(g, w) >= 0.98 and rel_l2(g, w) <= 0.2, (cosine(g, w), rel_l2(g, w))
    if mode == "bf16":
        emu_pos, emu_dir = bf16_encoding_grads(pt, epr.detach(), edr.detach(), torch.tensor(d_out, dtype=F64, device=DEV))
        assert rel_l2(N_(ep.grad), N_(emu_pos)) <= 1e-2, rel_l2(N_(ep.grad), N_(emu_pos))
        assert rel_l2(N_(ed.grad), N_(emu_dir)) <= 1e-2, rel_l2(N_(ed.grad), N_(emu_dir))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_frozen_field(mode):
    from nerf_sandbox_b200 import _lib
    net, _ = load_nerf(13, mode)
    case = make_case(7, 512, 64)
    G = [torch.tensor(g, device=DEV) for g in case["G"]]

    def grads():
        t, outs = run_fused(net, case, False, True, False)
        n0 = _lib.launch_count()
        loss_of(outs, G).backward()
        torch.cuda.synchronize()
        return {k: v.grad.clone() for k, v in t.items()}, _lib.launch_count() - n0

    trainable, n_train = grads()
    for q in net.parameters():
        q.requires_grad_(False)
    try:
        frozen, n_frozen = grads()
        frozen2, _ = grads()
    finally:
        for q in net.parameters():
            q.requires_grad_(True)
    for k in trainable:
        assert torch.equal(trainable[k], frozen[k]), k
        assert torch.equal(frozen[k], frozen2[k]), k
    # a frozen field runs no weight-gradient kernel: one wgrad launch in bf16 mode, one or more per layer in fp32 mode
    if mode == "bf16":
        assert n_train - n_frozen == 1, (n_train, n_frozen)
    else:
        assert n_train - n_frozen >= 10, (n_train, n_frozen)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_no_input_grad_keeps_launches_and_values(mode):
    """Rays that do not require grad: the backward launches exactly what nsb_field_bwd + nsb_composite_raw_bwd launch, and the
    forward's weights / acc / depth are bit-identical to the parent sequence of C calls."""
    from nerf_sandbox_b200 import _lib
    L = _lib.lib()
    net, _ = load_nerf(14, mode)
    B, Nn = 256, 64
    case = make_case(9, B, Nn)
    _, outs = run_fused(net, case, False, False, False, rays_grad=False)
    comp, w, acc, depth = outs
    n0 = _lib.launch_count()
    (comp * torch.tensor(case["G"][0], device=DEV)).sum().backward()
    torch.cuda.synchronize()
    n_module = _lib.launch_count() - n0

    o, d, z = (torch.tensor(case[k], device=DEV) for k in ("o", "d", "z"))
    rn, vd = torch.tensor(case["rn"], device=DEV), torch.tensor(case["vd"], device=DEV)
    packed = net.packed()
    wsb = L.nsb_field_workspace_bytes(B * Nn, net.mode, 1)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    raw = torch.empty((B * Nn, 4), device=DEV)
    P = _lib.ptr
    _lib.check(L.nsb_field_fwd_rays(P(o), P(d), P(z), P(rn), P(vd), P(packed), P(raw), P(ws), wsb, B, Nn, net.mode, 1, _lib.stream()))
    c2, w2, a2, d2 = (torch.empty(s, device=DEV) for s in ((B, 3), (B, Nn), (B, 1), (B, 1)))
    _lib.check(L.nsb_composite_raw_fwd(P(raw), None, 0.0, P(z), P(rn), P(c2), P(w2), P(a2), P(d2), B, Nn, 0, 0, 0, _lib.stream()))
    for a, b in ((comp, c2), (w, w2), (acc, a2), (depth, d2)):
        assert torch.equal(a, b)
    g = torch.zeros(_lib.N_PARAMS, device=DEV)
    d_raw = torch.empty_like(raw)
    gc = torch.tensor(case["G"][0], device=DEV)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    _lib.check(L.nsb_composite_raw_bwd(P(raw), None, 0.0, P(z), P(rn), P(gc), P(d_raw), B, Nn, 0, 0, 0, _lib.stream()))
    _lib.check(L.nsb_field_bwd(P(d_raw), P(packed), P(g), P(ws), wsb, B * Nn, net.mode, _lib.stream()))
    torch.cuda.synchronize()
    assert n_module == _lib.launch_count() - n0


@pytest.mark.gpu
def test_encoder_backward_matches_autograd():
    import nerf_sandbox_b200 as nsb
    x = np.random.default_rng(4).uniform(-3, 3, (2048, 3)).astype(np.float32)
    g = np.random.default_rng(5).standard_normal((2048, 63)).astype(np.float32)
    pe, _ = nsb.get_vanilla_nerf_encoders()
    xt = torch.tensor(x, device=DEV, requires_grad=True)
    (pe(xt) * torch.tensor(g, device=DEV)).sum().backward()
    xr = torch.tensor(x, dtype=F64, requires_grad=True)
    (encode(xr, 10) * torch.tensor(g, dtype=F64)).sum().backward()
    assert rel_l2(N_(xt.grad), N_(xr.grad)) < 1e-4


@pytest.mark.gpu
def test_depth_only_loss_reaches_parameters():
    """A loss on depth alone (no comp term) changes the field's gradients: the compositor backward takes g_depth."""
    from nerf_sandbox_b200 import render
    import nerf_sandbox_b200 as nsb
    net, p = load_nerf(15, "fp32")
    case = make_case(17, 256, 64)
    pe, de = nsb.get_vanilla_nerf_encoders()
    o, d, z, rn = (torch.tensor(case[k], device=DEV) for k in ("o", "d", "z", "rn"))
    _, _, _, depth = render.nerf_forward_pass(o, d, z, pos_enc=pe, dir_enc=de, nerf=net, white_bkgd=False, ray_norms=rn)
    (depth * torch.tensor(case["G"][3], device=DEV)).sum().backward()
    flat = N_(torch.cat([q.grad.reshape(-1) for q in net.ordered_params()]))
    pt = params_t(p, F64, DEV, grad=True)
    f64 = lambda k: torch.tensor(case[k], dtype=F64, device=DEV)
    outs = forward_pass(pt, f64("o"), f64("d"), f64("z"), f64("rn"), None, False)
    (outs[3] * torch.tensor(case["G"][3], dtype=F64, device=DEV)).sum().backward()
    ref = N_(torch.cat([pt[k].grad.reshape(-1) for k, _ in O.PARAM_SHAPES]))
    assert np.linalg.norm(flat) > 0 and rel_l2(flat, ref) < 5e-3
