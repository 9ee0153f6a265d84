"""CPU oracle for the vanilla-NeRF ray-march path (TEST INFRASTRUCTURE ONLY).

This file is a numpy fp32 restatement of the reference's hot path
(evan-wes/nerf-sandbox).  It is the *checker* for the CUDA kernels: only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it.  Nothing under ``nerf_sandbox_b200/``
imports it, and the product path raises when the CUDA library is missing.

Where the arithmetic lives: the reference delegates every op to PyTorch/ATen
(``requirements.txt:2`` lists ``torch`` unpinned; 2.11.0 in this image).  Each
function below restates the ATen op sequence of the cited reference lines in
numpy float32.  Parity pin: ``tests/make_golden.py`` imports the reference from
its checkout (``NSB_REFERENCE_SRC``, else BASELINE.json's ``reference_path``), runs it on seeded inputs and
commits the input/output vectors under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this file against them (bit-exact for
``sample_pdf`` bin indices and the stratified/merge samplers, <=2e-6 for the
floating-point outputs).  The reference's own unit tests pin no numerics for
this path (SURVEY.md section 4), so those generated vectors are the pin.

All arrays are float32 unless stated; parameter dicts use the reference's
``state_dict`` keys (``mlp.0.weight`` ... ``color_out.bias``).
"""
from __future__ import annotations

import numpy as np

F32 = np.float32


def _f(x):
    return np.asarray(x, dtype=F32)


# --------------------------------------------------------------------------
# a1. Positional encoder -- models/encoders.py:73-106 (factory :108-123)
# --------------------------------------------------------------------------
def positional_encode(x: np.ndarray, num_freqs: int, include_input: bool = True) -> np.ndarray:
    """gamma(x) = [x | sin(2^k x_d), k-major then d | cos(2^k x_d) same order].

    encoders.py:61 (freq_bands = 2**linspace(0, L-1, L)), :95 (xb = x[...,None,:]*fb[:,None]),
    :97-98 (sin, cos), :101 (cat on the freq axis, then flatten), :104 (input prepended).
    """
    x = _f(x)
    fb = (F32(2.0) ** np.arange(num_freqs, dtype=F32)).astype(F32)       # exact powers of two
    xb = x[..., None, :] * fb[:, None]                                   # (..., L, D)
    enc = np.concatenate([np.sin(xb), np.cos(xb)], axis=-2)              # (..., 2L, D)
    enc = enc.reshape(*x.shape[:-1], -1).astype(F32)
    if include_input:
        enc = np.concatenate([x, enc], axis=-1)
    return enc


# --------------------------------------------------------------------------
# a2/a3. NeRF MLP -- models/mlps.py:41-134 (layout), :192-278 (forward)
# --------------------------------------------------------------------------
PARAM_SHAPES = [
    ("mlp.0.weight", (256, 63)), ("mlp.0.bias", (256,)),
    ("mlp.1.weight", (256, 256)), ("mlp.1.bias", (256,)),
    ("mlp.2.weight", (256, 256)), ("mlp.2.bias", (256,)),
    ("mlp.3.weight", (256, 256)), ("mlp.3.bias", (256,)),
    ("mlp.4.weight", (256, 319)), ("mlp.4.bias", (256,)),
    ("mlp.5.weight", (256, 256)), ("mlp.5.bias", (256,)),
    ("mlp.6.weight", (256, 256)), ("mlp.6.bias", (256,)),
    ("mlp.7.weight", (256, 256)), ("mlp.7.bias", (256,)),
    ("feature.weight", (256, 256)), ("feature.bias", (256,)),
    ("sigma_out.weight", (1, 256)), ("sigma_out.bias", (1,)),
    ("color_fc.weight", (128, 283)), ("color_fc.bias", (128,)),
    ("color_out.weight", (3, 128)), ("color_out.bias", (3,)),
]
N_PARAMS = sum(int(np.prod(s)) for _, s in PARAM_SHAPES)  # 595,844 (SURVEY section 5)


def init_params(rng: np.random.Generator, sigma_bias: float | None = None) -> dict:
    """Random-init weights with the reference's init *distributions*
    (mlps.py:178-190: Kaiming-uniform trunk/feature/color_fc, zero biases;
    PyTorch default for sigma_out/color_out).  Not bit-identical to torch's
    RNG stream -- parity tests load torch-generated weights from the goldens."""
    p = {}
    for name, shp in PARAM_SHAPES:
        if name.endswith("weight"):
            fan_in = shp[1]
            base = name.rsplit(".", 1)[0]
            if base.startswith("mlp") or base == "color_fc":
                bound = np.sqrt(6.0 / fan_in)            # gain sqrt(2) * sqrt(3/fan_in)
            elif base == "feature":
                bound = np.sqrt(3.0 / fan_in)            # gain 1
            else:
                bound = 1.0 / np.sqrt(fan_in)            # nn.Linear default (kaiming a=sqrt(5))
            p[name] = rng.uniform(-bound, bound, size=shp).astype(F32)
        else:
            base = name.rsplit(".", 1)[0]
            if base in ("sigma_out", "color_out"):
                fan_in = dict(PARAM_SHAPES)[base + ".weight"][1]
                bound = 1.0 / np.sqrt(fan_in)
                p[name] = rng.uniform(-bound, bound, size=shp).astype(F32)
            else:
                p[name] = np.zeros(shp, dtype=F32)
    if sigma_bias is not None:
        p["sigma_out.bias"] = np.full((1,), sigma_bias, dtype=F32)
    return p


def flatten_params(p: dict) -> np.ndarray:
    return np.concatenate([_f(p[n]).reshape(-1) for n, _ in PARAM_SHAPES])


def unflatten_params(flat: np.ndarray) -> dict:
    out, off = {}, 0
    for n, s in PARAM_SHAPES:
        k = int(np.prod(s))
        out[n] = _f(flat[off:off + k]).reshape(s)
        off += k
    return out


_CHUNK = 8192     # rows per block: keeps the elementwise passes cache-resident (numpy runs them on one thread)


def _mlp_forward_block(p, enc_pos, enc_dir, keep):
    h = enc_pos
    xs, hs = [], []
    for i in range(8):
        if i == 4:                                        # mlps.py:225-227: cat([h, enc_pos]) (h first)
            h = np.concatenate([h, enc_pos], axis=-1)
        xs.append(h)
        h = h @ p[f"mlp.{i}.weight"].T
        h += p[f"mlp.{i}.bias"]
        np.maximum(h, F32(0), out=h)                      # :244
        hs.append(h)
    sigma_raw = h @ p["sigma_out.weight"].T + p["sigma_out.bias"]                 # :265
    feat = h @ p["feature.weight"].T + p["feature.bias"]                          # :268 (no act)
    cin = np.concatenate([feat, enc_dir], axis=-1)                                # :271
    c = np.maximum(cin @ p["color_fc.weight"].T + p["color_fc.bias"], F32(0))     # :272
    rgb_raw = c @ p["color_out.weight"].T + p["color_out.bias"]                   # :273
    out = np.concatenate([rgb_raw, sigma_raw], axis=-1).astype(F32)               # :276
    return out, (dict(xs=xs, hs=hs, cin=cin, c=c) if keep else None)


def mlp_forward(p: dict, enc_pos: np.ndarray, enc_dir: np.ndarray, keep: bool = False):
    """mlps.py:221-278.  Returns raw [r,g,b,sigma] (Q,4); with keep=True also the
    tensors the backward needs (a list of per-row-block caches)."""
    enc_pos, enc_dir = _f(enc_pos), _f(enc_dir)
    outs, caches = [], []
    for s in range(0, max(enc_pos.shape[0], 1), _CHUNK):
        o, c = _mlp_forward_block(p, enc_pos[s:s + _CHUNK], enc_dir[s:s + _CHUNK], keep)
        outs.append(o); caches.append(c)
    out = np.concatenate(outs, axis=0)
    return (out, caches) if keep else out


def _mlp_backward_block(p, cache, d_out, g):
    xs, hs, cin, c = cache["xs"], cache["hs"], cache["cin"], cache["c"]
    h8 = hs[7]
    d_rgb = _f(d_out[:, :3]); d_sig = _f(d_out[:, 3:4])

    def acc(name, val):
        g[name] = val if name not in g else g[name] + val

    acc("color_out.weight", d_rgb.T @ c); acc("color_out.bias", d_rgb.sum(0))
    dc = (d_rgb @ p["color_out.weight"]) * (c > 0)
    acc("color_fc.weight", dc.T @ cin); acc("color_fc.bias", dc.sum(0))
    dfeat = (dc @ p["color_fc.weight"])[:, :256]
    acc("feature.weight", dfeat.T @ h8); acc("feature.bias", dfeat.sum(0))
    acc("sigma_out.weight", d_sig.T @ h8); acc("sigma_out.bias", d_sig.sum(0))
    dh = dfeat @ p["feature.weight"] + d_sig @ p["sigma_out.weight"]
    for i in range(7, -1, -1):
        dh *= (hs[i] > 0)
        acc(f"mlp.{i}.weight", dh.T @ xs[i]); acc(f"mlp.{i}.bias", dh.sum(0))
        if i > 0:
            dh = dh @ p[f"mlp.{i}.weight"]
            if i == 4:
                dh = np.ascontiguousarray(dh[:, :256])


def mlp_backward(p: dict, caches: list, d_out: np.ndarray) -> dict:
    """Autograd of mlp_forward w.r.t. the parameters only (inputs carry no grad,
    SURVEY section 8 a12)."""
    g = {}
    s = 0
    for cache in caches:
        n = cache["c"].shape[0]
        _mlp_backward_block(p, cache, d_out[s:s + n], g)
        s += n
    return {k: _f(v) for k, v in g.items()}


# --------------------------------------------------------------------------
# a5. Volume compositor -- utils/render_utils.py:108-167
# --------------------------------------------------------------------------
def _nan_to_num(x, nan=0.0, posinf=None, neginf=None):
    return np.nan_to_num(x, nan=nan,
                         posinf=np.finfo(F32).max if posinf is None else posinf,
                         neginf=np.finfo(F32).min if neginf is None else neginf).astype(F32)


def volume_render_rays(rgb, sigma, z, ray_norm=None, white_bkgd=False, eps=1e-10,
                       infinite_last_bin=False, keep=False):
    rgb, sigma, z = _f(rgb), _f(sigma), _f(z)
    B, N = z.shape
    eps = F32(eps)
    d_fin = z[:, 1:] - z[:, :-1]                                                   # :131
    last = np.full((B, 1), 1e10 if infinite_last_bin else 0.0, dtype=F32)          # :132-135
    deltas = np.concatenate([d_fin, last], axis=-1)                                # :136
    if ray_norm is not None:
        deltas = deltas * _f(ray_norm).reshape(B, 1)                               # :139-141
    with np.errstate(over="ignore", invalid="ignore"):
        sd_raw = sigma * deltas
        sdt = np.minimum(np.maximum(sd_raw, F32(0)), F32(60))                      # :144
        alphas = F32(1) - np.exp(-sdt)                                             # :145
        shifted = np.concatenate([np.ones((B, 1), F32), F32(1) - alphas + eps], axis=-1)   # :148-149
        trans = np.cumprod(shifted, axis=-1, dtype=F32)[:, :-1]                    # :150
        w_raw = trans * alphas                                                     # :153
        weights = _nan_to_num(w_raw, 0.0, 0.0, 0.0)                                # :154
        s = weights.sum(-1, keepdims=True, dtype=F32)
        acc = np.clip(s, F32(0), F32(1))                                           # :156
        depth = (weights * z).sum(-1, keepdims=True, dtype=F32) / (acc + eps)      # :157
        c_raw = (weights[..., None] * rgb).sum(-2, dtype=F32)                      # :160
        if white_bkgd:
            c_raw = c_raw + (F32(1) - acc)                                         # :162
        comp = np.clip(_nan_to_num(c_raw, 0.0, 1.0, 0.0), F32(0), F32(1))          # :165
    if keep:
        return comp, weights, acc, depth, dict(rgb=rgb, z=z, deltas=deltas, sd_raw=sd_raw, alphas=alphas,
                                               trans=trans, w_raw=w_raw, weights=weights, s=s, acc=acc,
                                               c_raw=c_raw, white=white_bkgd, eps=eps)
    return comp, weights, acc, depth


def volume_render_backward(cache, g_comp, g_weights=None, g_acc=None, g_depth=None):
    """Autograd of volume_render_rays w.r.t. (rgb, sigma), reproducing ATen's
    masks: clamp passes grad on the closed interval, nan_to_num where finite,
    cumprod_backward's division form (no exact zeros occur: 1-a+1e-10 >= 1e-10).
    Returns (d_rgb (B,N,3), d_sigma (B,N))."""
    rgb, z, deltas, alphas, trans = cache["rgb"], cache["z"], cache["deltas"], cache["alphas"], cache["trans"]
    weights, s, acc, c_raw, eps = cache["weights"], cache["s"], cache["acc"], cache["c_raw"], cache["eps"]
    B, N = z.shape
    g_comp = _f(g_comp)
    m_c = (np.isfinite(c_raw) & (c_raw >= 0) & (c_raw <= 1)).astype(F32)
    gc = g_comp * m_c                                                              # (B,3)
    g_accv = np.zeros((B, 1), F32) if g_acc is None else _f(g_acc).reshape(B, 1).copy()
    G = np.zeros((B, N), F32) if g_weights is None else _f(g_weights).copy()
    if cache["white"]:
        g_accv = g_accv - gc.sum(-1, keepdims=True)
    if g_depth is not None:
        gd = _f(g_depth).reshape(B, 1)
        swz = (weights * z).sum(-1, keepdims=True, dtype=F32)
        G = G + gd * z / (acc + eps)
        g_accv = g_accv - gd * swz / ((acc + eps) * (acc + eps))
    g_s = g_accv * ((s >= 0) & (s <= 1))
    G = G + g_s + (rgb * gc[:, None, :]).sum(-1)
    d_rgb = weights[..., None] * gc[:, None, :]
    G = G * np.isfinite(cache["w_raw"])
    f = F32(1) - alphas + eps
    Gw = G * weights                                                               # = dT_i * T_i
    suffix = np.cumsum(Gw[:, ::-1], axis=-1, dtype=F32)[:, ::-1] - Gw              # sum_{i>k}
    d_alpha = G * trans - suffix / f
    d_sdt = d_alpha * (F32(1) - alphas)                                            # exp(-sdt)
    sd = cache["sd_raw"]
    d_sigma = d_sdt * deltas * ((sd >= 0) & (sd <= 60))
    return _f(d_rgb), _f(d_sigma)


# --------------------------------------------------------------------------
# a4. nerf_forward_pass -- utils/render_utils.py:171-283
# --------------------------------------------------------------------------
def _normalize(v):
    n = np.sqrt((v * v).sum(-1, keepdims=True, dtype=F32))
    return (v / np.maximum(n, F32(1e-12))).astype(F32)              # F.normalize, :219


def ray_points(rays_o, rays_d_unit, z_vals, ray_norms):
    """render_utils.py:211-215."""
    zm = z_vals if ray_norms is None else z_vals * _f(ray_norms).reshape(-1, 1)
    return (_f(rays_o)[:, None, :] + _f(rays_d_unit)[:, None, :] * zm[..., None]).astype(F32)


def nerf_forward_pass(rays_o, rays_d_unit, z_vals, *, params, white_bkgd, ray_norms=None,
                      viewdirs_world_unit=None, raw_noise=None, raw_noise_std=0.0, training=False,
                      infinite_last_bin=False, keep=False, Lx=10, Ld=4):
    """raw_noise: explicit N(0,1) draws (B*N,) replacing torch.randn at :240."""
    z_vals = _f(z_vals)
    B, N = z_vals.shape
    pts = ray_points(rays_o, rays_d_unit, z_vals, ray_norms)
    vd = _normalize(_f(viewdirs_world_unit if viewdirs_world_unit is not None else rays_d_unit))   # :218-222
    vdirs = np.broadcast_to(vd[:, None, :], pts.shape)
    epos = positional_encode(pts.reshape(-1, 3), Lx)                                # :259
    edir = positional_encode(vdirs.reshape(-1, 3), Ld)                              # :260
    if keep:
        raw, mcache = mlp_forward(params, epos, edir, keep=True)
    else:
        raw = mlp_forward(params, epos, edir)
    rgb = (F32(1) / (F32(1) + np.exp(-raw[:, :3]))).astype(F32)                     # :236 sigmoid
    sig_pre = raw[:, 3]
    if training and raw_noise_std > 0.0:                                            # :239-241
        sig_pre = sig_pre + _f(raw_noise).reshape(-1) * F32(raw_noise_std)
    sigma = np.maximum(sig_pre, F32(0))                                             # :246 relu
    rn = None if ray_norms is None else _f(ray_norms).reshape(B, 1)
    res = volume_render_rays(rgb.reshape(B, N, 3), sigma.reshape(B, N), z_vals, rn, white_bkgd,
                             1e-10, infinite_last_bin, keep=keep)                   # :269-276
    if keep:
        comp, w, acc, depth, vcache = res
        return comp, w, acc, depth, dict(m=mcache, v=vcache, rgb=rgb, sig_pre=sig_pre, raw=raw)
    return res


def nerf_forward_pass_backward(params, cache, g_comp):
    """Parameter grads of one pass given dL/d(comp_rgb)."""
    d_rgb, d_sigma = volume_render_backward(cache["v"], g_comp)
    rgb = cache["rgb"]
    d_raw = np.empty_like(cache["raw"])
    d_raw[:, :3] = d_rgb.reshape(-1, 3) * rgb * (F32(1) - rgb)
    d_raw[:, 3] = d_sigma.reshape(-1) * (cache["sig_pre"] > 0)
    return mlp_backward(params, cache["m"], d_raw), d_raw


# --------------------------------------------------------------------------
# a6. Stratified coarse sampler -- train/trainer.py:901-908; eval render_utils.py:330-331
# --------------------------------------------------------------------------
def linspace01(n: int) -> np.ndarray:
    """ATen linspace(0,1,n) fp32 (RangeFactories symmetric fill): step=(end-start)/(n-1);
    i<n/2: start+step*i, else end-step*(n-1-i) evaluated as ONE fused multiply-add (the
    vectorised CPU kernel contracts it; verified bitwise against torch 2.11 for n in 2..256)."""
    if n == 1:
        return np.zeros(1, F32)
    step = F32(1.0) / F32(n - 1)
    i = np.arange(n)
    lo = (step * i.astype(F32)).astype(F32)
    hi = (1.0 - np.float64(step) * (n - 1 - i)).astype(F32)          # exact product, single rounding == fma
    return np.where(i < n // 2, lo, hi).astype(F32)


def coarse_z(near: float, far: float, nc: int) -> np.ndarray:
    t = linspace01(nc)
    return (F32(near) * (F32(1) - t) + F32(far) * t).astype(F32)     # trainer.py:902


def stratified_z(near: float, far: float, nc: int, U: np.ndarray) -> np.ndarray:
    """U (B,nc) in [0,1) replaces torch.rand_like at trainer.py:907."""
    zc = np.broadcast_to(coarse_z(near, far, nc), U.shape)
    mids = F32(0.5) * (zc[:, 1:] + zc[:, :-1])                      # :904
    lower = np.concatenate([zc[:, :1], mids], -1)                   # :905
    upper = np.concatenate([mids, zc[:, -1:]], -1)                  # :906
    z = lower + (upper - lower) * _f(U)                             # :907
    return np.sort(z, axis=-1).astype(F32)                          # :908


# --------------------------------------------------------------------------
# a7. Interval weights -- train/trainer.py:926-928
# --------------------------------------------------------------------------
def interval_bins(z: np.ndarray, w: np.ndarray):
    bins_mid = F32(0.5) * (z[:, 1:] + z[:, :-1])
    wb = F32(0.5) * (w[:, 1:] + w[:, :-1]) + F32(1e-5)
    return bins_mid.astype(F32), wb.astype(F32)


# --------------------------------------------------------------------------
# a8. sample_pdf -- utils/sampling_utils.py:5-64
# --------------------------------------------------------------------------
def pdf_edges(bins: np.ndarray, M: int) -> np.ndarray:
    bins = _f(bins)
    if bins.ndim != 2:
        raise ValueError(f"Expected (B,.) tensors: bins={bins.shape}")
    if bins.shape[-1] == M + 1:                                     # :22-23
        return bins
    if bins.shape[-1] == M:                                         # :24-33
        if M == 1:
            d = np.full_like(bins, 1e-3)
            return np.concatenate([bins - F32(0.5) * d, bins + F32(0.5) * d], -1)
        lo = bins[:, :1] - F32(0.5) * (bins[:, 1:2] - bins[:, :1])
        hi = bins[:, -1:] + F32(0.5) * (bins[:, -1:] - bins[:, -2:-1])
        inter = F32(0.5) * (bins[:, 1:] + bins[:, :-1])
        return np.concatenate([lo, inter, hi], -1).astype(F32)
    raise ValueError(f"Incompatible shapes: bins={bins.shape}, M={M}")


def pdf_cdf(weights: np.ndarray) -> np.ndarray:
    """:38-41.  cumsum is sequential fp32 like ATen's CPU kernel."""
    w = np.maximum(_f(weights) + F32(1e-5), F32(0))
    pdf = (w / w.sum(-1, keepdims=True, dtype=F32)).astype(F32)
    cdf = np.cumsum(pdf, axis=-1, dtype=F32)
    return np.concatenate([np.zeros((w.shape[0], 1), F32), cdf], -1).astype(F32)


def invert_cdf(edges: np.ndarray, cdf: np.ndarray, u: np.ndarray):
    """:51-64.  Returns (samples (B,n), inds (B,n) int64) -- inds is
    searchsorted(cdf, u, right=True), the quantity that must be bit-exact."""
    B, M1 = cdf.shape
    inds = np.stack([np.searchsorted(cdf[b], u[b], side="right") for b in range(B)]).astype(np.int64)
    below = np.clip(inds - 1, 0, M1 - 1)
    above = np.clip(inds, 1, M1 - 1)
    cdf_lo = np.take_along_axis(cdf, below, -1); cdf_hi = np.take_along_axis(cdf, above, -1)
    e_lo = np.take_along_axis(edges, below, -1); e_hi = np.take_along_axis(edges, above, -1)
    denom = cdf_hi - cdf_lo
    denom = np.where(denom < F32(1e-5), F32(1), denom)              # :62
    t = (u - cdf_lo) / denom
    return (e_lo + t * (e_hi - e_lo)).astype(F32), inds


def sample_pdf(bins, weights, n_samples, *, deterministic=False, u=None, cdf=None, return_inds=False):
    """u: explicit uniforms (B,n) replacing torch.rand at :48; cdf: explicit CDF
    (B,M+1) to pin the searchsorted indices independently of summation order."""
    weights = _f(weights)
    if weights.ndim != 2:
        raise ValueError(f"Expected (B,.) tensors: weights={weights.shape}")
    B, M = weights.shape
    edges = pdf_edges(bins, M)
    if cdf is None:
        cdf = pdf_cdf(weights)
    if deterministic:                                               # :44-46
        u = np.broadcast_to(linspace01(n_samples), (B, n_samples)).copy()
    elif u is None:
        raise ValueError("oracle needs explicit uniforms when not deterministic")
    out, inds = invert_cdf(edges, _f(cdf), _f(u))
    return (out, inds) if return_inds else out


# --------------------------------------------------------------------------
# a9. merge -- train/trainer.py:981
# --------------------------------------------------------------------------
def merge_sorted(zc, zf):
    return np.sort(np.concatenate([_f(zc), _f(zf)], -1), axis=-1)


# --------------------------------------------------------------------------
# a10. loss -- train/trainer.py:999-1006 ;  psnr trainer.py:77-78
# --------------------------------------------------------------------------
def _guard(x):
    return np.clip(_nan_to_num(x, 0.0, 1.0, 0.0), F32(0), F32(1))


def loss_and_grads(comp_c, comp_f, target):
    cc, cf, t = _guard(comp_c), _guard(comp_f), _guard(target)
    n = F32(cc.size)
    mse_c = ((cc - t) ** 2).sum(dtype=F32) / n
    mse_f = ((cf - t) ** 2).sum(dtype=F32) / n
    psnr = F32(-10.0) * np.log10(np.maximum(mse_f, F32(1e-10)))
    m_c = (np.isfinite(comp_c) & (comp_c >= 0) & (comp_c <= 1))
    m_f = (np.isfinite(comp_f) & (comp_f >= 0) & (comp_f <= 1))
    g_c = (F32(2) * (cc - t) / n) * m_c
    g_f = (F32(2) * (cf - t) / n) * m_f
    return F32(mse_c + mse_f), F32(psnr), _f(g_c), _f(g_f)


# --------------------------------------------------------------------------
# Whole train step -- train/trainer.py:876-1013 (+ backward, a12)
# --------------------------------------------------------------------------
def train_step(params_c, params_f, batch, *, near, far, nc, nf, U, u_fine, noise_c, noise_f,
               white_bkgd=True, raw_noise_std=1.0, infinite_last_bin=True, det_fine=False,
               want_grads=True):
    """batch keys as trainer.py:880-884.  U (B,nc), u_fine (B,nf), noise_c (B*nc,),
    noise_f (B*(nc+nf),) are the explicit random draws."""
    o, d = batch["rays_o_marching"], batch["rays_d_marching_unit"]
    rn, vd, tgt = batch["rays_d_marching_norm"], batch["rays_d_world_unit"], batch["rgb"]
    zc = stratified_z(near, far, nc, U)
    comp_c, w_c, _, _, cache_c = nerf_forward_pass(
        o, d, zc, params=params_c, white_bkgd=white_bkgd, ray_norms=rn, viewdirs_world_unit=vd,
        raw_noise=noise_c, raw_noise_std=raw_noise_std, training=True,
        infinite_last_bin=infinite_last_bin, keep=True)
    bins_mid, wb = interval_bins(zc, w_c)
    zf = sample_pdf(bins_mid, wb, nf, deterministic=det_fine, u=u_fine)
    z_all = merge_sorted(zc, zf)
    comp_f, _, acc_f, depth_f, cache_f = nerf_forward_pass(
        o, d, z_all, params=params_f, white_bkgd=white_bkgd, ray_norms=rn, viewdirs_world_unit=vd,
        raw_noise=noise_f, raw_noise_std=raw_noise_std, training=True,
        infinite_last_bin=infinite_last_bin, keep=True)
    loss, psnr, g_c, g_f = loss_and_grads(comp_c, comp_f, tgt)
    out = dict(loss=loss, psnr=psnr, comp_c=_guard(comp_c), comp_f=_guard(comp_f), zc=zc, zf=zf,
               z_all=z_all, w_c=w_c, acc_f=acc_f, depth_f=depth_f)
    if want_grads:
        out["grads_c"], _ = nerf_forward_pass_backward(params_c, cache_c, g_c)
        out["grads_f"], _ = nerf_forward_pass_backward(params_f, cache_f, g_f)
    return out


def adam_step(p, g, m, v, step, lr=5e-4, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam (trainer.py:383-386) single-tensor formula, fp32."""
    p, g, m, v = _f(p), _f(g), _f(m), _f(v)
    m = F32(b1) * m + F32(1 - b1) * g
    v = F32(b2) * v + F32(1 - b2) * g * g
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    denom = np.sqrt(v) / F32(np.sqrt(bc2)) + F32(eps)
    p = p - F32(lr / bc1) * (m / denom)
    return _f(p), _f(m), _f(v)


# --------------------------------------------------------------------------
# a11. Eval render of a ray tile -- utils/render_utils.py:337-417 (one chunk)
# --------------------------------------------------------------------------
def render_rays_eval(params_c, params_f, rays_o, rays_d_unit, ray_norms, viewdirs, *, near, far, nc, nf,
                     white_bkgd=True, infinite_last_bin=False):
    B = rays_o.shape[0]
    zc = np.broadcast_to(coarse_z(near, far, nc), (B, nc)).copy()                   # :330-331,351
    comp_c, w_c, acc_c, depth_c = nerf_forward_pass(
        rays_o, rays_d_unit, zc, params=params_c, white_bkgd=white_bkgd, ray_norms=ray_norms,
        viewdirs_world_unit=viewdirs, infinite_last_bin=infinite_last_bin)
    if nf is None or nf <= 0 or params_f is None:                                   # :381-385
        return dict(rgb=comp_c, acc=acc_c, depth=depth_c, z_all=zc)
    bins_mid, wb = interval_bins(zc, w_c)                                           # :388-390
    zf = sample_pdf(bins_mid, wb, nf, deterministic=True)                           # :394
    z_all = merge_sorted(zc, zf)                                                    # :395
    comp_f, _, acc_f, depth_f = nerf_forward_pass(
        rays_o, rays_d_unit, z_all, params=params_f, white_bkgd=white_bkgd, ray_norms=ray_norms,
        viewdirs_world_unit=viewdirs, infinite_last_bin=infinite_last_bin)
    return dict(rgb=comp_f, acc=acc_f, depth=depth_f, z_all=z_all, w_c=w_c)


# --------------------------------------------------------------------------
# Synthetic inputs -- SURVEY section 8d cfg1/cfg2 recipe (no dataset needed)
# --------------------------------------------------------------------------
def synthetic_rays(rng: np.random.Generator, B: int, radius: float = 4.0311):
    o = rng.standard_normal((B, 3)).astype(F32)
    o = (F32(radius) * o / np.linalg.norm(o, axis=-1, keepdims=True)).astype(F32)
    d = (-o + F32(0.35) * rng.standard_normal((B, 3)).astype(F32)).astype(F32)
    d = (d / np.linalg.norm(d, axis=-1, keepdims=True)).astype(F32)
    norms = rng.uniform(1.0, 1.12, size=(B, 1)).astype(F32)
    tgt = rng.uniform(0.0, 1.0, size=(B, 3)).astype(F32)
    return dict(rays_o_marching=o, rays_d_marching_unit=d, rays_d_marching_norm=norms,
                rays_d_world_unit=d.copy(), rgb=tgt)


# --------------------------------------------------------------------------
# Ray generation + NDC warp -- utils/ray_utils.py:10-136 (SURVEY section 8f rank 1)
# --------------------------------------------------------------------------
def camera_rays(H, W, K, c2w, *, convention="opengl", pixel_center=False, as_ndc=False, near_plane=1.0, pixels_xy=None):
    K, c2w = _f(K), _f(c2w)
    R, t = c2w[:3, :3], c2w[:3, 3]
    if pixels_xy is None:                                                    # :44-54
        ys, xs = np.meshgrid(np.arange(H, dtype=F32), np.arange(W, dtype=F32), indexing="ij")
        x, y = xs.reshape(-1), ys.reshape(-1)
    else:                                                                    # :55-60
        px = _f(pixels_xy).reshape(-1, 2)
        x, y = px[:, 0], px[:, 1]
    if pixel_center:
        x, y = x + F32(0.5), y + F32(0.5)
    xc, yc = (x - K[0, 2]) / K[0, 0], (y - K[1, 2]) / K[1, 1]                # :63-67
    conv = (convention or "opengl").lower()
    one = np.ones_like(xc)
    if conv in ("opengl", "blender", "nerf"):
        dc = np.stack([xc, -yc, -one], -1)
    elif conv in ("opencv", "colmap"):
        dc = np.stack([xc, yc, one], -1)
    elif conv in ("pytorch3d", "p3d"):
        dc = np.stack([xc, -yc, one], -1)
    else:
        raise ValueError(f"Unknown convention '{convention}'")
    d = (dc @ R.T).astype(F32)                                               # :80
    nrm = np.sqrt((d * d).sum(-1, keepdims=True, dtype=F32))                 # :81
    du = (d / (nrm + F32(1e-9))).astype(F32)                                 # :82
    o = np.broadcast_to(t, d.shape).astype(F32)
    if not as_ndc:                                                           # :86-90
        return o, du, nrm, o, du, nrm
    sx, sy = F32(2.0) * K[0, 0] / F32(W), F32(2.0) * K[0, 0] / F32(H)        # :100-102
    tn = -(F32(near_plane) + o[:, 2]) / (d[:, 2] + F32(1e-9))                # :108
    ow = o + tn[:, None] * d
    oz, dz = ow[:, 2] + F32(1e-9), d[:, 2] + F32(1e-9)
    o0, o1, o2 = -sx * (ow[:, 0] / oz), -sy * (ow[:, 1] / oz), F32(1) + F32(2) * F32(near_plane) / oz      # :112-114
    d0 = -sx * (d[:, 0] / dz - ow[:, 0] / oz); d1 = -sy * (d[:, 1] / dz - ow[:, 1] / oz); d2 = -F32(2) * F32(near_plane) / oz
    om, dm = np.stack([o0, o1, o2], -1).astype(F32), np.stack([d0, d1, d2], -1).astype(F32)
    nn = np.sqrt((dm * dm).sum(-1, keepdims=True, dtype=F32))               # :125
    return o, du, nrm, om, (dm / np.maximum(nn, F32(1e-12))).astype(F32), nn  # :126
