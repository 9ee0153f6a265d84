"""Every tile of the field backward against the same points run alone, and against float64, at the sizes training runs.

Both arithmetic modes divide the backward into 128-point tiles: bf16 mode by field_dgrad_kernel (CTA pairs, iterating once
tiles > 2 * num_sms), field_dinput_kernel and field_wgrad_kernel (each CTA walks tiles `tile += cta_count`, a second tile per
CTA once the 13 jobs want more than num_sms CTAs, ~12 tiles); fp32 mode by head_bwd_kernel (one warp per point, grid capped at
4 * num_sms blocks = 32 * num_sms points per sweep) and split_gemm's split-K weight gradient (splits of a multiple of 16 points,
so a tile can straddle two splits).  Whole-step tolerances cannot see a tile that is dropped, counted twice or paired with
another tile's activations: at 1,536 tiles that moves the gradient by ~1/1536.

Every point's forward, stash, dY rows and input gradients depend on that point alone, and the weight gradient is a sum over
points.  So the tests zero d_raw everywhere except on a group of tiles and run the backward over the whole batch (same stash,
same schedule, same CTAs): the result must equal the gradient of those points run as a batch of their own, element by element,
within 2^-20 * (|dY|^T |X|)_ij (sum |dY| for biases; float32 sums of the same products in another order; 2^-18 for groups in
bf16 mode, see WG_TOL_BF16_GROUP), with the magnitudes from the float64 restatement below.  A single tile in bf16 mode must
match bit for bit.  A dropped tile in a group of eight is ~1e-2 of that magnitude, four orders
above the bound.  d_out has a nonzero mean so that tile contributions do not cancel.

The float64 restatement (`mlp_grads`) writes the backward of test_gpu_input_grads.mlp out layer by layer, so that it also
returns the magnitudes; with `rnd=bf16r` it rounds where the bf16 training kernels round.  The CPU tests pin it to autograd,
to the oracle and to test_gpu_tc.bf16_emulated_mlp.

Each GPU test prints the largest ratio to its bound it measured (pytest -s)."""
import math

import numpy as np
import pytest
import torch

import test_gpu_input_grads as IG
import test_gpu_tc as TC
from oracle import nerf_oracle as O

DEV = "cuda"
F64 = torch.float64
TILE = 128
WG_TOL = 2.0 ** -20          # isolated tile / group vs the same points alone, per element, relative to |dY|^T |X|
# bf16 groups: tcgen05 adds every MMA into its fp32 accumulator with truncation (up to 1 ulp each).  Alone, each of a group's
# tiles has a wgrad CTA of its own (8 MMAs per accumulator); in the whole batch, tiles that map to the same CTA share one
# accumulator (up to 64).  Measured 1.26 * 2^-20 on a B200; a dropped tile is still three orders above this bound.
WG_TOL_BF16_GROUP = 2.0 ** -18
SUM_TOL = 2.0 ** -14         # sum of the isolated groups vs the unmasked batch (many more partial sums)
NAMES = [n for n, _ in O.PARAM_SHAPES]
SIZES_ = [int(np.prod(s)) for _, s in O.PARAM_SHAPES]


# ------------------------------------------------------------------------------------------------ float64 restatement
def bf16r(t):
    """round to nearest even bf16, kept in t's dtype (the kernels' __float2bfloat16_rn)"""
    return t.to(torch.bfloat16).to(t.dtype)


def mlp_grads(p, ep, ed, d_out, rnd=None):
    """mlps.py:221-278 and its backward, written out: raw[Q,4], the parameter gradients of sum(raw * d_out) (state_dict
    names), d gamma(x), d gamma(d), and the magnitudes |dY|^T |X| (weights) / sum |dY| (biases) of every gradient.
    rnd=None: plain arithmetic in the dtype of the inputs.  rnd=bf16r: rounding where the bf16 training kernels round --
    trunk / feature / color_fc weights, both encodings, every stashed activation and every dY image (sigma_out / color_out
    weights stay fp32: CUDA-core heads)."""
    r = rnd or (lambda t: t)
    W = {k: r(v) if k.endswith("weight") and not k.startswith(("sigma_out", "color_out")) else v for k, v in p.items()}
    gx, gd = r(ep), r(ed)
    h, xs, hs = gx, [], []
    for l in range(8):
        x = torch.cat([h, gx], -1) if l == 4 else h
        xs.append(x)
        f = torch.relu(x @ W[f"mlp.{l}.weight"].T + p[f"mlp.{l}.bias"])
        h = r(f)
        hs.append(h)
    sig = f @ p["sigma_out.weight"].T + p["sigma_out.bias"]
    cin = torch.cat([r(h @ W["feature.weight"].T + p["feature.bias"]), gd], -1)
    cf = torch.relu(cin @ W["color_fc.weight"].T + p["color_fc.bias"])
    raw = torch.cat([cf @ p["color_out.weight"].T + p["color_out.bias"], sig], -1)
    cb = r(cf)
    d_rgb, d_sig = d_out[:, :3], d_out[:, 3:4]
    pairs = {"color_out": (d_rgb, cb), "sigma_out": (d_sig, hs[7])}
    dc = r((d_rgb @ p["color_out.weight"]) * (cb > 0))
    pairs["color_fc"] = (dc, cin)
    dfeat = r(dc @ W["color_fc.weight"][:, :256])
    pairs["feature"] = (dfeat, hs[7])
    dy = r((dfeat @ W["feature.weight"] + d_sig @ p["sigma_out.weight"]) * (hs[7] > 0))
    dys = {}
    for l in range(7, -1, -1):
        pairs[f"mlp.{l}"] = (dy, xs[l])
        dys[l] = dy
        if l > 0:
            dy = r((dy @ W[f"mlp.{l}.weight"][:, :256]) * (hs[l - 1] > 0))
    g, mag = {}, {}
    for name, (a, x) in pairs.items():
        g[name + ".weight"], g[name + ".bias"] = a.T @ x, a.sum(0)
        mag[name + ".weight"], mag[name + ".bias"] = a.abs().T @ x.abs(), a.abs().sum(0)
    d_ep = dys[0] @ W["mlp.0.weight"] + dys[4] @ W["mlp.4.weight"][:, 256:]
    d_ed = dc @ W["color_fc.weight"][:, 256:]
    return raw, g, d_ep, d_ed, mag


def flat(d):
    return torch.cat([d[n].reshape(-1) for n in NAMES])


def ray_encodings(o, d, z, rn, vd):
    """The points + encodings step of forward_pass (render_utils.py:211-223), i.e. what nsb_field_fwd_rays feeds the MLP."""
    B, N = z.shape
    zm = z if rn is None else z * rn.reshape(B, 1)
    pts = o[:, None, :] + d[:, None, :] * zm[..., None]
    v = torch.nn.functional.normalize(vd if vd is not None else d, dim=-1)
    return IG.encode(pts.reshape(-1, 3), 10), IG.encode(v[:, None, :].expand_as(pts).reshape(-1, 3), 4)


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


# ------------------------------------------------------------------------------------------------ CPU: pin the restatement
def _cpu_case(Q=300, seed=3):
    rng = np.random.default_rng(seed)
    p = O.init_params(rng, sigma_bias=0.3)
    ep = O.positional_encode(rng.uniform(-4, 4, (Q, 3)).astype(np.float32), 10)
    ed = O.positional_encode(O._normalize(rng.standard_normal((Q, 3)).astype(np.float32)), 4)
    d_out = (rng.standard_normal((Q, 4)) + 0.5).astype(np.float32)
    return p, ep, ed, d_out


def test_restatement_matches_autograd_and_oracle():
    p, ep, ed, d_out = _cpu_case()
    pt = IG.params_t(p, grad=True)
    ept, edt = (torch.tensor(a, dtype=F64, requires_grad=True) for a in (ep, ed))
    dt = torch.tensor(d_out, dtype=F64)
    raw, g, d_ep, d_ed, mag = mlp_grads({k: v.detach() for k, v in pt.items()}, ept.detach(), edt.detach(), dt)
    want = IG.mlp(pt, ept, edt)
    (want * dt).sum().backward()
    assert rel_l2(raw, want.detach()) < 1e-12
    for n in NAMES:
        assert rel_l2(g[n], pt[n].grad) < 1e-12, n
        assert bool((mag[n] >= g[n].abs() * (1 - 1e-12)).all()), n          # a magnitude bounds its sum
    assert rel_l2(d_ep, ept.grad) < 1e-12 and rel_l2(d_ed, edt.grad) < 1e-12
    raw_o, caches = O.mlp_forward(p, ep, ed, keep=True)
    assert rel_l2(raw, torch.tensor(raw_o)) < 1e-6
    assert rel_l2(flat(g), torch.tensor(O.flatten_params(O.mlp_backward(p, caches, d_out)))) < 1e-6


def test_bf16_emulation_matches_tc_emulation():
    """rnd=bf16r against the float32 numpy emulation the bf16 layer tests use, and against the input-gradient emulation of
    test_gpu_input_grads.  Evaluated in float32 it agrees with the former to float32 summation order (the roundings sit at
    the same points); in float64 some values land on the other side of a bf16 rounding than in float32, and those flips
    carry through the chain (measured 2e-4 on raw, 4e-3 on mlp.0.weight)."""
    p, ep, ed, d_out = _cpu_case()
    raw_t, g_t = TC.bf16_emulated_mlp(p, ep, ed, d_out)
    for dtype, bar_raw, bar_g in ((torch.float32, 1e-6, 1e-5), (F64, 1e-3, 1e-2)):
        pt = IG.params_t(p, dtype)
        raw, g, _, _, _ = mlp_grads(pt, *(torch.tensor(a, dtype=dtype) for a in (ep, ed, d_out)), bf16r)
        assert rel_l2(raw, torch.tensor(raw_t)) < bar_raw, (dtype, rel_l2(raw, torch.tensor(raw_t)))
        for n in NAMES:
            assert rel_l2(g[n], torch.tensor(g_t[n])) < bar_g, (dtype, n, rel_l2(g[n], torch.tensor(g_t[n])))
    ept, edt, dt = (torch.tensor(a, dtype=F64) for a in (ep, ed, d_out))
    _, _, d_ep, d_ed, _ = mlp_grads(pt, ept, edt, dt, bf16r)
    e_ep, e_ed = IG.bf16_encoding_grads(pt, ept, edt, dt)
    assert rel_l2(d_ep, e_ep) < 1e-12 and rel_l2(d_ed, e_ed) < 1e-12


def test_ray_encodings_match_oracle():
    rng = np.random.default_rng(6)
    r = O.synthetic_rays(rng, 40)
    z = np.sort(rng.uniform(2.0, 6.0, (40, 24)), -1).astype(np.float32)
    pts = O.ray_points(r["rays_o_marching"], r["rays_d_marching_unit"], z, r["rays_d_marching_norm"])
    vd = O._normalize(r["rays_d_world_unit"])
    want_p = O.positional_encode(pts.reshape(-1, 3), 10)
    want_d = O.positional_encode(np.broadcast_to(vd[:, None, :], pts.shape).reshape(-1, 3), 4)
    t = lambda a: torch.tensor(a, dtype=F64)
    ep, ed = ray_encodings(t(r["rays_o_marching"]), t(r["rays_d_marching_unit"]), t(z), t(r["rays_d_marching_norm"]).reshape(-1),
                           t(r["rays_d_world_unit"]))
    # the oracle works in float32: at the 2^9 frequency its phase error reaches ~1e-4
    assert rel_l2(ep, t(want_p)) < 1e-4 and rel_l2(ed, t(want_d)) < 1e-6


# ------------------------------------------------------------------------------------------------ GPU harness
REPORT = {}


def note(key, value):
    """Keep the largest value measured for `key`; printed when the module finishes."""
    REPORT[key] = max(REPORT.get(key, 0.0), float(value))


@pytest.fixture(scope="module", autouse=True)
def _print_report():
    yield
    if REPORT:
        print("\nmeasured maxima (ratio to bound, or distance):")
        for k in sorted(REPORT):
            print(f"  {k}: {REPORT[k]:.4g}")


class Field:
    """One net's packed weights in one mode, driven through the C ABI."""

    def __init__(self, p, mode):
        from nerf_sandbox_b200 import _lib
        self.lib, self.L = _lib, _lib.lib()
        self.name = mode
        self.mode = {"fp32": _lib.MODE_FP32, "bf16": _lib.MODE_BF16}[mode]
        fl = torch.tensor(O.flatten_params(p), device=DEV)
        self.packed = torch.empty(self.L.nsb_packed_weights_bytes(), dtype=torch.uint8, device=DEV)
        self.lib.check(self.L.nsb_pack_weights(fl.data_ptr(), self.packed.data_ptr(), self.mode, self.lib.stream()), "pack")
        self.p64 = {k: torch.tensor(v, dtype=F64, device=DEV) for k, v in p.items()}
        self.p32 = {k: torch.tensor(v, device=DEV) for k, v in p.items()}
        self.rnd = bf16r if mode == "bf16" else None

    def _ws(self, Q, fill):
        wsb = self.L.nsb_field_workspace_bytes(Q, self.mode, 1)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        if fill is not None:
            ws.fill_(fill)
        return ws, wsb

    def fwd(self, ep, ed, fill=None):
        """training forward with stash; returns raw and the state the backward needs"""
        P, Q = self.lib.ptr, ep.shape[0]
        ws, wsb = self._ws(Q, fill)
        raw = torch.full((Q, 4), float("nan"), device=DEV)
        self.lib.check(self.L.nsb_field_fwd_enc(P(ep), P(ed), P(self.packed), P(raw), P(ws), wsb, Q, self.mode, 1,
                                                self.lib.stream()), "nsb_field_fwd_enc")
        return raw, (ws, wsb, Q)

    def fwd_rays(self, o, d, z, rn, vd, fill=None):
        P, (B, N) = self.lib.ptr, z.shape
        ws, wsb = self._ws(B * N, fill)
        raw = torch.full((B * N, 4), float("nan"), device=DEV)
        self.lib.check(self.L.nsb_field_fwd_rays(P(o), P(d), P(z), P(rn), P(vd), P(self.packed), P(raw), P(ws), wsb, B, N,
                                                 self.mode, 1, self.lib.stream()), "nsb_field_fwd_rays")
        return raw, (ws, wsb, B * N)

    def bwd(self, state, d_raw, grads=True):
        """nsb_field_bwd_ex into a zeroed gradient buffer (it accumulates) and NaN-filled encoding gradients (it overwrites)"""
        P = self.lib.ptr
        ws, wsb, Q = state
        g = torch.zeros(self.lib.N_PARAMS, device=DEV) if grads else None
        dep = torch.full((Q, 63), float("nan"), device=DEV)
        ded = torch.full((Q, 27), float("nan"), device=DEV)
        self.lib.check(self.L.nsb_field_bwd_ex(P(d_raw), P(self.packed), P(g), P(dep), P(ded), P(ws), wsb, Q, self.mode,
                                               self.lib.stream()), "nsb_field_bwd_ex")
        return g, dep, ded

    def rays_bwd(self, dep, ded, o, d, z, rn, vd):
        P, (B, N) = self.lib.ptr, z.shape
        out = [torch.full((B, 3), float("nan"), device=DEV) for _ in range(3)]
        if vd is None:
            out[2] = None
        self.lib.check(self.L.nsb_encode_bwd_rays(P(dep), P(ded), P(o), P(d), P(z), P(rn), P(vd), P(out[0]), P(out[1]),
                                                  P(out[2]), B, N, self.lib.stream()), "nsb_encode_bwd_rays")
        return out

    def alone(self, ep, ed, d_out):
        """the same points as a batch of their own: raw, parameter and encoding gradients"""
        raw, st = self.fwd(ep, ed)
        return (raw,) + self.bwd(st, d_out)


@pytest.fixture(scope="module")
def fields():
    p = O.init_params(np.random.default_rng(2024), sigma_bias=0.3)
    return {m: Field(p, m) for m in ("fp32", "bf16")}


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def inputs(Q, seed):
    """encodings of random points / directions (what the MLP sees) and a d_out with a nonzero mean"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.rand((Q, 3), generator=g, device=DEV) * 8.0 - 4.0
    v = torch.nn.functional.normalize(torch.randn((Q, 3), generator=g, device=DEV), dim=-1)
    d_out = torch.randn((Q, 4), generator=g, device=DEV) + 0.5
    return IG.encode(x, 10).contiguous(), IG.encode(v, 4).contiguous(), d_out


def rows(tiles, Q):
    return torch.cat([torch.arange(t * TILE, min(Q, (t + 1) * TILE), device=DEV) for t in tiles])


def masked(d_out, idx):
    d = torch.zeros_like(d_out)
    d[idx] = d_out[idx]
    return d


def ratio_to_bound(a, b, mag, tol):
    """max over elements of |a - b| / (tol * m), m = max(float64 magnitude, |b|): where a ReLU mask of a near-zero
    pre-activation flips between the kernel and the float64 restatement, the restatement misses that point's term.  An
    element with m = 0 must match exactly (inf otherwise)."""
    m = torch.maximum(mag, b.abs().double()) * tol
    diff = (a.double() - b.double()).abs()
    r = torch.where(m > 0, diff / torch.where(m > 0, m, 1.0), torch.where(diff > 0, math.inf, 0.0))
    return float(r.max())


def assert_rows_only(full, idx, alone, what):
    """encoding gradients of an isolated group: bitwise those of the points alone, exactly zero (and written) elsewhere"""
    assert torch.equal(full[idx], alone), (what, float((full[idx] - alone).abs().max()))
    rest = full.clone()
    rest[idx] = 0
    assert bool((rest == 0).all()), (what, "rows outside the group", int((rest != 0).sum()))


def check_group(F, state, ep, ed, d_out, idx, tag, bitwise, vs_f64, encs=None):
    """The whole-batch backward with d_raw on `idx` only against the same points alone, and (vs_f64) its parameter
    gradients against float64.  Appends (rows, kernel and float64 encoding gradients) to `encs` for a comparison over all
    groups of a size.  Returns the isolated gradient and its magnitudes (for the superposition check)."""
    a_g, a_ep, a_ed = F.bwd(state, masked(d_out, idx))
    _, b_g, b_ep, b_ed = F.alone(ep[idx], ed[idx], d_out[idx])
    assert_rows_only(a_ep, idx, b_ep, tag + " d_enc_pos")
    assert_rows_only(a_ed, idx, b_ed, tag + " d_enc_dir")
    ep64, ed64, do64 = ep[idx].double(), ed[idx].double(), d_out[idx].double()
    _, g_ref, dep_ref, ded_ref, mag = mlp_grads(F.p64, ep64, ed64, do64, F.rnd)
    mag = flat(mag)
    if bitwise:
        assert torch.equal(a_g, b_g), (tag, float((a_g - b_g).abs().max()))
    tol = WG_TOL_BF16_GROUP if F.name == "bf16" and not bitwise else WG_TOL
    r = ratio_to_bound(a_g, b_g, mag, tol)
    note(f"{F.name} {'tile' if bitwise else 'group'} vs alone: ratio to its bound ({tol:.3g} |dY||X|)", r)
    if not bitwise:
        note(f"{F.name} group vs alone not bitwise (1 = differed)", 0.0 if torch.equal(a_g, b_g) else 1.0)
    assert r <= 1.0, (tag, r)
    if vs_f64:
        if F.name == "fp32":
            e = rel_l2(a_g, flat(g_ref))
            note("fp32 group vs float64: flat rel L2", e)
            assert e <= 5e-3, (tag, e)
        else:
            off = 0
            for n, k in zip(NAMES, SIZES_):
                e = rel_l2(a_g[off:off + k], g_ref[n].reshape(-1))
                note("bf16 group vs float64 emulation: worst tensor rel L2", e)
                assert e <= 2e-2, (tag, n, e)
                off += k
        if encs is not None:
            encs.append((idx, a_ep[idx], a_ed[idx], dep_ref, ded_ref))
    return a_g, mag


def check_encodings(F, ep, ed, d_out, encs, tag):
    """Encoding gradients of every group of a size against float64, over all their points together.  They depend on each
    point alone (held bitwise to the points run alone above), so this is a check of the arithmetic, not of the schedule; a
    single group of 1,024 points holds zero to a few ReLU masks that flip between the kernel's and float64's sums, each worth
    ~1e-3 of relative L2 (fp32 mode), which the rule below only averages out over more points.
      fp32 mode: <= max(1e-4, 2 x the distance of the same composition in float32) (test_gpu_input_grads.py's rule);
      bf16 mode: <= 2e-2 against the float64 emulation (measured 0.8-1.5e-2 on single groups of 1,024 points)."""
    if not encs:
        return
    idx = torch.cat([e[0] for e in encs])
    got = [torch.cat([e[1] for e in encs]), torch.cat([e[2] for e in encs])]
    want = [torch.cat([e[3] for e in encs]), torch.cat([e[4] for e in encs])]
    if F.name == "fp32":
        _, _, dep32, ded32, _ = mlp_grads(F.p32, ep[idx], ed[idx], d_out[idx])
        bars = [max(1e-4, 2.0 * rel_l2(f32, w)) for f32, w in zip((dep32, ded32), want)]
    else:
        bars = [2e-2, 2e-2]
    for g, w, bar, what in zip(got, want, bars, ("d_enc_pos", "d_enc_dir")):
        note(f"{F.name} groups vs float64{' emulation' if F.name == 'bf16' else ''}: {what} rel L2 / bar", rel_l2(g, w) / bar)
        assert rel_l2(g, w) <= bar, (tag, what, rel_l2(g, w), bar)


# Sizes, as functions of the SM count S, and the regime each one exercises.
SIZES = {
    "1": lambda S: 1,                            # a single point: one ragged tile, one CTA per wgrad job
    "127": lambda S: 127,                        # one ragged tile, all but one row padding
    "128": lambda S: 128,                        # exactly one full tile
    "129": lambda S: 129,                        # a full tile and a one-point ragged tile (odd tile count: half a dgrad pair)
    "1000": lambda S: 1000,                      # 8 tiles, ragged; still one tile per wgrad CTA
    "12x128+1": lambda S: 12 * TILE + 1,         # 13 tiles: the 13 wgrad jobs want more than S CTAs -> a CTA takes a 2nd tile
    "32S": lambda S: 32 * S,                     # fp32 head_bwd_kernel: exactly one point per warp of its capped grid
    "32S+1": lambda S: 32 * S + 1,               # ... and one warp takes a second point
    "2Sx128": lambda S: 2 * S * TILE,            # dgrad: pairs == S, every CTA pair runs one iteration
    "2Sx128+1": lambda S: 2 * S * TILE + 1,      # dgrad: pairs > S, the CTA pairs iterate; ragged last tile
    "65536": lambda S: 65536,                    # coarse pass of a 1,024-ray step (64 samples)
    "196608": lambda S: 196608,                  # fine pass of a 1,024-ray step (64 + 128 samples)
    "524288": lambda S: 524288,                  # coarse pass of an 8,192-ray step
    "1572864": lambda S: 1572864,                # fine pass of an 8,192-ray step (bf16 only: the fp32 workspace is ~20 GB)
}
CASES = [(m, s) for m in ("fp32", "bf16") for s in SIZES if not (m == "fp32" and s == "1572864")]
FULL_COVER = 512              # up to this many tiles every tile is isolated (in groups); above, a sample


def single_tiles(T, S):
    """first, second, last (the ragged one when Q % 128 != 0), and the tiles around k * S and k * 2S"""
    c = {0, 1, T - 1}
    for step in (S, 2 * S):
        ks = sorted({1, 2, 3, T // step})
        for k in ks:
            c |= {k * step - 1, k * step}
    return sorted(t for t in c if 0 <= t < T)


def groups_of_eight(T):
    """t = j mod T/8 (8 spread tiles per group); the remainder of T / 8 tiles forms one more group.  Every tile is in exactly
    one group up to FULL_COVER tiles; above, a sample of the groups."""
    if T < 8:
        return [list(range(T))], True
    stride = T // 8
    js = range(stride) if T <= FULL_COVER else sorted({0, 1, stride // 2, stride - 1})
    gs = [[j + i * stride for i in range(8)] for j in js]
    if 8 * stride < T:
        gs.append(list(range(8 * stride, T)))
    return gs, T <= FULL_COVER


@pytest.mark.gpu
@pytest.mark.parametrize("mode,size", CASES)
def test_per_point_independence(fields, mode, size):
    """raw, d gamma(x) and d gamma(d) of the whole batch equal those of the same points run in chunks of 128, 1,000
    (rows land at other in-tile positions) and 37,889, bit for bit: each row is the same products on the same operands."""
    F = fields[mode]
    Q = SIZES[size](num_sms())
    ep, ed, d_out = inputs(Q, 1000 + Q)
    raw, st = F.fwd(ep, ed)
    _, dep, ded = F.bwd(st, d_out, grads=False)
    assert bool(torch.isfinite(raw).all() and torch.isfinite(dep).all() and torch.isfinite(ded).all())
    for c in (128, 1000, 37889):
        n = math.ceil(Q / c)
        picks = range(n) if n <= 256 else sorted({0, 1, n // 3, n // 2, n - 2, n - 1} | set(range(0, n, n // 48)))
        for i in picks:
            s, e = i * c, min(Q, (i + 1) * c)
            r2, st2 = F.fwd(ep[s:e], ed[s:e])
            _, dep2, ded2 = F.bwd(st2, d_out[s:e], grads=False)
            for got, want, what in ((r2, raw[s:e], "raw"), (dep2, dep[s:e], "d_enc_pos"), (ded2, ded[s:e], "d_enc_dir")):
                d = float((got - want).abs().max())
                note(f"{mode} per-point chunked vs whole: max |diff| of {what}", d)
                assert torch.equal(got, want), (c, i, what, d)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,size", CASES)
def test_tile_isolation(fields, mode, size):
    """Single tiles and groups of 8 spread tiles against the same points alone (bitwise for a single tile in bf16
    mode), groups of >= 8 tiles against float64, and the isolated groups summing to the unmasked gradient."""
    F = fields[mode]
    S = num_sms()
    Q = SIZES[size](S)
    T = math.ceil(Q / TILE)
    ep, ed, d_out = inputs(Q, 2000 + Q)
    _, st = F.fwd(ep, ed)
    for t in single_tiles(T, S):
        # one tile in bf16 mode: zero products elsewhere and one flushing CTA per job leave nothing order-dependent
        check_group(F, st, ep, ed, d_out, rows([t], Q), f"{size} tile {t}/{T}", bitwise=mode == "bf16", vs_f64=False)
    gs, cover = groups_of_eight(T)
    total, mags = torch.zeros(F.lib.N_PARAMS, device=DEV), torch.zeros(F.lib.N_PARAMS, dtype=F64, device=DEV)
    encs = []
    for grp in gs:
        a_g, mag = check_group(F, st, ep, ed, d_out, rows(grp, Q), f"{size} group {grp[:3]}../{T}", bitwise=False,
                               vs_f64=len(grp) >= 8, encs=encs)
        total += a_g
        mags += mag
    check_encodings(F, ep, ed, d_out, encs, size)
    if cover:
        # superposition: a sanity check of the bookkeeping above (the isolation checks are the detector)
        full, _, _ = F.bwd(st, d_out)
        r = ratio_to_bound(total, full, mags, SUM_TOL)
        note(f"{mode} superposition: ratio to 2^-14 |dY||X|", r)
        assert r <= 1.0, r


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("k", ["12", "2S"])
@pytest.mark.parametrize("r", [1, 5, 127])
def test_ragged_tail_poisoned_and_padded(fields, mode, k, r):
    """Q = 128 k + r.  The last (ragged) tile isolated: a workspace filled with 0xFF (NaN bit patterns) and one filled with
    0x00 give the same raw, encoding and parameter gradients (bitwise in bf16 mode; in fp32 mode head_bwd_kernel and the split-K
    flush add a tile's partials with float atomics in no fixed order, so there the parameter gradients are held to the
    isolation bound); and padding the batch to a whole tile with extra points whose d_out is zero changes nothing."""
    F = fields[mode]
    kk = 12 if k == "12" else 2 * num_sms()
    Q = TILE * kk + r
    ep, ed, d_out = inputs(Q + TILE - r, 3000 + Q)
    epQ, edQ, doQ = ep[:Q], ed[:Q], d_out[:Q]
    idx = rows([kk], Q)
    res = []
    for fill in (0xFF, 0x00):
        raw, st = F.fwd(epQ, edQ, fill=fill)
        g, dep, ded = F.bwd(st, masked(doQ, idx))
        assert bool(torch.isfinite(raw).all() and torch.isfinite(g).all() and torch.isfinite(dep).all() and torch.isfinite(ded).all())
        res.append((raw, g, dep, ded))
    (raw0, g0, dep0, ded0), (raw1, g1, dep1, ded1) = res
    assert torch.equal(raw0, raw1) and torch.equal(dep0, dep1) and torch.equal(ded0, ded1)
    _, _, _, _, mag = mlp_grads(F.p64, epQ[idx].double(), edQ[idx].double(), doQ[idx].double(), F.rnd)
    mag = flat(mag)
    if mode == "bf16":
        assert torch.equal(g0, g1), float((g0 - g1).abs().max())
    rp = ratio_to_bound(g0, g1, mag, WG_TOL)
    note(f"{mode} ragged tail poisoned vs zeroed: ratio to 2^-20 |dY||X|", rp)
    assert rp <= 1.0, rp
    # padded to the next multiple of 128 with points that carry no gradient
    dpad = torch.zeros_like(d_out)
    dpad[idx] = d_out[idx]
    _, stp = F.fwd(ep, ed, fill=0xFF)
    gp, depp, dedp = F.bwd(stp, dpad)
    assert torch.equal(depp[:Q], dep1) and torch.equal(dedp[:Q], ded1)
    assert bool((depp[Q:] == 0).all() and (dedp[Q:] == 0).all())
    rq = ratio_to_bound(gp, g1, mag, WG_TOL)
    note(f"{mode} ragged tail padded vs not: ratio to 2^-20 |dY||X|", rq)
    assert rq <= 1.0, rq


RAY_CASES = [(m, B, N) for m in ("fp32", "bf16") for B, N in ((1024, 64), (1024, 192), (333, 200), (37, 33), (5, 1))] + \
    [("bf16", 8192, 192)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,B,N", RAY_CASES)
def test_ray_entry_point(fields, mode, B, N):
    """nsb_field_fwd_rays -> nsb_field_bwd_ex with encoding outputs -> nsb_encode_bwd_rays: per-ray gradients do not depend
    on how the rays are batched, a d_raw on one ray gives every other ray exactly zero, and a group of rays matches the
    float64 composition (the fp32 mode) or its bf16 emulation (the bf16 mode)."""
    F = fields[mode]
    case = IG.make_case(500 + B + N, B, N, viewdirs=(B, N) != (333, 200))     # (333, 200): view-direction term into rays_d
    t = {k: (torch.tensor(case[k], device=DEV) if case[k] is not None else None) for k in ("o", "d", "z", "rn", "vd")}
    o, d, z, rn, vd = (t[k] for k in ("o", "d", "z", "rn", "vd"))
    d_out = torch.randn((B * N, 4), generator=torch.Generator(device=DEV).manual_seed(B * N), device=DEV) + 0.5

    def run(s, e, d_raw):
        sl = lambda a: None if a is None else a[s:e]
        raw, st = F.fwd_rays(sl(o), sl(d), sl(z), sl(rn), sl(vd))
        g, dep, ded = F.bwd(st, d_raw)
        return raw, g, F.rays_bwd(dep, ded, sl(o), sl(d), sl(z), sl(rn), sl(vd))

    raw, _, full = run(0, B, d_out)
    assert bool(torch.isfinite(raw).all()) and all(bool(torch.isfinite(x).all()) for x in full if x is not None)
    for c in (1, 5, 97):
        n = math.ceil(B / c)
        for i in (range(n) if n <= 64 else sorted({0, n // 2, n - 1} | set(range(0, n, n // 32)))):
            s, e = i * c, min(B, (i + 1) * c)
            r2, _, part = run(s, e, d_out[s * N:e * N].contiguous())
            assert torch.equal(r2, raw[s * N:e * N]), (c, i)
            for a, b in zip(part, full):
                if a is not None:
                    assert torch.equal(a, b[s:e]), (c, i, float((a - b[s:e]).abs().max()))
    # one ray isolated: exactly zero for every other ray, its own gradients bitwise those of the unmasked batch
    for ray in sorted({0, B // 2, B - 1}):
        idx = torch.arange(ray * N, (ray + 1) * N, device=DEV)
        _, _, iso = run(0, B, masked(d_out, idx))
        for a, b in zip(iso, full):
            if a is not None:
                assert torch.equal(a[ray], b[ray])
                rest = a.clone()
                rest[ray] = 0
                assert bool((rest == 0).all()), ray
    # a group of rays (>= 1024 points where the batch has them) against float64
    n_rays = min(B, math.ceil(1024 / N))
    R = torch.linspace(0, B - 1, n_rays, device=DEV).round().long().unique()
    idx = (R[:, None] * N + torch.arange(N, device=DEV)).reshape(-1)
    _, g, iso = run(0, B, masked(d_out, idx))
    keep = torch.zeros(B, dtype=torch.bool, device=DEV)
    keep[R] = True
    for a in iso:
        if a is not None:
            assert bool((a[~keep] == 0).all())

    def ref(dtype, rnd):
        pr = F.p64 if dtype == F64 else F.p32
        rt = {k: None if t[k] is None else t[k][R].to(dtype).requires_grad_(k in ("o", "d", "vd")) for k in t}
        ep, ed = ray_encodings(rt["o"], rt["d"], rt["z"], rt["rn"], rt["vd"])
        _, gr, dep, ded, _ = mlp_grads(pr, ep.detach(), ed.detach(), d_out[idx].to(dtype), rnd)
        ins = [rt[k] for k in ("o", "d", "vd") if rt[k] is not None]
        return gr, torch.autograd.grad((ep * dep).sum() + (ed * ded).sum(), ins)

    g64, r64 = ref(F64, F.rnd)
    got_rays = [a[R] for a in iso if a is not None]
    if mode == "fp32":
        e = rel_l2(g, flat(g64))
        note("fp32 rays group vs float64: flat rel L2", e)
        assert e <= 5e-3, e
        _, r32 = ref(torch.float32, None)
        for a, w, w32 in zip(got_rays, r64, r32):
            bar = max(1e-3, 2.0 * rel_l2(w32, w))
            note("fp32 rays group vs float64: ray grad rel L2 / bar", rel_l2(a, w) / bar)
            assert rel_l2(a, w) <= bar, (rel_l2(a, w), bar)
    else:
        # measured 2e-2 - 4.5e-2 (mlp.0.weight) on groups of 16 - 37 rays, and 8e-3 over all 1,024 rays x 64 samples: the
        # samples of one ray are correlated, so a group averages the bf16 rounding noise less than as many random points do
        bar = 6e-2 if len(idx) >= TILE else 0.15                 # 5 points: one flipped ReLU mask is already a few %
        off = 0
        for n, k in zip(NAMES, SIZES_):
            e = rel_l2(g[off:off + k], g64[n].reshape(-1))
            note("bf16 rays group vs float64 emulation: worst tensor rel L2", e)
            assert e <= bar, (n, e)
            off += k
        # the ray gradients weight d gamma(x) by up to 2^9 (highest frequency first), where the emulation's d gamma(x) is
        # noisiest: measured up to 7.0e-2 on groups of 16 - 37 rays (test_gpu_input_grads.py: 0.15 against plain float64)
        for a, w in zip(got_rays, r64):
            note("bf16 rays group vs float64 emulation: ray grad rel L2", rel_l2(a, w))
            assert rel_l2(a, w) <= 0.15, rel_l2(a, w)
