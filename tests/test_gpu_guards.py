"""Out-of-bounds hygiene of the round-2 kernels without a sanitizer (closed on this pool): every output buffer sits between two
guard zones of a sentinel value, sizes are ragged on purpose, and the values are checked against torch restatements."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
SENT = 12345.678


def guarded(shape, pad=4096):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * pad,), SENT, device=DEV, dtype=torch.float32)
    return buf, buf[pad:pad + n].view(*shape), pad


def assert_guards(buf, pad):
    assert bool((buf[:pad] == SENT).all()) and bool((buf[-pad:] == SENT).all()), "kernel wrote outside its output"


def _composite_ref(raw, z, rn, noise, flags_white=True, inf_last=True):
    r = raw.double()
    rgb = torch.sigmoid(r[..., :3]).requires_grad_()
    pre = (r[..., 3] + noise.double()).requires_grad_()
    sig = torch.relu(pre)
    zz = z.double()
    last = torch.full_like(zz[:, :1], 1e10 if inf_last else 0.0)
    delta = torch.cat([zz[:, 1:] - zz[:, :-1], last], -1) * rn.double()[:, None]
    alpha = 1 - torch.exp(-(sig * delta).clamp(0, 60))
    T = torch.cumprod(torch.cat([torch.ones_like(zz[:, :1]), 1 - alpha + 1e-10], -1), -1)[:, :-1]
    w = T * alpha
    acc = w.sum(-1).clamp(0, 1)
    comp = ((w[..., None] * rgb).sum(1) + ((1 - acc)[:, None] if flags_white else 0)).clamp(0, 1)
    return comp, w, rgb, pre


@pytest.mark.parametrize("N", [1, 31, 37, 64, 100, 192, 255, 256, 257, 300])
def test_raw_compositor_ragged_sizes_with_guards(N):
    """N <= 192 runs the one-warp run-layout kernels, 193..300 the multi-warp ones (partial runs when N is not a multiple of 32);
    the strided kernels (N > 1024) are covered by test_gpu_parity.py::test_compositor_ragged_and_long_rays."""
    from nerf_sandbox_b200 import _lib
    L = _lib.lib(); st = _lib.stream()
    B = 37
    g = torch.Generator(device=DEV); g.manual_seed(N)
    raw = torch.randn(B * N, 4, device=DEV, generator=g); raw[:, 3] = raw[:, 3] * 2 + 0.5
    z = torch.sort(torch.rand(B, N, device=DEV, generator=g) * 4 + 2, -1).values.contiguous()
    rn = torch.rand(B, device=DEV, generator=g) * 0.1 + 1.0
    noise = torch.randn(B * N, device=DEV, generator=g)
    cbuf, comp, p1 = guarded((B, 3)); wbuf, w, p2 = guarded((B, N)); abuf, acc, p3 = guarded((B,)); dbuf, dep, p4 = guarded((B,))
    _lib.check(L.nsb_composite_raw_fwd(_lib.ptr(raw), _lib.ptr(noise), 1.0, _lib.ptr(z), _lib.ptr(rn), _lib.ptr(comp), _lib.ptr(w), _lib.ptr(acc),
                                       _lib.ptr(dep), B, N, 7, 1, 0, st))
    gc = torch.randn(B, 3, device=DEV, generator=g)
    rbuf, d_raw, p5 = guarded((B * N, 4))
    _lib.check(L.nsb_composite_raw_bwd(_lib.ptr(raw), _lib.ptr(noise), 1.0, _lib.ptr(z), _lib.ptr(rn), _lib.ptr(gc), _lib.ptr(d_raw), B, N, 7, 1, 0, st))
    torch.cuda.synchronize()
    for b, p in ((cbuf, p1), (wbuf, p2), (abuf, p3), (dbuf, p4), (rbuf, p5)):
        assert_guards(b, p)
    c_ref, w_ref, rgb, pre = _composite_ref(raw.view(B, N, 4), z, rn, noise.view(B, N))
    (c_ref * gc.double()).sum().backward()
    assert float((comp.double() - c_ref.detach()).abs().max()) <= 2e-6 and float((w.double() - w_ref.detach()).abs().max()) <= 2e-6
    d = d_raw.view(B, N, 4).double()
    want_rgb = rgb.grad * (rgb * (1 - rgb)).detach()
    assert float((d[..., :3] - want_rgb).norm() / want_rgb.norm().clamp_min(1e-30)) <= 1e-5
    assert float((d[..., 3] - pre.grad).norm() / pre.grad.norm().clamp_min(1e-30)) <= 1e-5
    # in-kernel noise: forward and backward regenerate the same draws (the backward of the SAME noise is what training uses)
    _lib.check(L.nsb_composite_raw_fwd(_lib.ptr(raw), None, 1.0, _lib.ptr(z), _lib.ptr(rn), _lib.ptr(comp), _lib.ptr(w), None, None, B, N, 7, 9, 3, st))
    _lib.check(L.nsb_composite_raw_bwd(_lib.ptr(raw), None, 1.0, _lib.ptr(z), _lib.ptr(rn), _lib.ptr(gc), _lib.ptr(d_raw), B, N, 7, 9, 3, st))
    torch.cuda.synchronize()
    assert_guards(wbuf, p2); assert_guards(rbuf, p5)
    assert bool(torch.isfinite(d_raw).all()) and bool(torch.isfinite(comp).all())


@pytest.mark.parametrize("nc,nf", [(64, 128), (32, 64), (256, 512), (128, 64), (40, 70), (64, 100), (2, 1)])
def test_resample_merge_shapes_with_guards(nc, nf):
    """Multiples of 32 take the register-resident kernel, everything else the general one; both for deterministic and
    in-kernel draws.  The merged row must be exactly sort(cat(zc, z_fine)) of the kernel's own fine samples."""
    from nerf_sandbox_b200 import _lib
    L = _lib.lib(); st = _lib.stream()
    B = 53
    g = torch.Generator(device=DEV); g.manual_seed(nc * 1000 + nf)
    zc = torch.sort(torch.rand(B, nc, device=DEV, generator=g) * 4 + 2, -1).values.contiguous()
    wc = torch.rand(B, nc, device=DEV, generator=g) ** 3
    for det in (1, 0):
        abuf, z_all, p1 = guarded((B, nc + nf)); fbuf, z_f, p2 = guarded((B, nf))
        _lib.check(L.nsb_resample_merge(_lib.ptr(zc), _lib.ptr(wc), None, _lib.ptr(z_all), _lib.ptr(z_f), B, nc, nf, det, 5, 2, st))
        torch.cuda.synchronize()
        assert_guards(abuf, p1); assert_guards(fbuf, p2)
        za, zf = z_all.cpu().numpy(), z_f.cpu().numpy()
        assert np.isfinite(za).all() and (np.diff(za, axis=1) >= 0).all()
        assert np.array_equal(np.sort(np.concatenate([zc.cpu().numpy(), zf], 1), axis=1), za)
        if det:        # against torch's own sample_pdf restatement on the same inputs (deterministic u)
            mids = 0.5 * (zc[:, 1:] + zc[:, :-1]); wb = 0.5 * (wc[:, 1:] + wc[:, :-1]) + 1e-5
            if nc > 2:
                edges = torch.cat([mids[:, :1] - 0.5 * (mids[:, 1:2] - mids[:, :1]), 0.5 * (mids[:, 1:] + mids[:, :-1]),
                                   mids[:, -1:] + 0.5 * (mids[:, -1:] - mids[:, -2:-1])], -1)
                pdf = (wb + 1e-5).clamp_min(0); pdf = pdf / pdf.sum(-1, keepdim=True)
                cdf = torch.cat([torch.zeros_like(pdf[:, :1]), torch.cumsum(pdf, -1)], -1)
                u = torch.linspace(0, 1, nf, device=DEV).expand(B, nf).contiguous()
                inds = torch.searchsorted(cdf, u, right=True)
                below, above = (inds - 1).clamp(0, nc - 1), inds.clamp(1, nc - 1)
                c_lo, c_hi = torch.gather(cdf, 1, below), torch.gather(cdf, 1, above)
                den = torch.where(c_hi - c_lo < 1e-5, torch.ones_like(c_lo), c_hi - c_lo)
                ref = torch.gather(edges, 1, below) + (u - c_lo) / den * (torch.gather(edges, 1, above) - torch.gather(edges, 1, below))
                ok = (z_f - ref).abs() <= 2e-5
                assert float(ok.float().mean()) > 0.99              # (index flips at CDF ties with u = 1.0 aside)


def test_split_forward_ragged_sizes_matches_training_forward():
    """fp32 mode: the no-grad forward (fp16-split tensor-core kernel) against the grad-enabled forward (bf16-split layer GEMMs)
    on ragged point counts, raw outputs within 1e-4 relative + 2e-5 absolute."""
    import nerf_sandbox_b200 as nsb
    from oracle import nerf_oracle as O
    net = nsb.NeRF(63, 27, mode="fp32").to(DEV)
    with torch.no_grad():
        net.sigma_out.bias.fill_(0.3)
    rng = np.random.default_rng(0)
    for Q in (1, 5, 127, 128, 129, 1000, 128 * 9):
        ep = torch.from_numpy(O.positional_encode(rng.uniform(-4, 4, (Q, 3)).astype(np.float32), 10)).to(DEV)
        ed = torch.from_numpy(O.positional_encode(O._normalize(rng.standard_normal((Q, 3)).astype(np.float32)), 4)).to(DEV)
        with torch.no_grad():
            a = net(ep, ed)
        b = net(ep, ed).detach()
        assert a.shape == (Q, 4) and bool(torch.isfinite(a).all())
        assert bool(((a - b).abs() <= 1e-4 * b.abs() + 2e-5).all()), (Q, float((a - b).abs().max()))
