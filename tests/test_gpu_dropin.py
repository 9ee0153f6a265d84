"""The drop-in seam, driven by the REFERENCE'S OWN code (oracle/_ref = the unmodified reference package, vendored by
__graft_entry__.build()): after ``install()`` the reference's ``Trainer._train_step`` and its whole
``train_nerf.py --vanilla`` entry point run on the libnsb kernels.

* fp32 mode: the reference's unbound ``_train_step`` (train/trainer.py:876-1013) + backward + torch Adam must reproduce
  tests/golden/train_step.npz -- the outputs of the same reference function on its own PyTorch path -- to 1e-4.
* bf16 mode: the reference CLI (scripts/train_nerf.py main body) trains a tiny synthetic Blender scene end to end on the
  tensor-core path: constructor probes (log_nerf_arch, enable_debug, dump_run_debug's 8x8 forward probe and (4,63)
  sample_pdf case, utils/debug_utils.py:136-148, :322-329), sampler, AMP/GradScaler loop, validation render, checkpoint.
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def N(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope="module")
def ref():
    from baseline import ref_runner
    if not ref_runner.available():
        pytest.skip("oracle/_ref holds no reference (vendored by __graft_entry__.build() from NSB_REFERENCE_SRC, else BASELINE.json's reference_path)")
    TR, RU = ref_runner.import_reference()
    yield ref_runner, TR, RU
    from nerf_sandbox_b200.install import uninstall
    uninstall()


@pytest.mark.parametrize("fuse", [False, True])
def test_reference_train_step_through_install_matches_golden_fp32(ref, fuse):
    """fuse=False: the reference's own _train_step body on the rebound callables.  fuse=True (install's default): the same
    method replaced by the fused step (one library call), behind the same contract."""
    ref_runner, TR, RU = ref
    from nerf_sandbox_b200 import _hooks, _lib
    from nerf_sandbox_b200.install import install
    from oracle import nerf_oracle as O
    import nerf_sandbox_b200 as nsb
    install(mode="fp32", fuse_train_step=fuse)
    assert hasattr(TR.Trainer._train_step, "_nsb_original") == fuse
    assert TR.NeRF is nsb.NeRF and TR.nerf_forward_pass is nsb.nerf_forward_pass and TR.sample_pdf is nsb.sample_pdf
    g = golden("train_step")
    B, nc, nf = int(g["B"]), int(g["nc"]), int(g["nf"])
    dev = torch.device("cuda", 0)
    nets = []
    for seed in (int(g["seed_c"]), int(g["seed_f"])):
        p = O.init_params(np.random.default_rng(seed), sigma_bias=float(g["sigma_bias"]))
        net = TR.NeRF(63, 27, 8, 256, skip_pos=4, sigma_activation="relu")          # exactly trainer.py:326-341: no mode argument
        assert net.mode == _lib.MODE_FP32
        net.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
        nets.append(net.to(dev))
    pos_enc, dir_enc = TR.get_vanilla_nerf_encoders()
    ns = ref_runner.make_namespace(TR, dev, nets[0], nets[1], pos_enc.to(dev), dir_enc.to(dev), nc=nc, nf=nf)
    batch = {k: T(g[k]) for k in ("rays_o_marching", "rays_d_marching_unit", "rays_d_marching_norm", "rays_d_world_unit", "rgb")}
    # identical draws: the inline stratified sampler calls torch.rand_like (trainer.py:907); the resampler and the sigma
    # noise are drawn inside our kernels unless the providers hand them explicit tensors
    normals = [g["noise_c"], g["noise_f"]]
    _hooks.normal = lambda n, device: T(normals.pop(0)).reshape(-1)[:n]
    _hooks.uniform = lambda b, n, device: T(g["u_fine"]).reshape(b, n)
    _hooks.jitter = lambda b, n, device: T(g["U"]).reshape(b, n)              # (the fused step's stratified draws)
    launches = _lib.launch_count()
    orig = torch.rand_like
    torch.rand_like = lambda x, *a, **k: T(g["U"]).reshape(x.shape).to(x.dtype)
    try:
        out = TR.Trainer._train_step(ns, batch)
    finally:
        torch.rand_like = orig
        _hooks.normal = _hooks.uniform = _hooks.jitter = None
    assert not normals, "both passes must have consumed their noise"
    assert _lib.launch_count() > launches
    assert abs(float(out["loss"].detach()) - float(g["loss"])) <= 1e-4 * abs(float(g["loss"]))
    assert abs(float(out["psnr"]) - float(g["psnr"])) <= 1e-3
    np.testing.assert_allclose(N(out["comp_c"]), g["comp_c"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(N(out["comp_f"]), g["comp_f"], rtol=1e-4, atol=1e-6)
    out["loss"].backward()                                                            # trainer.py:717
    idx = g["grad_idx"]
    for tag, net in (("c", nets[0]), ("f", nets[1])):
        flat = N(torch.cat([p.grad.reshape(-1) for p in net.parameters()]))
        want = g[f"grad_samples_{tag}"]
        assert np.abs(flat[idx] - want).max() <= 2e-4 * np.abs(want).max() + 1e-9
        norms = np.array([float(p.grad.norm()) for p in net.parameters()])
        np.testing.assert_allclose(norms, g[f"grad_norms_{tag}"], rtol=5e-3, atol=1e-9)
    opt = torch.optim.Adam(list(nets[0].parameters()) + list(nets[1].parameters()), lr=5e-4)      # trainer.py:383-386
    opt.step()
    for tag, net in (("c", nets[0]), ("f", nets[1])):
        flat = N(torch.cat([p.reshape(-1) for p in net.parameters()]))
        # Adam's first step is lr * g / (|g| + eps): compare where |g| is well above the eps = 1e-8 knee (below it, gradient
        # differences of 1e-9 -- fp32 summation order -- move the step by a sizeable fraction of lr)
        well = np.abs(g[f"grad_samples_{tag}"]) > 1e-6
        assert well.mean() > 0.8
        np.testing.assert_allclose(flat[idx][well], g[f"adam_{tag}"][well], rtol=0, atol=2e-6)
        assert np.abs(flat[idx] - g[f"adam_{tag}"]).max() <= 1.001e-3


def _tiny_blender_scene(root, H=16, n_train=4):
    from PIL import Image
    rng = np.random.default_rng(0)

    def pose(th, ph):
        c = 4.0311 * np.array([np.cos(ph) * np.cos(th), np.cos(ph) * np.sin(th), np.sin(ph)])
        f = -c / np.linalg.norm(c); r = np.cross(f, [0, 0, 1.0]); r /= np.linalg.norm(r); u = np.cross(r, f)
        M = np.eye(4); M[:3, 0], M[:3, 1], M[:3, 2], M[:3, 3] = r, u, -f, c
        return M
    for split, n in (("train", n_train), ("val", 2), ("test", 2)):
        os.makedirs(os.path.join(root, split), exist_ok=True)
        frames = []
        for i in range(n):
            img = (rng.uniform(0, 1, (H, H, 4)) * 255).astype(np.uint8)
            img[..., 3] = 255 * (rng.uniform(size=(H, H)) > 0.3)
            Image.fromarray(img, "RGBA").save(os.path.join(root, split, f"r_{i}.png"))
            frames.append({"file_path": f"./{split}/r_{i}", "transform_matrix": pose(0.7 * i + 0.1, 0.5).tolist()})
        json.dump({"camera_angle_x": 0.6911112, "frames": frames}, open(os.path.join(root, f"transforms_{split}.json"), "w"))


def test_reference_cli_vanilla_trains_on_tensor_cores(ref, tmp_path, capsys):
    ref_runner, TR, RU = ref
    from nerf_sandbox_b200 import _lib
    from nerf_sandbox_b200.install import install
    import nerf_sandbox_b200 as nsb
    install(mode="bf16")                                          # default: fused Trainer._train_step
    assert hasattr(TR.Trainer._train_step, "_nsb_original")
    from nerf_sandbox.source.scripts import train_nerf as CLI
    scene, out_dir = str(tmp_path / "scene"), str(tmp_path / "out")
    _tiny_blender_scene(scene)
    argv = ["--data_root", scene, "--out_dir", out_dir, "--vanilla", "--data_kind", "blender", "--max_steps", "12", "--device", "cuda",
            "--log_every", "4", "--val_every", "6", "--ckpt_every", "12", "--eval_chunk", "100"]
    # the body of scripts/train_nerf.py main() (:383-419), so the trainer object can be inspected afterwards
    cfg = CLI.make_cfg_from_args(CLI.build_argparser().parse_args(argv))
    cfg = CLI.apply_vanilla_profile(cfg)
    cfg = CLI.apply_path_defaults_from_data_kind(cfg=cfg, data_kind=cfg.data_kind)
    os.makedirs(out_dir, exist_ok=True)
    before = _lib.launch_count()
    trainer = CLI.Trainer(cfg)
    assert isinstance(trainer.nerf_c, nsb.NeRF) and trainer.nerf_c.mode == _lib.MODE_BF16 and trainer.nerf_f.mode == _lib.MODE_BF16
    assert trainer.amp is True                                  # the reference's CUDA default: autocast + GradScaler around our ops
    p0 = torch.cat([p.detach().reshape(-1).clone() for p in trainer.nerf_f.parameters()])
    trainer.train()
    torch.cuda.synchronize()
    p1 = torch.cat([p.detach().reshape(-1) for p in trainer.nerf_f.parameters()])
    assert torch.isfinite(p1).all() and float((p1 - p0).abs().max()) > 0        # the optimiser moved the fine net
    assert _lib.launch_count() - before > 12 * 10                               # ... through libnsb kernels
    assert trainer.__dict__.get("_nsb_engine") not in (None, False)             # ... and the fused step engine was used
    dbg = json.load(open(os.path.join(out_dir, "run_debug.json")))
    assert "error" not in dbg["forward_probe"] and "error" not in dbg["hier_sampling"], dbg
    assert abs(dbg["forward_probe"]["weights_sum_minus_acc_maxabs"]) < 1e-4
    assert dbg["hier_sampling"]["zf_shape"] == [4, 32]
    ckpt = os.path.join(out_dir, "checkpoints", "ckpt_0000012.pt")
    assert os.path.isfile(ckpt)
    pngs = [f for r, _, fs in os.walk(out_dir) for f in fs if f.endswith(".png")]
    assert len(pngs) >= 3                                        # rgb / opacity / depth of the validation frame
    # the reference's checkpoint loads into the fast-path trainer (torch Adam state -> flat m / v) and back
    obj = torch.load(ckpt, map_location="cuda", weights_only=False)
    vt = nsb.VanillaTrainer("cuda", mode="bf16")
    vt.load_state_dict(obj)
    assert vt.adam_t == 12 and vt.global_step == 12
    np.testing.assert_array_equal(N(vt.nerf_f.flat_params()), N(p1))
    st = obj["opt"]["state"]
    np.testing.assert_array_equal(N(vt.nerf_c.unflatten(vt.m_c)[0]), N(st[0]["exp_avg"]))
    np.testing.assert_array_equal(N(vt.nerf_f.unflatten(vt.v_f)[3]), N(st[24 + 3]["exp_avg_sq"]))
    opt = torch.optim.Adam(vt.parameters(), lr=5e-4)
    opt.load_state_dict(vt.state_dict()["opt"])                  # and our checkpoint is a valid torch Adam state
    assert float(opt.state_dict()["state"][47]["step"]) == 12.0
