"""CPU-side checks of the test/bench helpers that the GPU box relies on: the piecewise oracle step used by the full-size
parity tests, the vendored reference arm, the package's mode default and checkpoint format helpers."""
import importlib.util
import os
import sys

import numpy as np
import pytest

from oracle import nerf_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fullsize_module():
    spec = importlib.util.spec_from_file_location("fullsize_helpers", os.path.join(ROOT, "tests", "test_gpu_fullsize.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_oracle_step_in_pieces_equals_whole_batch():
    """Loss and gradients of the 8,192-ray parity test are assembled from 1024-ray oracle pieces: exact for a mean-squared error."""
    fs = _fullsize_module()
    rng = np.random.default_rng(3)
    B, nc, nf = 48, 16, 24
    batch = O.synthetic_rays(rng, B); draws = fs._draws(rng, B, nc, nf)
    pc = O.init_params(np.random.default_rng(1), 0.4); pf = O.init_params(np.random.default_rng(2), 0.4)
    whole = O.train_step(pc, pf, batch, near=2.0, far=6.0, nc=nc, nf=nf, **draws)
    pieces = fs._oracle_step_in_pieces(pc, pf, batch, draws, near=2.0, far=6.0, nc=nc, nf=nf, piece=16)
    assert abs(float(whole["loss"]) - pieces["loss"]) <= 1e-6 * float(whole["loss"])
    assert abs(float(whole["psnr"]) - pieces["psnr"]) <= 1e-5
    np.testing.assert_allclose(whole["comp_f"], pieces["comp_f"], rtol=2e-6, atol=2e-7)       # (BLAS blocks differ with the row count)
    np.testing.assert_allclose(whole["comp_c"], pieces["comp_c"], rtol=2e-6, atol=2e-7)
    for tag in ("c", "f"):
        gw = O.flatten_params(whole[f"grads_{tag}"]).astype(np.float64)
        assert np.linalg.norm(gw - pieces[f"grads_{tag}"]) <= 1e-5 * np.linalg.norm(gw)


def test_scene_ground_truth_is_a_valid_image():
    fs = _fullsize_module()
    r = O.synthetic_rays(np.random.default_rng(0), 64)
    gt = fs.scene_gt(r["rays_o_marching"], r["rays_d_marching_unit"], r["rays_d_marching_norm"])
    assert gt.shape == (64, 3) and np.isfinite(gt).all() and gt.min() >= 0 and gt.max() <= 1 and gt.std() > 0.05


def test_reference_arm_runs_the_vendored_reference():
    """bench.py --impl reference / cpu_baseline: the reference's own Trainer._train_step + backward + Adam (oracle/_ref)."""
    from baseline import ref_runner
    if not ref_runner.available():
        pytest.skip("oracle/_ref holds no reference (vendored by __graft_entry__.build() from NSB_REFERENCE_SRC, else BASELINE.json's reference_path)")
    rng = np.random.default_rng(0)
    step, info = ref_runner.make_cpu_step(lambda i: O.synthetic_rays(rng, 32), nc=16, nf=16, threads=2)
    l0 = step(); l1 = step()
    assert np.isfinite([l0, l1]).all() and info["threads"] == 2
    # unmodified: the vendored files are byte-identical to the reference checkout when that is present
    src = os.path.join(ref_runner.reference_checkout(), "nerf_sandbox", "source", "train", "trainer.py")
    if os.path.isfile(src):
        assert open(src, "rb").read() == open(os.path.join(ref_runner.REF_DIR, "nerf_sandbox/source/train/trainer.py"), "rb").read()


def test_default_mode_selection():
    from nerf_sandbox_b200 import mlps
    prev = mlps.set_default_mode("bf16")
    try:
        assert mlps.get_default_mode() == "bf16"
        net = mlps.NeRF(63, 27)                       # how the reference builds it (train/trainer.py:326-341): no mode argument
        from nerf_sandbox_b200 import _lib
        assert net.mode == _lib.MODE_BF16 and mlps.NeRF(63, 27, mode="fp32").mode == _lib.MODE_FP32
        with pytest.raises(ValueError):
            mlps.set_default_mode("fp8")
    finally:
        mlps.set_default_mode(prev)
