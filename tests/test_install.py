"""The drop-in seam: install() rebinds the reference's by-name imports (only where the reference is present)."""
import sys

import pytest

from baseline import ref_runner

REF = ref_runner.REF_DIR          # the unmodified reference package, vendored by __graft_entry__.build()


@pytest.mark.skipif(not ref_runner.available(), reason="oracle/_ref holds no reference")
def test_install_rebinds_reference_names():
    sys.path.insert(0, REF)
    try:
        import nerf_sandbox_b200 as nsb
        from nerf_sandbox_b200.install import install, uninstall
        done = install(mode="bf16")
        from nerf_sandbox_b200 import mlps
        assert mlps.get_default_mode() == "bf16"
        mlps.set_default_mode("fp32")
        import nerf_sandbox.source.train.trainer as T
        import nerf_sandbox.source.utils.render_utils as RU
        import nerf_sandbox.source.utils.validation_renderer as VR
        assert T.NeRF is nsb.NeRF and T.nerf_forward_pass is nsb.nerf_forward_pass and T.sample_pdf is nsb.sample_pdf
        assert T.get_vanilla_nerf_encoders is nsb.get_vanilla_nerf_encoders and T.volume_render_rays is nsb.volume_render_rays
        assert RU.render_image_chunked is nsb.render_image_chunked and VR.render_image_chunked is nsb.render_image_chunked
        assert "nerf_sandbox.source.train.trainer" in done
        # the reference Trainer's constructor probes (trainer.py:367-380) work on our NeRF
        m = T.NeRF(63, 27, 8, 256, skip_pos=4)
        T.log_nerf_arch(m, logger=lambda s: None); m._debug_dump_arch_once(); m.enable_debug(3, lambda s: None)
        orig = T.NeRF
        uninstall()
        assert T.NeRF is not orig and T.NeRF.__module__.startswith("nerf_sandbox.source")      # the reference's own class is back
    finally:
        sys.path.remove(REF)
        for k in [k for k in sys.modules if k.startswith("nerf_sandbox.")]:
            del sys.modules[k]
