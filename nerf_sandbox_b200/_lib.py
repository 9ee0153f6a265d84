"""ctypes binding of libnsb.so (C ABI: include/nsb.h).

There is no CPU fallback: if the shared library is missing the import of any op raises, and every
op refuses non-CUDA tensors.  Build with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C nerf_sandbox_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnsb.so")
CSRC = os.path.join(_HERE, "csrc")

MODE_FP32, MODE_BF16 = 0, 1
PACK_TRAIN_ONLY = 0x100
WHITE_BKGD, INFINITE_LAST_BIN, TRAINING, SIGMA_SOFTPLUS = 1, 2, 4, 8
N_PARAMS = 595844

_p, _i64, _i32, _u32, _u64, _f32, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_uint32, C.c_uint64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/nsb.h declares (tests/test_abi.py checks)
SIGNATURES = {
    "nsb_version": (_i32, []),
    "nsb_error_string": (C.c_char_p, [_i32]),
    "nsb_last_cuda_error": (C.c_char_p, []),
    "nsb_launch_count": (_i64, []),
    "nsb_stratified_z": (_i32, [_p, _p, _i64, _i32, _f32, _f32, _i32, _u64, _u64, _p]),
    "nsb_sample_pdf": (_i32, [_p, _i32, _p, _i32, _p, _p, _p, _p, _i64, _i32, _i32, _u64, _u64, _p]),
    "nsb_resample_merge": (_i32, [_p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u64, _u64, _p]),
    "nsb_composite_fwd": (_i32, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _u32, _f32, _p]),
    "nsb_composite_bwd": (_i32, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _u32, _f32, _p]),
    "nsb_composite_raw_fwd": (_i32, [_p, _p, _f32, _p, _p, _p, _p, _p, _p, _i64, _i32, _u32, _u64, _u64, _p]),
    "nsb_composite_raw_bwd": (_i32, [_p, _p, _f32, _p, _p, _p, _p, _i64, _i32, _u32, _u64, _u64, _p]),
    "nsb_composite_raw_bwd_ex": (_i32, [_p, _p, _f32, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _u32, _u64, _u64, _p]),
    "nsb_composite_raw_bwd_mse": (_i32, [_p, _p, _f32, _p, _p, _p, _f32, _p, _i64, _i32, _u32, _u64, _u64, _p]),
    "nsb_mse_loss": (_i32, [_p, _p, _p, _p, _p, _p, _i64, _f32, _p]),
    "nsb_encode": (_i32, [_p, _p, _i64, _i32, _i32, _i32, _p]),
    "nsb_encode_bwd": (_i32, [_p, _p, _p, _i64, _i32, _i32, _i32, _p]),
    "nsb_encode_bwd_rays": (_i32, [_p] * 10 + [_i64, _i32, _p]),
    "nsb_packed_weights_bytes": (_sz, []),
    "nsb_pack_weights": (_i32, [_p, _p, _i32, _p]),
    "nsb_pack_weights_batch": (_i32, [_p, _p, _i32, _i32, _p]),
    "nsb_field_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "nsb_field_fwd_enc": (_i32, [_p, _p, _p, _p, _p, _sz, _i64, _i32, _i32, _p]),
    "nsb_field_fwd_rays": (_i32, [_p, _p, _p, _p, _p, _p, _p, _p, _sz, _i64, _i32, _i32, _i32, _p]),
    "nsb_field_bwd": (_i32, [_p, _p, _p, _p, _sz, _i64, _i32, _p]),
    "nsb_field_bwd_ex": (_i32, [_p, _p, _p, _p, _p, _p, _sz, _i64, _i32, _p]),
    "nsb_adam_step": (_i32, [_p, _p, _p, _p, _i64, _f32, _f32, _f32, _f32, _i64, _f32, _p, _p]),
    "nsb_grad_clip": (_i32, [_p, _i64, _f32, _f32, _p, _p]),
    "nsb_adam_allreduce_step": (_i32, [_p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _i32, _i32, _u32, _i64, _f32, _f32, _f32, _f32, _i64, _f32, _p, _p]),
    "nsb_peer_status": (_i32, [C.POINTER(C.c_int)]),
    "nsb_train_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "nsb_train_fwd_bwd": (_i32, [_p] * 13 + [_sz, _i64, _i32, _i32, _f32, _f32, _f32, _u32, _i32, _i32, _f32, _u64, _u64,
                                 _p, _p, _p, _p, _p]),
    "nsb_train_step": (_i32, [_p] * 14 + [_sz, _i64, _i32, _i32, _f32, _f32, _f32, _u32, _i32, _i32, _u64, _f32, _f32, _i64, _f32, _f32, _f32,
                              _f32, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _p]),
    "nsb_train_workspace_bytes_ex": (_sz, [_i64, _i32, _i32, _i32, _i32]),
    "nsb_train_fwd_bwd_ex": (_i32, [_p] * 13 + [_sz, _i64, _i32, _i32, _f32, _f32, _f32, _u32, _i32, _i32, _f32, _u64, _u64]
                             + [_p] * 8),
    "nsb_render_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "nsb_render_rays": (_i32, [_p] * 10 + [_sz, _i64, _i32, _i32, _f32, _f32, _u32, _i32, _p]),
    "nsb_frame_output": (_i32, [_p, _p, _p, _i64, C.c_double, C.c_double, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    "nsb_camera_rays": (_i32, [_i32, _i32, _p, _p, _i32, _i32, _i32, _i32, _f32, _p, _i64] + [_p] * 7),
    "nsb_camera_rays_bwd_workspace_bytes": (_sz, [_i64, _i32]),
    "nsb_camera_rays_bwd": (_i32, [_i32, _i32, _p, _p, _i32, _p, _i32, _i32, _i32, _f32, _p, _i64] + [_p] * 8 + [_sz, _p]),
    "nsb_sample_pixel_batch": (_i32, [_p, _i32, _i32, _i32, _i32, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _f32,
                                      _i64, _u64, _u64] + [_p] * 10),
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile libnsb.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("nvcc build of libnsb.so failed")
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: nerf_sandbox_b200 has no CPU/PyTorch fallback. "
                "Build it with `make -C nerf_sandbox_b200/csrc` (or __graft_entry__.build()).")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)           # AttributeError if the library does not export it
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


class NsbError(RuntimeError):
    pass


def check(code: int, what: str = "") -> None:
    if code == 0:
        return
    L = lib()
    msg = L.nsb_error_string(code).decode()
    if code == -3:
        msg += ": " + L.nsb_last_cuda_error().decode()
    if code == -1:
        raise ValueError(f"libnsb {what}: {msg}")
    raise NsbError(f"libnsb {what}: {msg}")


def ptr(t: torch.Tensor | None) -> int | None:
    """Device pointer of a contiguous fp32/int64 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("nerf_sandbox_b200 ops take CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("nerf_sandbox_b200 ops take contiguous tensors")
    return t.data_ptr()


def f32c(t: torch.Tensor | None) -> torch.Tensor | None:
    """Contiguous fp32 view/copy (the reference accepts any float dtype; the kernels compute in fp32)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("nerf_sandbox_b200 ops take CUDA tensors only (no CPU fallback)")
    return t.detach().to(torch.float32).contiguous()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(lib().nsb_launch_count())
