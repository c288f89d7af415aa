"""ctypes binding of libattwarp_sm100.so (the C ABI in include/attwarp.h).

The product path has no CPU fallback: if the shared library is missing this module raises on
first use with the build command, and every wrapper raises ``AttWarpError`` (or the reference's
exception type, mapped by the callers) on a non-zero status.
"""

from __future__ import annotations

import ctypes as C
import os

import torch

_LIB_NAME = "libattwarp_sm100.so"
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)

OK, ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_WORKSPACE = 0, -1, -2, -3, -4

U8, F32, F64, BF16, F16 = 0, 1, 2, 3, 4
LAYOUT_HWC, LAYOUT_CHW = 0, 1
TRANSFORM_IDS = {"identity": 0, "square": 1, "sqrt": 2, "exp": 3, "log": 4}

TORCH_DTYPE_IDS = {torch.uint8: U8, torch.float32: F32, torch.float64: F64,
                   torch.bfloat16: BF16, torch.float16: F16}


class AttWarpError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"attwarp status {status}: {message}")
        self.status = status


class TransformParams(C.Structure):
    _fields_ = [("transform", C.c_int32), ("apply_inverse", C.c_int32),
                ("exp_scale", C.c_double), ("exp_divisor", C.c_double)]


class RaggedImage(C.Structure):
    """attwarp_ragged_image: one image of a ragged batch (device pointers, dense HWC uint8)."""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("H", C.c_int32), ("W", C.c_int32),
                ("Ho", C.c_int32), ("Wo", C.c_int32)]


def make_transform(name="identity", exp_scale=1.0, exp_divisor=1.0, apply_inverse=False):
    return TransformParams(TRANSFORM_IDS[name], 1 if apply_inverse else 0,
                           float(exp_scale), float(exp_divisor))


_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t
_tp = C.POINTER(TransformParams)

# name -> (restype, argtypes); must list every symbol include/attwarp.h declares
SIGNATURES = {
    "attwarp_abi_version": (_i, []),
    "attwarp_last_error": (C.c_char_p, []),
    "attwarp_device_info": (_i, [C.POINTER(_i)] * 3),
    "attwarp_set_sm_share": (_i, [_i]),
    "attwarp_aggregate_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "attwarp_aggregate_attention": (_i, [_vp, _i, _i, _i, _i, _i, _i64, _i64, _i64, _vp, _f, _vp,
                                         _sz, _vp, _i, _f, _vp]),
    "attwarp_maps_workspace_bytes": (_sz, [_i, _i, _i]),
    "attwarp_maps_from_attention": (_i, [_vp, _i, _i, _i, _i, _i, _i, _tp, _vp, _sz, _vp, _vp, _vp]),
    "attwarp_maps_from_tokens": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _tp, _vp, _vp, _vp]),
    "attwarp_maps_from_cdf": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "attwarp_remap_bilinear": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "attwarp_warp_from_attention_tokens": (_i, [_vp, _i, _i, _i, _i, _i64, _i64, _i64, _vp, _i, _i,
                                                _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _tp, _vp,
                                                _sz, _vp, _vp, _vp, C.POINTER(_vp), _vp]),
    "attwarp_revise_mask": (_i, [_vp, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "attwarp_resize_lanczos_u8": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "attwarp_maps_from_mask_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "attwarp_maps_from_mask": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _tp, _vp, _sz, _vp, _vp, _vp]),
    "attwarp_warp_from_pdfs": (_i, [_vp, _vp, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i,
                                    _vp, _vp, _vp, _vp, _vp]),
    "attwarp_ragged_workspace_bytes": (_sz, [_vp, _i]),
    "attwarp_ragged_last_launches": (_i, []),
    "attwarp_warp_ragged_from_tokens": (_i, [_vp, _i, _i, _i, _vp, _i, _tp, _vp, _sz, _vp]),
    "attwarp_ragged_attention_workspace_bytes": (_sz, [_vp, _i]),
    "attwarp_warp_ragged_from_attention": (_i, [_vp, _vp, _i, _i, _i, _tp, _vp, _sz, _vp]),
    "attwarp_ragged_mask_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "attwarp_warp_ragged_from_mask": (_i, [_vp, _vp, _i, _i, _i, _i, _tp, _vp, _sz, _vp, _vp, _vp]),
    "attwarp_png_max_bytes": (_sz, [_i, _i, _i]),
    "attwarp_png_workspace_bytes": (_sz, [_vp, _i]),
    "attwarp_encode_png": (_i, [_vp, _i, _vp, _sz, _vp, _sz, _vp, _vp]),
    "attwarp_jpeg_probe": (_i, [_vp, _sz, _vp]),
    "attwarp_jpeg_workspace_bytes": (_sz, [_vp, _i]),
    "attwarp_decode_jpeg": (_i, [_vp, _i, _vp, _sz, _vp, _vp]),
    "attwarp_png_probe": (_i, [_vp, _sz, _vp]),
    "attwarp_png_decode_workspace_bytes": (_sz, [_vp, _i]),
    "attwarp_decode_png": (_i, [_vp, _i, _vp, _sz, _vp, _vp]),
    "attwarp_overlay_workspace_bytes": (_sz, [_vp, _i, _i]),
    "attwarp_attention_overlay": (_i, [_vp, _i, _i, _i, _i, _i, C.c_double, _vp, _sz, _vp]),
    "attwarp_warp_image_host":(_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _tp, _vp,
                                     C.POINTER(_i)]),
    "attwarp_safe_softmax": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "attwarp_mix_with_uniform": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "attwarp_cdf_from_density": (_i, [_vp, _i, _i, _vp, _vp]),
    "attwarp_make_strictly_increasing": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "attwarp_interp_linear_rows": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "attwarp_gt_marginals": (_i, [_vp, _i, _i, _i, _vp, _sz, _vp, _vp, _vp]),
    "attwarp_upsample_right_inverse": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "attwarp_adaptive_avg_pool2d": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "attwarp_pool_attention": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "attwarp_safe_softmax_backward": (_i, [_vp, _vp, _i, _i, _f, _vp, _vp]),
    "attwarp_mix_with_uniform_backward": (_i, [_vp, _i, _i, _f, _vp, _vp]),
    "attwarp_upsample_right_inverse_backward": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "attwarp_safe_softmax_mix": (_i, [_vp, _i, _i, _f, _f, _vp, _vp]),
    "attwarp_safe_softmax_mix_backward": (_i, [_vp, _vp, _i, _i, _f, _f, _vp, _vp]),
    "attwarp_pdf_l1_loss_workspace_bytes": (_sz, [_i]),
    "attwarp_pdf_l1_loss": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _sz, _vp, _vp]),
    "attwarp_pdf_l1_loss_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp,
                                          _vp, _vp, _vp]),
}

_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load (once) and return the ctypes handle.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(_LIB_PATH):
        raise ImportError(
            f"{_LIB_NAME} not found at {_LIB_PATH}: the CUDA extension is not built and there is "
            "no CPU fallback. Build it with `python -m attwarp_b200.build` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`).")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.attwarp_abi_version() != 1:
        raise ImportError(f"{_LIB_NAME}: ABI version {lib.attwarp_abi_version()} != 1; rebuild")
    _lib = lib
    return lib


def check(status: int):
    if status != OK:
        msg = load().attwarp_last_error().decode("utf-8", "replace")
        raise AttWarpError(status, msg)


def ptr(t):
    """Raw device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("attwarp_b200: tensors must live on a CUDA device "
                               "(there is no CPU implementation in this package)")
