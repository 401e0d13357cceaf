"""ctypes binding of libdd_b200.so (include/dd_b200.h).

The product path has no CPU or library fallback: if the shared library is missing, or a call
returns non-zero, a RuntimeError is raised with the library's own error text.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_longlong, c_size_t, c_void_p

import torch  # noqa: F401  (loads libcudart.so.12 into the process before our library)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdd_b200.so")

DD_F32, DD_BF16 = 0, 1
IN_VIEWS, IN_U8 = 1, 2          # dd_conv_c1_* in_flags
IMPL_AUTO, IMPL_SIMT, IMPL_TCGEN05 = 0, 1, 2

_P, _I, _L, _Z, _F = c_void_p, c_int, c_longlong, c_size_t, c_float

# name -> (restype, argtypes); mirrors include/dd_b200.h declaration by declaration
SIGNATURES = {
    "dd_version": (_I, []),
    "dd_last_error": (_I, [c_char_p, _Z]),
    "dd_launch_count": (_L, []),
    "dd_stitch_f32": (_I, [_P, _P, _I, _I, _I, _P]),
    "dd_stitch_mask_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "dd_stitch_u8": (_I, [_P, _P, _I, _I, _I, _P]),
    "dd_unstitch_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "dd_u8_to_f32": (_I, [_P, _P, _L, _P]),
    "dd_conv_c1_fwd": (_I, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "dd_conv_c1_fwd_bits": (_I, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "dd_encoder_c1c2_fused_fwd": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "dd_conv_c1_wgrad": (_I, [_P, _I, _P, _I, _P, _P, _P, _Z, _I, _I, _I, _I, _P]),
    "dd_conv_c1_dgrad": (_I, [_P, _I, _P, _P, _I, _I, _I, _I, _I, _P]),
    "dd_conv3x3_c32_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dd_conv3x3_c32_dgrad": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dd_conv3x3_c32_fwd_bits": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dd_conv3x3_c32_dgrad_bits": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dd_conv3x3_c32_wgrad": (_I, [_P, _P, _P, _P, _P, _Z, _I, _I, _I, _I, _I, _I, _P]),
    "dd_conv_wgrad_workspace_bytes": (_Z, []),
    "dd_pool4_fwd": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "dd_pool4_fwd_f32": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "dd_pool4_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "dd_nhwc_to_nchw_f32": (_I, [_P, _I, _P, _I, _I, _I, _I, _P]),
    "dd_nchw_f32_to_nhwc": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "dd_relu_mask": (_I, [_P, _P, _P, _I, _L, _P]),
    "dd_linear_fwd": (_I, [_P, _I, _P, _P, _P, _P, _Z, _I, _I, _L, _I, _P]),
    "dd_linear_dgrad": (_I, [_P, _P, _P, _I, _P, _Z, _I, _I, _L, _I, _P]),
    "dd_linear_wgrad": (_I, [_P, _P, _I, _P, _P, _I, _I, _L, _I, _P]),
    "dd_linear_wgrad_acc": (_I, [_P, _P, _I, _P, _P, _I, _I, _L, _I, _I, _P]),
    "dd_linear_bwd_adam": (_I, [_P, _P, _P, _P, _P, _P, _I, _P, _P, _Z, _I, _I, _L, _F, _F, _F, _F, _F, _L, _P]),
    "dd_linear_bwd_adam_acc": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _Z, _I, _I, _L, _F, _F, _F, _F, _F, _L, _P]),
    "dd_linear_bwd_adam_sumsq": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _Z, _I, _I, _L, _F, _F, _F, _F, _F, _L, _P, _P,
                                      _Z, _P]),
    "dd_linear_workspace_bytes": (_Z, [_I, _I, _L]),
    "dd_linear_tc_supported": (_I, [_I, _I, _L]),
    "dd_bce_ts_fwd": (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _Z, _L, _P]),
    "dd_bce_bwd": (_I, [_P, _P, _I, _P, _P, _L, _P]),
    "dd_bce_ts_workspace_bytes": (_Z, []),
    "dd_threat_score_f32": (_I, [_P, _P, _P, _P, _Z, _L, _P]),
    "dd_conv2d_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _Z, _P]),
    "dd_conv2d_dgrad": (_I, [_P, _P, _P, _P, _P, _I, _P, _Z, _P]),
    "dd_conv2d_wgrad": (_I, [_P, _P, _P, _P, _P, _I, _P, _Z, _P]),
    "dd_conv2d_workspace_bytes": (_Z, [_P]),
    "dd_conv2d_tc_supported": (_I, [_P, _I, _I]),
    "dd_view_extract": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "dd_view_extract_bwd": (_I, [_P, _I, _P, _I, _I, _I, _I, _I, _P]),
    "dd_nhwc_place": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "dd_sigmoid_bwd": (_I, [_P, _P, _P, _I, _L, _P]),
    "dd_bce_prob_fwd": (_I, [_P, _P, _P, _P, _Z, _L, _P]),
    "dd_bce_prob_bwd": (_I, [_P, _P, _P, _P, _L, _P]),
    "dd_bce_prob_workspace_bytes": (_Z, []),
    "dd_ats_bounding_boxes": (_I, [_P, _I, _P, _I, _P, _P, _P]),
    "dd_boxes_to_map": (_I, [_P, _I, _P, _I, _P, _P]),
    "dd_mse_fwd": (_I, [_P, _P, _P, _P, _Z, _L, _P]),
    "dd_mse_bwd": (_I, [_P, _P, _P, _P, _L, _P]),
    "dd_adam_step": (_I, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _L, _F, _P]),
    "dd_adam_step_sharded": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _L, _L, _F, _F, _F, _F, _F, _L, _F, _I, _P]),
    "dd_grad_sumsq_workspace_bytes": (_Z, []),
    "dd_grad_sumsq": (_I, [_P, _P, _I, _F, _P, _P, _Z, _P]),
    "dd_adam_step_clipped": (_I, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _L, _F, _P, _P]),
    "dd_adam_step_sharded_sumsq": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _L, _L, _F, _F, _F, _F, _F, _L, _F, _I, _P, _P, _Z, _P]),
    "dd_grad_sumsq_each_workspace_bytes": (_Z, []),
    "dd_grad_sumsq_each": (_I, [_P, _P, _P, _I, _P, _Z, _P]),
    "dd_grad_sumsq_each_replicas": (_I, [_P, _I, _I, _F, _P, _P, _P, _I, _P, _Z, _P]),
}



class ConvDesc(ctypes.Structure):
    """dd_conv_desc (include/dd_b200.h): the forward layer, for all three passes."""
    _fields_ = [(n, c_int) for n in ("B", "Cin", "Cout", "Hi", "Wi", "Ho", "Wo", "kh", "kw", "sh", "sw", "ph", "pw",
                                     "dh", "dw", "transposed")]


_lib = None


def load() -> ctypes.CDLL:
    """Load the library once; raise (never fall back) when it is absent or incomplete."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C driving-dirty_b200/csrc`). There is no CPU or PyTorch fallback for this path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the binary disagree
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def last_error() -> str:
    buf = ctypes.create_string_buffer(512)
    load().dd_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(code: int, what: str) -> None:
    if code != 0:
        kind = "dd_status" if code < 0 else "cudaError"
        raise RuntimeError(f"{what} failed ({kind} {code}): {last_error()}")


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)


def launch_count() -> int:
    return int(load().dd_launch_count())


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return DD_F32
    if dt == torch.bfloat16:
        return DD_BF16
    raise RuntimeError(f"unsupported activation dtype {dt}")
