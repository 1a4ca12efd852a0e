"""ctypes binding of libpasn_b200.so (the C ABI declared in include/pasn.h).

There is no CPU implementation behind this module: if the shared library is missing, or a
compute entry point is called without a CUDA device, it raises -- it never falls back.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpasn_b200.so")

PASN_F32, PASN_BF16, PASN_F16 = 0, 1, 2
PASN_LAYOUT_NCS, PASN_LAYOUT_NSC = 0, 1
PASN_OCC_ABS = 0
PASN_PATH_AUTO, PASN_PATH_GENERIC, PASN_PATH_TCGEN05, PASN_PATH_TILED = 0, 1, 2, 3

# every symbol include/pasn.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = [
    "pasn_abi_version", "pasn_strerror", "pasn_tcgen05_supported", "pasn_head_workspace_bytes",
    "pasn_packed_weights_bytes", "pasn_pack_weights", "pasn_head_forward", "pasn_occurrence_only",
    "pasn_push_record_bytes", "pasn_push_init", "pasn_push_decode", "pasn_push_reduce", "pasn_push_write_prototypes",
    "pasn_push_merge_peers", "pasn_push_capture",
    "pasn_debug_launch_count", "pasn_debug_time_main_kernel", "pasn_debug_last_main_kernel_ms",
    "pasn_debug_sm100_error", "pasn_debug_set_trace", "pasn_debug_fault", "pasn_debug_set_fault",
    "pasn_head_backward_workspace_bytes", "pasn_head_backward", "pasn_similarity_stats", "pasn_occurrence_lnorm",
    "pasn_debug_tc_gemm_desc_bytes", "pasn_debug_tc_gemm", "pasn_debug_set_gemm_trace",
]


# torch dtype -> pasn_dtype of the feature / occurrence maps the library takes
DTYPES = {torch.float32: PASN_F32, torch.bfloat16: PASN_BF16, torch.float16: PASN_F16}


class PasnDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("N", "C", "D", "P", "K", "S", "dtype", "layout", "occ_act", "path")]


class PasnWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "addon_w1", "addon_b1", "addon_w2", "addon_b2", "occ_w1", "occ_b1", "occ_w2", "occ_b2", "occ_w3",
        "prototypes", "last_layer")]


class PasnGrads(C.Structure):
    _fields_ = PasnWeights._fields_


class PasnPushArgs(C.Structure):
    _fields_ = [("labels", C.c_void_p), ("proto_class", C.c_void_p), ("global_offset", C.c_int64),
                ("best_key", C.c_void_p), ("best_vec", C.c_void_p)]


PASN_CAPTURE_MAX_SLOTS = 8


class PasnCaptureSlot(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("row_bytes", C.c_int64), ("clip_stride_bytes", C.c_int64),
                ("proto_stride_bytes", C.c_int64)]


class PasnError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the library (once).  Raises if it has not been built (run ``python -c 'import __graft_entry__ as g; g.build()'``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PasnError(
            f"{LIB_PATH} not found: build it with `make -C protoasnet_b200/csrc` (or __graft_entry__.build()). "
            "protoasnet_b200 has no CPU/PyTorch fallback for the prototype head.")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i32, i64 = C.c_void_p, C.c_size_t, C.c_int32, C.c_int64
    lib.pasn_abi_version.restype = C.c_int
    lib.pasn_strerror.restype = C.c_char_p
    lib.pasn_strerror.argtypes = [C.c_int]
    lib.pasn_tcgen05_supported.restype = C.c_int
    lib.pasn_tcgen05_supported.argtypes = [C.POINTER(PasnDims)]
    lib.pasn_head_workspace_bytes.restype = sz
    lib.pasn_head_workspace_bytes.argtypes = [C.POINTER(PasnDims)]
    lib.pasn_packed_weights_bytes.restype = sz
    lib.pasn_packed_weights_bytes.argtypes = [C.POINTER(PasnDims)]
    lib.pasn_pack_weights.restype = C.c_int
    lib.pasn_pack_weights.argtypes = [C.POINTER(PasnWeights), C.POINTER(PasnDims), vp, vp]
    lib.pasn_head_forward.restype = C.c_int
    lib.pasn_head_forward.argtypes = [vp, C.POINTER(PasnWeights), vp, C.POINTER(PasnDims), vp, vp, vp, vp, vp,
                                      C.POINTER(PasnPushArgs), vp, sz, vp]
    lib.pasn_occurrence_only.restype = C.c_int
    lib.pasn_occurrence_only.argtypes = [vp, C.POINTER(PasnWeights), vp, C.POINTER(PasnDims), vp, vp, sz, vp]
    lib.pasn_push_init.restype = C.c_int
    lib.pasn_push_init.argtypes = [vp, i32, vp]
    lib.pasn_push_decode.restype = C.c_int
    lib.pasn_push_decode.argtypes = [vp, i32, vp, vp, vp]
    lib.pasn_push_record_bytes.restype = sz
    lib.pasn_push_record_bytes.argtypes = [i32, i32]
    lib.pasn_push_reduce.restype = C.c_int
    lib.pasn_push_reduce.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.pasn_push_merge_peers.restype = C.c_int
    lib.pasn_push_merge_peers.argtypes = [vp, vp, i32, i32, C.c_uint32, i32, i32, vp, vp, vp, vp, vp]
    lib.pasn_push_capture.restype = C.c_int
    lib.pasn_push_capture.argtypes = [vp, i32, i64, i32, C.POINTER(PasnCaptureSlot), i32, vp]
    lib.pasn_push_write_prototypes.restype = C.c_int
    lib.pasn_push_write_prototypes.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.pasn_debug_launch_count.restype = C.c_ulonglong
    lib.pasn_debug_time_main_kernel.restype = C.c_int
    lib.pasn_debug_time_main_kernel.argtypes = [C.c_int]
    lib.pasn_debug_last_main_kernel_ms.restype = C.c_float
    lib.pasn_debug_set_trace.restype = C.c_int
    lib.pasn_debug_set_trace.argtypes = [vp]
    lib.pasn_head_backward_workspace_bytes.restype = C.c_size_t
    lib.pasn_head_backward_workspace_bytes.argtypes = [C.POINTER(PasnDims)]
    lib.pasn_head_backward.restype = C.c_int
    lib.pasn_head_backward.argtypes = [vp, C.POINTER(PasnWeights), C.POINTER(PasnDims), vp, vp, vp, C.POINTER(PasnGrads),
                                       vp, vp, C.c_size_t, vp]
    lib.pasn_similarity_stats.restype = C.c_int
    lib.pasn_similarity_stats.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          vp, vp, vp, vp, vp, vp]
    lib.pasn_occurrence_lnorm.restype = C.c_int
    lib.pasn_occurrence_lnorm.argtypes = [vp, C.c_int32, C.c_int64, C.c_int32, C.c_int32, vp, vp, vp]
    lib.pasn_debug_fault.restype = C.c_int
    lib.pasn_debug_set_fault.restype = C.c_int
    lib.pasn_debug_set_fault.argtypes = [C.c_int]
    lib.pasn_debug_sm100_error.restype = C.c_int
    lib.pasn_debug_sm100_error.argtypes = [vp, C.POINTER(PasnDims), vp]
    lib.pasn_debug_tc_gemm_desc_bytes.restype = sz
    lib.pasn_debug_tc_gemm.restype = C.c_int
    lib.pasn_debug_tc_gemm.argtypes = [vp, sz, vp]
    lib.pasn_debug_set_gemm_trace.restype = C.c_int
    lib.pasn_debug_set_gemm_trace.argtypes = [vp]
    if lib.pasn_abi_version() != 2:
        raise PasnError("libpasn_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(status: int, what: str = "pasn call") -> None:
    if status != 0:
        msg = load().pasn_strerror(status).decode()
        raise PasnError(f"{what} failed: {msg} (status {status})")
