"""CPU checks of fp16 mode (PASN_F16) at the C ABI: which shapes the tensor-core families take, and the full ctypes mirror of
pasn::tcg::Gemm with its fp16 operand switch (used by the GEMM cases of tests/test_fp16_gpu.py)."""
import ctypes as C

import torch
import pytest

import protoasnet_b200 as pasn
from protoasnet_b200 import _lib, synth
from tests.test_tc_gemm_gpu import Aux, Output

OUT_F16 = 4


class Gemm(C.Structure):     # pasn::tcg::Gemm, every field (a subclass of the older mirror would be padded to 456 bytes)
    _fields_ = [("A", C.c_void_p), ("lda", C.c_longlong), ("a_bs", C.c_longlong), ("a_batched", C.c_int), ("ka", C.c_int),
                ("a_mn_major", C.c_int), ("a_rows", C.c_int),
                ("B", C.c_void_p), ("ldb", C.c_longlong), ("b_bs", C.c_longlong), ("b_batched", C.c_int), ("kb", C.c_int),
                ("b_mn_major", C.c_int), ("b_rows", C.c_int),
                ("M", C.c_int), ("N", C.c_int), ("K", C.c_int), ("batch", C.c_int), ("k_rows_per_batch", C.c_int),
                ("npass", C.c_int), ("a_off", C.c_int * 4), ("b_off", C.c_int * 4), ("bn", C.c_int),
                ("bias", C.c_void_p), ("rowparts", C.c_void_p), ("nparts", C.c_int), ("colvec", C.c_void_p),
                ("addin", Aux), ("signin", Aux), ("mask", Aux), ("act", C.c_int), ("out", Output * 2),
                ("psum", C.c_void_p), ("psum_rounded", C.c_int), ("pair", C.c_int),
                ("rowstat", C.c_void_p), ("dotvec", C.c_void_p), ("dot_ld", C.c_longlong), ("dot_mod", C.c_int),
                ("group", C.c_int), ("group_rows", C.c_int), ("group_items", C.c_int), ("stat_rows", C.c_longlong),
                ("dot_early", C.c_int), ("ab_f16", C.c_int)]


def _dims(cfg, dtype=_lib.PASN_F16, path=_lib.PASN_PATH_AUTO, n=8):
    d = synth.CONFIGS[cfg]
    S = 1
    for v in d.spatial:
        S *= v
    return _lib.PasnDims(n, d.C, d.D, d.P, d.K, S, dtype, _lib.PASN_LAYOUT_NCS, _lib.PASN_OCC_ABS, path)


def test_fp16_gemm_mirror_matches_the_library():
    assert _lib.load().pasn_debug_tc_gemm_desc_bytes() == C.sizeof(Gemm) == 448


def test_fp16_dims_take_tensor_core_shapes_only():
    lib = _lib.load()
    assert lib.pasn_head_workspace_bytes(C.byref(_dims("cfg3_video_b1024"))) > 0       # fused shape
    assert lib.pasn_packed_weights_bytes(C.byref(_dims("cfg3_video_b1024"))) > 0
    for cfg in ("tiny_video", "odd_video"):                                               # generic-only shapes: refused
        assert lib.pasn_head_workspace_bytes(C.byref(_dims(cfg))) == 0
        assert lib.pasn_head_backward_workspace_bytes(C.byref(_dims(cfg))) == 0
        assert lib.pasn_tcgen05_supported(C.byref(_dims(cfg))) == 0
    gen = _dims("cfg3_video_b1024", path=_lib.PASN_PATH_GENERIC)                          # the CUDA-core path: refused
    assert lib.pasn_head_workspace_bytes(C.byref(gen)) == 0
    w = _lib.PasnWeights()
    assert lib.pasn_head_forward(16, C.byref(w), None, C.byref(_dims("tiny_video")), 16, 16, None, None, None, None, 16, 16,
                                 None) == -4


def test_fp16_generic_only_head_raises_up_front():
    m = pasn.construct_Video_XProtoNet(pasn.FeatureInput(24), prototype_shape=(8, 16, 1, 1, 1), num_classes=4)
    x = torch.zeros(1, 24, 2, 3, 3, dtype=torch.float16)
    with pytest.raises(_lib.PasnError, match=r"x\.float\(\)"):
        m._rt.make_dims(x.cuda() if torch.cuda.is_available() else _CudaLike(x), m.kernel_path)


class _CudaLike:
    """a CPU tensor that passes make_dims' device check (the shape / dtype rules are host logic)"""

    def __init__(self, t):
        self._t = t
        self.is_cuda = True

    def __getattr__(self, name):
        return getattr(self._t, name)
