"""CPU-side checks of pasn_head_backward_ex (the backward with every upstream gradient of the head): the library exports
it, the ctypes mirror of pasn_upstream has the C layout, and argument validation works without a GPU."""
import ctypes as C

from protoasnet_b200 import _lib


def test_backward_ex_is_exported_and_upstream_is_five_pointers():
    lib = _lib.load()
    assert hasattr(lib, "pasn_head_backward_ex")
    assert "pasn_head_backward_ex" in _lib.SYMBOLS
    assert C.sizeof(_lib.PasnUpstream) == 5 * C.sizeof(C.c_void_p)
    assert [f for f, _ in _lib.PasnUpstream._fields_] == ["grad_logits", "grad_similarity", "grad_distance",
                                                         "grad_occurrence", "grad_features"]


def test_backward_ex_argument_validation_without_gpu():
    lib = _lib.load()
    w, g, up = _lib.PasnWeights(), _lib.PasnGrads(), _lib.PasnUpstream()
    bad = _lib.PasnDims(1, 8, 7, 4, 2, 9, 0, 0, 0, 0)          # odd D
    ok = _lib.PasnDims(0, 8, 6, 4, 2, 9, 0, 0, 0, 1)           # no clips: nothing to do
    call = lib.pasn_head_backward_ex
    assert call(None, C.byref(w), C.byref(bad), C.byref(up), C.byref(g), None, None, 0, None) == -1
    assert call(None, C.byref(w), C.byref(ok), None, C.byref(g), None, None, 0, None) == -1   # `up` is required
    assert call(None, C.byref(w), C.byref(ok), C.byref(up), None, None, None, 0, None) == -1
    assert call(None, C.byref(w), C.byref(ok), C.byref(up), C.byref(g), None, None, 0, None) == 0
