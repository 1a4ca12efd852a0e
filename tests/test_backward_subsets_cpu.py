"""CPU-side checks of the backward's NULL-means-not-wanted rule and of pasn_last_layer_backward: the export and its ctypes
argument types, and argument validation, which answers before anything reaches the device."""
import ctypes as C

from protoasnet_b200 import _lib


def test_last_layer_backward_is_exported_with_argtypes():
    lib = _lib.load()
    assert "pasn_last_layer_backward" in _lib.SYMBOLS
    f = lib.pasn_last_layer_backward
    assert f.restype is C.c_int
    assert f.argtypes == [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]


def test_last_layer_backward_argument_validation_without_gpu():
    f = _lib.load().pasn_last_layer_backward
    fake = 256   # never dereferenced: every call below is refused or has no clips
    for n, p, k in ((-1, 4, 2), (3, 0, 2), (3, 4, 0), (3, -4, 2), (0, 0, 2), (0, 4, -1)):
        assert f(fake, fake, n, p, k, fake, None) == -1, (n, p, k)
    assert f(None, fake, 3, 4, 2, fake, None) == -1
    assert f(fake, None, 3, 4, 2, fake, None) == -1
    assert f(fake, fake, 3, 4, 2, None, None) == -1
    assert f(None, None, 0, 4, 2, None, None) == 0   # N = 0: nothing to do, NULL pointers allowed


def test_backward_ex_takes_null_gradients_but_not_a_null_grads_struct():
    lib = _lib.load()
    w, g, up = _lib.PasnWeights(), _lib.PasnGrads(), _lib.PasnUpstream()   # every gradient pointer NULL
    ok = _lib.PasnDims(0, 8, 6, 4, 2, 9, 0, 0, 0, 1)
    call = lib.pasn_head_backward_ex
    assert call(None, C.byref(w), C.byref(ok), C.byref(up), None, None, None, 0, None) == -1
    assert call(None, C.byref(w), C.byref(ok), C.byref(up), C.byref(g), None, None, 0, None) == 0
    assert lib.pasn_head_backward(None, C.byref(w), C.byref(ok), None, None, None, C.byref(g), None, None, 0, None) == 0
    # clips, but no gradient wanted: done before the feature map or the workspace would be needed
    some = _lib.PasnDims(3, 8, 6, 4, 2, 9, 0, 0, 0, 1)
    assert call(None, C.byref(w), C.byref(some), C.byref(up), C.byref(g), None, None, 0, None) == 0
