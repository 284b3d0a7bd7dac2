"""CPU checks of the typed entry points of the device-resident loss (bfloat16 / float16 logits): they are exported,
and their workspace bound is the fp32 one plus, for a reduced-precision call with a gradient, exactly the fp32
staging region of the gradient rows."""
import ctypes

import pytest

from pytorch_end2end_speech_recognition_b200 import _lib

SHAPES = [(1, 1, 1, 0), (30, 30, 4, 8), (775, 62, 32, 75), (1000, 3386, 64, 150), (37, 14075, 3, 11), (0, 5, 2, 3)]


def bound(lib, T, V, B, L, dtype=None, need_grad=1):
    n = ctypes.c_size_t()
    if dtype is None:
        assert lib.b200ctc_get_workspace_bound(T, V, B, L, ctypes.byref(n)) == 0
    else:
        assert lib.b200ctc_get_workspace_bound_typed(T, V, B, L, dtype, need_grad, ctypes.byref(n)) == 0
    return n.value


def test_typed_symbols_are_exported():
    lib = _lib.load()
    for name in ("b200ctc_loss_and_grad_dev_typed", "b200ctc_get_workspace_bound_typed", "b200ctc_scale_grads"):
        assert name in _lib.EXPORTED_SYMBOLS
        assert hasattr(lib, name)


@pytest.mark.parametrize("shape", SHAPES)
def test_float32_bound_equals_the_untyped_bound(shape):
    lib = _lib.load()
    for need_grad in (0, 1):
        assert bound(lib, *shape, dtype=_lib.FLOAT32, need_grad=need_grad) == bound(lib, *shape)


@pytest.mark.parametrize("dtype", [_lib.BFLOAT16, _lib.FLOAT16])
@pytest.mark.parametrize("shape", SHAPES)
def test_reduced_bound_adds_exactly_the_staging_region(shape, dtype):
    lib = _lib.load()
    T, V, B, _ = shape
    staging = (4 * T * B * V + 255) // 256 * 256
    assert bound(lib, *shape, dtype=dtype, need_grad=1) == bound(lib, *shape) + staging
    assert bound(lib, *shape, dtype=dtype, need_grad=0) == bound(lib, *shape)


def test_unknown_dtype_is_rejected():
    lib = _lib.load()
    n = ctypes.c_size_t()
    assert lib.b200ctc_get_workspace_bound_typed(10, 30, 2, 5, 3, 1, ctypes.byref(n)) == 1     # invalid value
    assert lib.b200ctc_get_workspace_bound_typed(10, 30, 2, 5, -1, 1, ctypes.byref(n)) == 1


def test_scale_grads_rejects_bad_arguments():
    lib = _lib.load()
    one = ctypes.c_void_p(16)                                   # never dereferenced: every call below is rejected
    assert lib.b200ctc_scale_grads(one, one, _lib.FLOAT32, 2, 3, 4, one, 1, None) == 1    # fp32 has no such pass
    assert lib.b200ctc_scale_grads(one, one, 3, 2, 3, 4, one, 1, None) == 1
    assert lib.b200ctc_scale_grads(one, one, _lib.BFLOAT16, 2, 3, 4, one, 2, None) == 1   # n_scale neither 1 nor B
    assert lib.b200ctc_scale_grads(None, one, _lib.BFLOAT16, 2, 3, 4, one, 3, None) == 1
    assert lib.b200ctc_scale_grads(one, one, _lib.FLOAT16, 2, 3, 0, one, 1, None) == 1     # V < 1
    assert lib.b200ctc_scale_grads(None, None, _lib.FLOAT16, 0, 3, 4, None, 1, None) == 0  # nothing to do
