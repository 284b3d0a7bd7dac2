"""CPU checks of the typed entry points of the decoders and the posterior softmax (bfloat16 / float16 input): they are
exported and declared, an unknown element type is rejected before any pointer is used, and an empty batch is a no-op."""
import ctypes
import os
import re

import pytest

from pytorch_end2end_speech_recognition_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPED = ("b200ctc_greedy_decode_typed", "b200ctc_beam_search_typed", "b200ctc_softmax_temperature_typed")
P = ctypes.c_void_p(16)                         # never dereferenced: every call below returns before using it


def test_decode_typed_symbols_are_exported_and_declared():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "b200ctc.h")).read()
    for name in TYPED:
        assert name in _lib.EXPORTED_SYMBOLS
        assert re.search(r"B200CTC_API\s+int\s+%s\s*\(" % name, header)
        assert getattr(lib, name).argtypes is not None and getattr(lib, name).restype is ctypes.c_int


def greedy(lib, dtype, B=2, ptr=P):
    return lib.b200ctc_greedy_decode_typed(ptr, dtype, 40, 4, ptr, 10, 4, B, 0, ptr, ptr, None)


def beam(lib, dtype, B=2, ptr=P):
    return lib.b200ctc_beam_search_typed(ptr, dtype, 40, 4, ptr, 10, 4, B, 0, 2, ptr, ptr, ptr, ptr, 1 << 20, None)


def softmax(lib, dtype, B=2, ptr=P):
    return lib.b200ctc_softmax_temperature_typed(ptr, dtype, 40, 4, 10, 4, B, 1.0, ptr, None)


@pytest.mark.parametrize("call", [greedy, beam, softmax])
@pytest.mark.parametrize("dtype", [3, -1])
def test_unknown_dtype_is_rejected(call, dtype):
    assert call(_lib.load(), dtype) == 1                                  # invalid value


@pytest.mark.parametrize("call", [greedy, beam, softmax])
@pytest.mark.parametrize("dtype", [_lib.FLOAT32, _lib.BFLOAT16, _lib.FLOAT16])
def test_empty_batch_is_a_no_op(call, dtype):
    assert call(_lib.load(), dtype, B=0, ptr=None) == 0
