"""CPU tests of the batched word-error call: its C-ABI symbols and workspace query, the oracle's word rule, and
that the product path refuses host tensors."""
import ctypes

import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from oracle import word_ref
from pytorch_end2end_speech_recognition_b200 import _lib

NAMES = ("b200ctc_word_errors_workspace", "b200ctc_word_errors")


def test_word_error_symbols_are_exported_and_declared():
    lib = _lib.load()
    for name in NAMES:
        assert name in _lib.EXPORTED_SYMBOLS
        assert hasattr(lib, name)
        assert getattr(lib, name).restype is ctypes.c_int


@pytest.mark.parametrize("B,R,H", [(0, 0, 0), (1, 0, 5), (3, 17, 9), (128, 400, 420), (2, 17000, 17000)])
def test_workspace_query_covers_both_backtraces(B, R, H):
    lib = _lib.load()
    n = ctypes.c_size_t()
    assert lib.b200ctc_word_errors_workspace(B, R, H, ctypes.byref(n)) == 0
    chars = (R + 1) * (H + 1)                              # character CTA: one byte per cell
    words = ((R + 1) // 2 + 1) * ((H + 1) // 2 + 1)        # word CTA: at most (n + 1) // 2 words per sequence
    assert n.value >= B * (chars + words)


def test_workspace_query_rejects_bad_sizes():
    lib = _lib.load()
    n = ctypes.c_size_t()
    for args in [(-1, 4, 4), (2, -1, 4), (2, 4, -1)]:
        assert lib.b200ctc_word_errors_workspace(*args, ctypes.byref(n)) == 1
    assert lib.b200ctc_word_errors_workspace(2, 4, 4, None) == 1


def test_word_errors_rejects_bad_arguments_before_any_cuda_call():
    lib = _lib.load()
    buf = (ctypes.c_int * 64)()
    p = ctypes.addressof(buf)
    # stride < max, negative sizes, null outputs
    assert lib.b200ctc_word_errors(p, 3, p, p, 4, p, 1, 4, 4, 0, p, p, p, p, 256, None) == 1
    assert lib.b200ctc_word_errors(p, 4, p, p, 4, p, -1, 4, 4, 0, p, p, p, p, 256, None) == 1
    assert lib.b200ctc_word_errors(p, 4, p, p, 4, p, 1, 4, 4, 0, None, p, p, p, 256, None) == 1
    assert lib.b200ctc_word_errors(p, 4, p, p, 4, p, 1, 4, 4, 0, p, p, None, p, 256, None) == 1
    # a workspace one byte short of the query
    n = ctypes.c_size_t()
    assert lib.b200ctc_word_errors_workspace(1, 4, 4, ctypes.byref(n)) == 0
    assert lib.b200ctc_word_errors(p, 4, p, p, 4, p, 1, 4, 4, 0, p, p, p, p, n.value - 257, None) == 4
    # an empty batch is a no-op
    assert lib.b200ctc_word_errors(None, 0, None, None, 0, None, 0, 0, 0, 0, None, None, None, None, 0, None) == 0


@pytest.mark.parametrize("seq,space,words", [
    ([7, 1, 7, 7, 2, 7], 7, [(1,), (2,)]),
    ([7, 7, 7], 7, []),
    ([], 7, []),
    ([3, 1, 4, 1], 7, [(3, 1, 4, 1)]),
    ([3, 1, 4, 1], -1, [(3, 1, 4, 1)]),
    ([5, 6, 0, 5, 0, 0, 6, 5], 0, [(5, 6), (5,), (6, 5)]),
])
def test_oracle_split_rule(seq, space, words):
    assert word_ref.split_words(seq, space) == words


def test_oracle_word_errors():
    s = 0
    # "ab c" against "a bc": both words differ, no characters do
    assert word_ref.word_errors([1, 2, s, 3], [1, s, 2, 3], s) == ((2, 2, 0, 0), (0, 0, 0, 0), (2, 3))
    # an all-space reference has no words and no characters
    assert word_ref.word_errors([s, s], [4, s, 5], s) == ((2, 0, 2, 0), (2, 0, 2, 0), (0, 0))
    assert word_ref.word_errors([4, s, 5], [], s) == ((2, 0, 0, 2), (2, 0, 0, 2), (2, 2))


def test_word_errors_refuses_host_tensors():
    refs = torch.zeros((2, 3), dtype=torch.int32)
    lens = torch.tensor([3, 3], dtype=torch.int32)
    with pytest.raises(b200.B200CTCError):
        b200.word_errors(refs, lens, refs, lens, space=0)
