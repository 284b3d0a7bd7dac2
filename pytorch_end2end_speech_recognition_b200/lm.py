"""Token-level back-off n-gram language model for shallow fusion in the GPU prefix beam search.

``NGramLM(arpa_path, symbols, blank=0, device=None)`` reads an ARPA file (order 1..8) whose words are the decoder's
symbols (``symbols[c]``: the string of decoder id ``c``; ``symbols[blank]`` is not read) and copies the model to a CUDA
device once.  Pass it to ``beam_search_decode``, ``BeamSearchDecoder`` or ``evaluate_batch`` with ``alpha`` (LM weight)
and ``beta`` (insertion bonus).  What the file must satisfy is listed at ``b200ctc_ngram_lm_create``
(include/b200ctc.h); a file that does not raises ``B200CTCError``.
"""

import ctypes
import os

import torch

from . import _lib
from ._lib import B200CTCError


class NGramLM(object):
    """An n-gram model on one CUDA device.  ``order``: N; ``counts``: the n-grams kept per order (1..N), after the
    ones that name a word no symbol maps to are dropped.  ``close()`` (or garbage collection) frees it."""

    def __init__(self, arpa_path, symbols, blank=0, device=None):
        self._h = None
        symbols = list(symbols)
        V = len(symbols)
        if not 0 <= int(blank) < V:
            raise B200CTCError("blank must index symbols")
        if device is None:
            index = torch.cuda.current_device() if torch.cuda.is_available() else 0
        else:
            d = torch.device(device)
            if d.type != "cuda":
                raise B200CTCError("an NGramLM lives on a CUDA device: this decoder has no CPU path")
            index = d.index if d.index is not None else (torch.cuda.current_device() if torch.cuda.is_available() else 0)
        lib = _lib.load()
        arr = (ctypes.c_char_p * V)(*[None if (c == blank or s is None) else str(s).encode("utf-8")
                                      for c, s in enumerate(symbols)])
        h = ctypes.c_void_p()
        _lib.check(lib.b200ctc_ngram_lm_create(os.fsencode(os.fspath(arpa_path)), arr, V, int(blank), int(index),
                                               ctypes.byref(h)), "b200ctc_ngram_lm_create")
        self._h = h
        self._lib = lib
        self.V = V
        self.blank = int(blank)
        self.device = torch.device("cuda", int(index))
        order = ctypes.c_int()
        counts = (ctypes.c_longlong * 8)()
        _lib.check(lib.b200ctc_ngram_lm_info(h, ctypes.byref(order), counts), "b200ctc_ngram_lm_info")
        self.order = order.value
        self.counts = [int(counts[k]) for k in range(self.order)]

    @property
    def handle(self):
        if self._h is None:
            raise B200CTCError("the NGramLM is closed")
        return self._h

    def close(self):
        if self._h is not None:
            self._lib.b200ctc_ngram_lm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
