"""Batched greedy (best-path) CTC decoding on the GPU.

Mirror of ``models/pytorch_v3/ctc/decoders/greedy_decoder.py`` (class ``GreedyDecoder``, same
constructor and call signature): ``GreedyDecoder(blank_index)(logits[B,T,V], x_lens[B])``.
The reference moves the whole logits tensor to the host (ctc.py:436-437) and loops over B*T
frames in python; here the argmax / collapse / blank removal run as CUDA kernels
(csrc/greedy.cu) and only the hypotheses come back.
"""

import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import B200CTCError

# element types the decoders and the posterior softmax read (b200ctc_dtype_t); a 16-bit value is widened to fp32 as
# it is loaded, so results equal those of the fp32 call on ``x.float()``
DTYPES = {torch.float32: _lib.FLOAT32, torch.bfloat16: _lib.BFLOAT16, torch.float16: _lib.FLOAT16}


def greedy_decode(logits, x_lens, blank=0):
    """logits: CUDA fp32, bfloat16 or float16 [B,T,V] (any batch/time strides, unit vocabulary stride);
    x_lens: int tensor/array [B].  Returns device tensors (tokens[B,T] int32 padded with -1,
    lens[B] int32); no host synchronisation.  16-bit logits are decoded as they are, with the result of
    ``greedy_decode(logits.float(), ...)``."""
    if not isinstance(logits, torch.Tensor) or not logits.is_cuda:
        raise B200CTCError("logits must be a CUDA tensor: this decoder has no CPU path")
    if logits.dtype not in DTYPES or logits.dim() != 3:
        raise B200CTCError("logits must be float32, bfloat16 or float16 [B, T, V]")
    lib = _lib.load()
    if logits.stride(2) != 1 and logits.size(2) > 1:
        logits = logits.contiguous()
    B, T, V = logits.shape
    dev = logits.device
    if isinstance(x_lens, torch.Tensor):
        lens = x_lens.to(device=dev, dtype=torch.int32).contiguous()
    else:
        lens = torch.as_tensor(np.ascontiguousarray(np.asarray(x_lens), dtype=np.int32)).to(dev)
    if lens.numel() != B:
        raise B200CTCError("x_lens must have one entry per utterance")
    with torch.cuda.device(dev):
        tokens = torch.empty((B, T), dtype=torch.int32, device=dev)
        out_lens = torch.empty(B, dtype=torch.int32, device=dev)
        st = lib.b200ctc_greedy_decode_typed(logits.data_ptr(), DTYPES[logits.dtype], logits.stride(0), logits.stride(1),
                                             lens.data_ptr(), T, V, B, int(blank), tokens.data_ptr(), out_lens.data_ptr(),
                                             torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(st, "b200ctc_greedy_decode_typed")
    return tokens, out_lens


class GreedyDecoder(object):
    """Drop-in for the reference's numpy ``GreedyDecoder`` (greedy_decoder.py:14-47)."""

    def __init__(self, blank_index):
        self._blank = blank_index

    def __call__(self, logits, x_lens, device=None):
        """logits: np.ndarray or tensor [B,T,V]; x_lens: [B].  Returns what the reference
        returns: an array of per-utterance int arrays (2-D when all hypotheses have equal
        length, as ``np.array(list_of_arrays)`` used to produce)."""
        if isinstance(logits, np.ndarray):
            dev = torch.device(device if device is not None else "cuda")
            logits_t = torch.from_numpy(np.ascontiguousarray(logits, dtype=np.float32)).to(dev)
        else:
            logits_t = logits if logits.is_cuda else logits.to(device if device is not None else "cuda")
            if logits_t.dtype not in (torch.bfloat16, torch.float16):
                logits_t = logits_t.float()
        tokens, lens = greedy_decode(logits_t, x_lens, self._blank)
        tokens = tokens.cpu().numpy()
        lens = lens.cpu().numpy()
        hyps = [tokens[b, :lens[b]].astype(np.int64) for b in range(tokens.shape[0])]
        if len(hyps) > 0 and all(len(h) == len(hyps[0]) for h in hyps):
            return np.array(hyps)
        out = np.empty(len(hyps), dtype=object)
        for i, h in enumerate(hyps):
            out[i] = h
        return out


def beam_search_decode(log_probs, x_lens, beam_width, blank=0, return_scores=False, lm=None, alpha=0.0, beta=0.0):
    """Batched CTC prefix beam search on the GPU.
    log_probs: CUDA fp32, bfloat16 or float16 [B,T,V] log-probabilities (any batch/time strides); x_lens [B].
    Returns device tensors (tokens[B,T] int32 padded with -1, lens[B] int32[, scores[B] fp32]); 16-bit inputs give
    the result of ``beam_search_decode(log_probs.float(), ...)``.
    lm: an ``NGramLM`` loaded for these V symbols and this blank on the device of ``log_probs``; candidates are then
    ranked with the LM score ``S(prefix + c) = S(prefix) + alpha * ln P(c | prefix) + beta`` added, and the hypothesis
    includes ``alpha * ln P(</s> | prefix)`` (shallow fusion; include/b200ctc.h, b200ctc_beam_search_lm), as does its
    score.  Without an LM, alpha and beta must be 0."""
    if lm is None and (float(alpha) != 0.0 or float(beta) != 0.0):
        raise B200CTCError("alpha and beta weight a language model: pass lm=NGramLM(...)")
    if not isinstance(log_probs, torch.Tensor) or not log_probs.is_cuda:
        raise B200CTCError("log_probs must be a CUDA tensor: this decoder has no CPU path")
    if log_probs.dtype not in DTYPES or log_probs.dim() != 3:
        raise B200CTCError("log_probs must be float32, bfloat16 or float16 [B, T, V]")
    if not 1 <= int(beam_width) <= 64:
        raise B200CTCError("beam_width must be in 1..64")
    lib = _lib.load()
    if log_probs.stride(2) != 1 and log_probs.size(2) > 1:
        log_probs = log_probs.contiguous()
    B, T, V = log_probs.shape
    dev = log_probs.device
    if isinstance(x_lens, torch.Tensor):
        lens = x_lens.to(device=dev, dtype=torch.int32).contiguous()
    else:
        lens = torch.as_tensor(np.ascontiguousarray(np.asarray(x_lens), dtype=np.int32)).to(dev)
    if lens.numel() != B:
        raise B200CTCError("x_lens must have one entry per utterance")
    with torch.cuda.device(dev):
        tokens = torch.empty((B, T), dtype=torch.int32, device=dev)
        out_lens = torch.empty(B, dtype=torch.int32, device=dev)
        scores = torch.empty(B, dtype=torch.float32, device=dev)
        n = ctypes.c_size_t()
        stream = torch.cuda.current_stream(dev)
        if lm is None:
            _lib.check(lib.b200ctc_beam_search_workspace(B, T, V, int(beam_width), ctypes.byref(n)), "b200ctc_beam_search_workspace")
            ws = torch.empty(max(n.value, 1), dtype=torch.uint8, device=dev)
            st = lib.b200ctc_beam_search_typed(log_probs.data_ptr(), DTYPES[log_probs.dtype], log_probs.stride(0),
                                               log_probs.stride(1), lens.data_ptr(), T, V, B, int(blank), int(beam_width),
                                               tokens.data_ptr(), out_lens.data_ptr(), scores.data_ptr(), ws.data_ptr(),
                                               ws.numel(), stream.cuda_stream)
            _lib.check(st, "b200ctc_beam_search_typed")
        else:
            _lib.check(lib.b200ctc_beam_search_lm_workspace(B, T, V, int(beam_width), ctypes.byref(n)),
                       "b200ctc_beam_search_lm_workspace")
            ws = torch.empty(max(n.value, 1), dtype=torch.uint8, device=dev)
            st = lib.b200ctc_beam_search_lm(log_probs.data_ptr(), DTYPES[log_probs.dtype], log_probs.stride(0),
                                            log_probs.stride(1), lens.data_ptr(), T, V, B, int(blank), int(beam_width),
                                            lm.handle, float(alpha), float(beta), tokens.data_ptr(), out_lens.data_ptr(),
                                            scores.data_ptr(), ws.data_ptr(), ws.numel(), stream.cuda_stream)
            _lib.check(st, "b200ctc_beam_search_lm")
        ws.record_stream(stream)
    return (tokens, out_lens, scores) if return_scores else (tokens, out_lens)


class BeamSearchDecoder(object):
    """Drop-in for the reference's numpy ``BeamSearchDecoder`` (beam_search_decoder.py:22-124): same
    constructor and call signature.  Without ``lm``, ``alpha`` / ``beta`` (language-model weight, insertion bonus)
    are accepted and, as in the reference (whose LM hook is a TODO, :103), unused; with an ``NGramLM`` they weight
    it (``beam_search_decode(..., lm=lm, alpha=alpha, beta=beta)``)."""

    def __init__(self, blank_index, space_index=-1, lm=None):
        self._blank = blank_index
        self._space = space_index
        self._lm = lm

    def __call__(self, log_probs, x_lens, beam_width=1, alpha=0., beta=0., device=None):
        if isinstance(log_probs, np.ndarray):
            dev = torch.device(device if device is not None else "cuda")
            lp = torch.from_numpy(np.ascontiguousarray(log_probs, dtype=np.float32)).to(dev)
        else:
            lp = log_probs if log_probs.is_cuda else log_probs.to(device if device is not None else "cuda")
            if lp.dtype not in (torch.bfloat16, torch.float16):
                lp = lp.float()
        if self._lm is None:
            tokens, lens = beam_search_decode(lp, x_lens, beam_width, self._blank)
        else:
            tokens, lens = beam_search_decode(lp, x_lens, beam_width, self._blank, lm=self._lm, alpha=alpha, beta=beta)
        tokens = tokens.cpu().numpy()
        lens = lens.cpu().numpy()
        hyps = [tokens[b, :lens[b]].astype(np.int64) for b in range(tokens.shape[0])]
        if len(hyps) > 0 and all(len(h) == len(hyps[0]) for h in hyps):
            return np.array(hyps)
        out = np.empty(len(hyps), dtype=object)
        for i, h in enumerate(hyps):
            out[i] = h
        return out
