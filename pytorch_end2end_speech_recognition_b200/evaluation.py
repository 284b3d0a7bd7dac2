"""Evaluation on the GPU (SURVEY 8(f) rank 4): batched edit distance with error counts, word and space-free
character error counts of character-level hypotheses, the fused posterior softmax, and one call that turns a
mini-batch of logits into error counts.

Mirrors of the reference (same names, argument meaning and results):
  * ``compute_wer(ref, hyp, normalize)``  -- utils/evaluation/edit_distance.py:53-126
  * ``posteriors(logits, temperature)``   -- the tensor work of CTC.posteriors, models/pytorch_v3/ctc/ctc.py:455-502
  * ``evaluate_batch(...)``               -- the per-utterance loop of the metric code
    (examples/timit/s5/exp/metrics/phone.py:50-108 and its twins: decode, then compute_wer per utterance, with
    ``eval_batch_size=1`` in train.py:283) as greedy decode + edit distance kernels over the whole mini-batch.
"""

import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import B200CTCError
from .decode import DTYPES, beam_search_decode, greedy_decode


def _padded_i32(seqs, dev):
    """list of int sequences -> ([B, Lmax] int32 CUDA tensor, [B] int32 CUDA lengths)."""
    lens = np.array([len(s) for s in seqs], dtype=np.int32)
    width = max(int(lens.max(initial=0)), 1)
    out = np.zeros((len(seqs), width), dtype=np.int32)
    for b, s in enumerate(seqs):
        out[b, :len(s)] = np.asarray(s, dtype=np.int32)
    return torch.from_numpy(out).to(dev), torch.from_numpy(lens).to(dev)


def edit_distance(refs, ref_lens, hyps, hyp_lens):
    """Batched Levenshtein distance with error counts on the GPU.

    refs ``[B, Rmax]`` / hyps ``[B, Hmax]`` CUDA int tensors of token ids (padded), ref_lens / hyp_lens ``[B]``.
    Returns a CUDA int32 tensor ``[B, 4]``: distance, substitutions, insertions, deletions -- the values
    ``compute_wer(ref, hyp)`` of the reference returns for every pair.  No host synchronisation."""
    if not (isinstance(refs, torch.Tensor) and refs.is_cuda and isinstance(hyps, torch.Tensor) and hyps.is_cuda):
        raise B200CTCError("refs and hyps must be CUDA tensors: the evaluation kernels have no CPU path")
    if refs.dim() != 2 or hyps.dim() != 2 or refs.size(0) != hyps.size(0):
        raise B200CTCError("refs and hyps must be [B, Rmax] and [B, Hmax]")
    dev = refs.device
    refs = refs.to(torch.int32).contiguous()
    hyps = hyps.to(device=dev, dtype=torch.int32).contiguous()
    ref_lens = torch.as_tensor(ref_lens).to(device=dev, dtype=torch.int32).contiguous()
    hyp_lens = torch.as_tensor(hyp_lens).to(device=dev, dtype=torch.int32).contiguous()
    B, R, H = refs.size(0), refs.size(1), hyps.size(1)
    if ref_lens.numel() != B or hyp_lens.numel() != B:
        raise B200CTCError("ref_lens and hyp_lens must have one entry per pair")
    lib = _lib.load()
    out = torch.empty((B, 4), dtype=torch.int32, device=dev)
    n = ctypes.c_size_t()
    _lib.check(lib.b200ctc_edit_distance_workspace(B, R, H, ctypes.byref(n)), "b200ctc_edit_distance_workspace")
    with torch.cuda.device(dev):
        ws = torch.empty(max(n.value, 1), dtype=torch.uint8, device=dev)
        st = lib.b200ctc_edit_distance(refs.data_ptr(), refs.stride(0) if B else R, ref_lens.data_ptr(),
                                       hyps.data_ptr(), hyps.stride(0) if B else H, hyp_lens.data_ptr(), B, R, H,
                                       out.data_ptr(), ws.data_ptr(), ws.numel(),
                                       torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(st, "b200ctc_edit_distance")
        ws.record_stream(torch.cuda.current_stream(dev))
    return out


def _rows_i32(x, dev):
    """``[B, L]`` -> (int32 tensor on ``dev`` with contiguous, non-overlapping rows, its row stride).  A row view of a
    wider tensor is kept as it is."""
    x = x.to(device=dev, dtype=torch.int32)
    if (x.size(1) > 1 and x.stride(1) != 1) or (x.size(0) > 1 and x.stride(0) < x.size(1)):
        x = x.contiguous()
    return x, (x.stride(0) if x.size(0) > 1 else x.size(1))


def word_errors(refs, ref_lens, hyps, hyp_lens, space):
    """Word and space-free character error counts of character-level hypotheses for a whole batch, on the GPU.

    refs ``[B, Rmax]`` / hyps ``[B, Hmax]`` CUDA int tensors of token ids (padded; any row stride), ref_lens /
    hyp_lens ``[B]`` tensors or arrays; ``space`` is the word-boundary id in the same id space.  The words of a
    sequence are its maximal runs of tokens other than ``space`` (``str.split()``: leading, trailing and repeated
    spaces make no empty word).  Returns CUDA int32 tensors ``(word_errors[B,4], char_errors[B,4], ref_counts[B,2])``:
    ``compute_wer`` over the words, ``compute_wer`` over both sequences with the spaces removed, and the number of
    reference words and of non-space reference tokens.  WER = ``word_errors[:, 0].sum() / ref_counts[:, 0].sum()``,
    CER = ``char_errors[:, 0].sum() / ref_counts[:, 1].sum()``.  No host synchronisation."""
    if not (isinstance(refs, torch.Tensor) and refs.is_cuda and isinstance(hyps, torch.Tensor) and hyps.is_cuda):
        raise B200CTCError("refs and hyps must be CUDA tensors: the evaluation kernels have no CPU path")
    if refs.dim() != 2 or hyps.dim() != 2 or refs.size(0) != hyps.size(0):
        raise B200CTCError("refs and hyps must be [B, Rmax] and [B, Hmax]")
    if not -2 ** 31 <= int(space) < 2 ** 31:
        raise B200CTCError("space must be an int32 token id")
    dev = refs.device
    (refs, ref_stride), (hyps, hyp_stride) = _rows_i32(refs, dev), _rows_i32(hyps, dev)
    ref_lens = torch.as_tensor(ref_lens).to(device=dev, dtype=torch.int32).contiguous()
    hyp_lens = torch.as_tensor(hyp_lens).to(device=dev, dtype=torch.int32).contiguous()
    B, R, H = refs.size(0), refs.size(1), hyps.size(1)
    if ref_lens.numel() != B or hyp_lens.numel() != B:
        raise B200CTCError("ref_lens and hyp_lens must have one entry per pair")
    lib = _lib.load()
    word4 = torch.empty((B, 4), dtype=torch.int32, device=dev)
    char4 = torch.empty((B, 4), dtype=torch.int32, device=dev)
    counts = torch.empty((B, 2), dtype=torch.int32, device=dev)
    n = ctypes.c_size_t()
    _lib.check(lib.b200ctc_word_errors_workspace(B, R, H, ctypes.byref(n)), "b200ctc_word_errors_workspace")
    with torch.cuda.device(dev):
        ws = torch.empty(max(n.value, 1), dtype=torch.uint8, device=dev)
        st = lib.b200ctc_word_errors(refs.data_ptr(), ref_stride, ref_lens.data_ptr(), hyps.data_ptr(), hyp_stride,
                                     hyp_lens.data_ptr(), B, R, H,
                                     int(space), word4.data_ptr(), char4.data_ptr(), counts.data_ptr(), ws.data_ptr(),
                                     ws.numel(), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(st, "b200ctc_word_errors")
    return word4, char4, counts


def compute_wer(ref, hyp, normalize=False, device="cuda"):
    """Drop-in for ``utils.evaluation.edit_distance.compute_wer`` (:53-126): ``ref`` / ``hyp`` are lists of
    hashable tokens (words, phones, characters).  Returns ``(wer, sub, ins, dele)``."""
    vocab = {}
    r = [vocab.setdefault(t, len(vocab)) for t in ref]
    h = [vocab.setdefault(t, len(vocab)) for t in hyp]
    dev = torch.device(device)
    refs, ref_lens = _padded_i32([r], dev)
    hyps, hyp_lens = _padded_i32([h], dev)
    d, sub, ins, dele = (int(x) for x in edit_distance(refs, ref_lens, hyps, hyp_lens)[0].cpu())
    wer = d / len(ref) if normalize else d
    return wer, sub, ins, dele


def posteriors(logits, temperature=1.0):
    """``softmax(logits / temperature)`` over the last axis in one pass (CTC.posteriors, ctc.py:486).
    logits: CUDA fp32, bfloat16 or float16 ``[B, T, V]`` (any batch / time strides).  Returns a CUDA fp32 tensor
    ``[B, T, V]`` for every input type (the reference hands it to numpy, which has no bfloat16): for 16-bit logits
    exactly ``posteriors(logits.float(), temperature)``."""
    if not isinstance(logits, torch.Tensor) or not logits.is_cuda or logits.dtype not in DTYPES or logits.dim() != 3:
        raise B200CTCError("logits must be a CUDA float32, bfloat16 or float16 tensor [B, T, V]")
    if logits.stride(2) != 1 and logits.size(2) > 1:
        logits = logits.contiguous()
    B, T, V = logits.shape
    out = torch.empty((B, T, V), dtype=torch.float32, device=logits.device)
    with torch.cuda.device(logits.device):
        st = _lib.load().b200ctc_softmax_temperature_typed(logits.data_ptr(), DTYPES[logits.dtype], logits.stride(0),
                                                           logits.stride(1), T, V, B, float(temperature), out.data_ptr(),
                                                           torch.cuda.current_stream(logits.device).cuda_stream)
        _lib.check(st, "b200ctc_softmax_temperature_typed")
    return out


def evaluate_batch(logits, x_lens, ys, y_lens, blank=0, label_offset=1, beam_width=1, lm=None, alpha=0.0, beta=0.0):
    """Decode (greedy for ``beam_width == 1``, else prefix beam search on ``log_softmax(logits)``, the choice
    ``CTC.decode`` makes, ctc.py:435-441) + edit distance for a whole mini-batch, device resident.

    logits ``[B, T, V]`` CUDA, fp32, bfloat16 or float16 (the beam search decodes fp32 log-probabilities of the
    widened logits, as autocast's ``log_softmax`` gives them); ys ``[B, Lmax]`` reference labels WITHOUT the blank offset (as the dataset
    stores them), y_lens ``[B]``.  The hypotheses are shifted by ``-label_offset`` exactly as ``CTC.decode`` does
    (``best_hyps -= 1``, ctc.py:444).  Returns ``(errors[B,4] int32 CUDA, hyp_tokens[B,T], hyp_lens[B])`` with
    errors = (distance, sub, ins, del) per utterance; ``errors.sum(0)`` over a data set divided by
    ``y_lens.sum()`` gives PER / CER and its breakdown (phone.py:119-126), with spaces counted as tokens.  For the
    WER of a character model pass ``ys`` and the returned hypotheses to ``word_errors``.
    With ``lm`` (an ``NGramLM``) every beam width, 1 included, decodes with the LM-fused beam search weighted by
    ``alpha`` and ``beta``; without one they must be 0."""
    if lm is not None:
        tokens, hyp_lens = beam_search_decode(torch.log_softmax(logits, dim=-1, dtype=torch.float32), x_lens, beam_width,
                                              blank, lm=lm, alpha=alpha, beta=beta)
    elif float(alpha) != 0.0 or float(beta) != 0.0:
        raise B200CTCError("alpha and beta weight a language model: pass lm=NGramLM(...)")
    elif int(beam_width) == 1:
        tokens, hyp_lens = greedy_decode(logits, x_lens, blank)
    else:
        tokens, hyp_lens = beam_search_decode(torch.log_softmax(logits, dim=-1, dtype=torch.float32), x_lens, beam_width,
                                              blank)
    hyps = tokens - int(label_offset)                       # padding (-1) becomes more negative: never read
    dev = logits.device
    refs = torch.as_tensor(ys).to(device=dev, dtype=torch.int32)
    if refs.dim() != 2:
        raise B200CTCError("ys must be [B, Lmax]")
    return edit_distance(refs, y_lens, hyps, hyp_lens), hyps, hyp_lens
