"""GPU tests of the prefix beam search with an n-gram language model fused in: tokens, lengths and fp32 scores equal
to the LM-fused oracle (oracle/beam_lm_ref.py with oracle/lm_ref.py) on random history-closed ARPA files of orders 1-6
and on a model counted from a corpus, the LM-free results at alpha = beta = 0, the 16-bit and strided inputs, the
decoder class and evaluate_batch, and the rejections."""
import os

import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from oracle import beam_lm_ref, beam_ref, eval_ref, lm_ref

pytestmark = pytest.mark.gpu


def _symbols(V, blank):
    return ["_" if c == blank else "t%d" % c for c in range(V)]


def _random_lm(tmp_path, V, blank, order, seed, per_order=150):
    """Symbols t1.. of the vocabulary, all but the last as unigrams (the last maps to <unk>)."""
    symbols = _symbols(V, blank)
    words = [s for c, s in enumerate(symbols) if c != blank]
    path = lm_ref.random_arpa(str(tmp_path / ("lm%d_%d.arpa" % (order, seed))), words[:-1] or words, order, seed,
                              per_order=per_order)
    return path, symbols


def _log_probs(rng, B, T, V, blank, scale=2.0):
    logits = (rng.randn(B, T, V) * scale).astype(np.float32)
    logits[:, :, blank] += 1.0
    return torch.log_softmax(torch.from_numpy(logits), dim=-1)


def _check_against_oracle(lp, x_lens, W, blank, lm, ref_lm, alpha, beta):
    tokens, lens, scores = b200.beam_search_decode(lp.cuda(), x_lens, W, blank=blank, return_scores=True, lm=lm,
                                                   alpha=alpha, beta=beta)
    tokens, lens, scores = tokens.cpu().numpy(), lens.cpu().numpy(), scores.cpu().numpy()
    for b in range(lp.shape[0]):
        hyp, score = beam_lm_ref.beam_search(lp[b].numpy(), x_lens[b], W, blank=blank, lm=ref_lm, alpha=alpha, beta=beta)
        assert list(tokens[b, :lens[b]]) == hyp, b
        assert np.all(tokens[b, lens[b]:] == -1)
        assert scores[b] == np.float32(score), (b, scores[b], score)


@pytest.mark.parametrize("B,T,V,W,blank,order", [
    (3, 20, 4, 1, 0, 1), (3, 24, 6, 4, 2, 2), (4, 30, 12, 10, 0, 3), (2, 16, 30, 16, 5, 4), (2, 10, 62, 10, 0, 5),
    (2, 8, 200, 64, 0, 6), (2, 14, 5, 64, 4, 3), (3, 12, 40, 33, 0, 2)])
def test_fused_search_matches_the_oracle(tmp_path, B, T, V, W, blank, order):
    rng = np.random.RandomState(B * 1000 + T * 10 + V + W + order)
    path, symbols = _random_lm(tmp_path, V, blank, order, seed=V + order)
    lm = b200.NGramLM(path, symbols, blank=blank)
    ref_lm = lm_ref.ArpaLM(path, symbols, blank)
    assert lm.order == order and len(lm.counts) == order
    lp = _log_probs(rng, B, T, V, blank)
    x_lens = rng.randint(T // 2, T + 1, size=B)
    x_lens[-1] = 0                                        # an empty utterance: only the end of sentence is scored
    for alpha, beta in [(0.5, 1.0), (1.5, -0.75), (0.3, 0.0)]:
        _check_against_oracle(lp, x_lens, W, blank, lm, ref_lm, alpha, beta)
    lm.close()


def test_counted_lm_matches_the_oracle(tmp_path):
    rng = np.random.RandomState(11)
    V, blank = 9, 0
    symbols = _symbols(V, blank)
    corpus = [[symbols[c] for c in rng.randint(1, V, size=rng.randint(3, 12))] for _ in range(300)]
    path = lm_ref.counted_arpa(str(tmp_path / "counted.arpa"), corpus, 3)
    lm = b200.NGramLM(path, symbols)
    ref_lm = lm_ref.ArpaLM(path, symbols)
    lp = _log_probs(rng, 4, 40, V, blank)
    x_lens = np.array([40, 35, 22, 40])
    for alpha, beta in [(0.8, 0.5), (2.0, -1.0)]:
        _check_against_oracle(lp, x_lens, 10, blank, lm, ref_lm, alpha, beta)


def test_loader_counts_drop_unmapped_ngrams(tmp_path):
    from test_lm_host import HAND_ARPA, HAND_SYMBOLS
    p = tmp_path / "hand.arpa"
    p.write_text(HAND_ARPA)
    lm = b200.NGramLM(str(p), HAND_SYMBOLS)
    assert lm.order == 3 and lm.counts == [6, 4, 2]
    ref_lm = lm_ref.ArpaLM(str(p), HAND_SYMBOLS)
    rng = np.random.RandomState(3)
    lp = _log_probs(rng, 3, 15, 5, 0)
    _check_against_oracle(lp, np.array([15, 9, 12]), 6, 0, lm, ref_lm, 1.2, 0.4)


def test_zero_weights_reproduce_the_lm_free_search(golden_dir, tmp_path):
    z = np.load(os.path.join(golden_dir, "beam_golden.npz"))
    lms = {}
    for i in range(int(z["n_cases"])):
        lp, x_lens, W = z["log_probs_%d" % i], z["x_lens_%d" % i], int(z["beam_%d" % i])
        V = lp.shape[2]
        if V not in lms:
            path, symbols = _random_lm(tmp_path, V, 0, 3, seed=V)
            lms[V] = b200.NGramLM(path, symbols)
        tokens, lens = b200.beam_search_decode(torch.from_numpy(lp).cuda(), x_lens, W, lm=lms[V], alpha=0.0, beta=0.0)
        tokens, lens = tokens.cpu().numpy(), lens.cpu().numpy()
        assert np.array_equal(lens, z["hyp_lens_%d" % i]), i
        offs = np.concatenate([[0], np.cumsum(lens)])
        for b in range(lp.shape[0]):
            assert np.array_equal(tokens[b, :lens[b]], z["hyp_flat_%d" % i][offs[b]:offs[b + 1]]), (i, b)
    rng = np.random.RandomState(21)
    V, blank = 30, 3
    path, symbols = _random_lm(tmp_path, V, blank, 4, seed=77)
    lm = b200.NGramLM(path, symbols, blank=blank)
    lp = _log_probs(rng, 4, 45, V, blank)
    x_lens = np.array([45, 40, 0, 31])
    tokens, lens, scores = b200.beam_search_decode(lp.cuda(), x_lens, 10, blank=blank, return_scores=True, lm=lm)
    tokens, lens, scores = tokens.cpu().numpy(), lens.cpu().numpy(), scores.cpu().numpy()
    for b in range(4):
        hyp, score = beam_ref.beam_search(lp[b].numpy(), x_lens[b], 10, blank=blank)
        assert list(tokens[b, :lens[b]]) == hyp
        assert scores[b] == np.float32(score)


def test_16_bit_and_strided_inputs_give_the_fp32_result(tmp_path):
    rng = np.random.RandomState(8)
    B, T, V, blank = 3, 40, 30, 0
    path, symbols = _random_lm(tmp_path, V, blank, 3, seed=5)
    lm = b200.NGramLM(path, symbols)
    lp = _log_probs(rng, B, T, V, blank).cuda()
    x_lens = np.array([40, 33, 27])
    for dt in (torch.bfloat16, torch.float16):
        low = lp.to(dt)
        t1, l1, s1 = b200.beam_search_decode(low, x_lens, 8, return_scores=True, lm=lm, alpha=0.7, beta=0.3)
        t2, l2, s2 = b200.beam_search_decode(low.float(), x_lens, 8, return_scores=True, lm=lm, alpha=0.7, beta=0.3)
        assert torch.equal(t1, t2) and torch.equal(l1, l2) and torch.equal(s1, s2)
    tm = lp.transpose(0, 1).contiguous().transpose(0, 1)   # time-major storage, [B, T, V] view
    t1, l1, s1 = b200.beam_search_decode(tm, x_lens, 8, return_scores=True, lm=lm, alpha=0.7, beta=0.3)
    t2, l2, s2 = b200.beam_search_decode(lp, x_lens, 8, return_scores=True, lm=lm, alpha=0.7, beta=0.3)
    assert torch.equal(t1, t2) and torch.equal(l1, l2) and torch.equal(s1, s2)


def test_decoder_class_and_evaluate_batch(tmp_path):
    rng = np.random.RandomState(9)
    B, T, V = 4, 50, 12
    path, symbols = _random_lm(tmp_path, V, 0, 3, seed=12)
    lm = b200.NGramLM(path, symbols)
    ref_lm = lm_ref.ArpaLM(path, symbols)
    logits = (rng.randn(B, T, V) * 2).astype(np.float32)
    logits[:, :, 0] += 1.0
    x_lens = np.array([50, 44, 40, 33])
    lp = torch.log_softmax(torch.from_numpy(logits).cuda(), dim=-1).cpu().numpy()
    hyps = b200.BeamSearchDecoder(blank_index=0, lm=lm)(lp, x_lens, beam_width=5, alpha=0.9, beta=0.6)
    for b in range(B):
        assert list(hyps[b]) == beam_lm_ref.beam_search(lp[b], x_lens[b], 5, lm=ref_lm, alpha=0.9, beta=0.6)[0]
    y_lens = np.array([12, 9, 10, 7])
    ys = np.zeros((B, 12), np.int64)
    for b in range(B):
        ys[b, :y_lens[b]] = rng.randint(0, V - 1, size=y_lens[b])
    for W in (1, 5):
        errors, hyp_t, hyp_lens = b200.evaluate_batch(torch.from_numpy(logits).cuda(), x_lens, ys, y_lens, beam_width=W,
                                                      lm=lm, alpha=0.9, beta=0.6)
        errors, hyp_t, hyp_lens = errors.cpu().numpy(), hyp_t.cpu().numpy(), hyp_lens.cpu().numpy()
        for b in range(B):
            h = np.asarray(beam_lm_ref.beam_search(lp[b], x_lens[b], W, lm=ref_lm, alpha=0.9, beta=0.6)[0], np.int64) - 1
            assert np.array_equal(hyp_t[b, :hyp_lens[b]], h)
            assert tuple(errors[b]) == eval_ref.compute_wer(list(ys[b, :y_lens[b]]), list(h))


def test_a_strong_lm_changes_an_ambiguous_hypothesis(tmp_path):
    p = tmp_path / "prefer_b.arpa"
    p.write_text("\\data\\\nngram 1=4\n\n\\1-grams:\n-99 <s>\n-0.5 </s>\n-3.0 a\n-0.1 b\n\n\\end\\\n")
    symbols = ["_", "a", "b"]
    lm = b200.NGramLM(str(p), symbols)
    ref_lm = lm_ref.ArpaLM(str(p), symbols)
    lp = torch.log(torch.tensor([[[0.1, 0.46, 0.44]]], dtype=torch.float32))
    plain, _ = b200.beam_search_decode(lp.cuda(), [1], 3)
    fused, fused_len = b200.beam_search_decode(lp.cuda(), [1], 3, lm=lm, alpha=1.0, beta=0.0)
    assert plain[0, 0].item() == 1 and fused[0, 0].item() == 2 and fused_len[0].item() == 1
    assert beam_lm_ref.beam_search(lp[0].numpy(), 1, 3, lm=ref_lm, alpha=1.0)[0] == [2]


def test_mismatched_lm_is_rejected(tmp_path):
    path, symbols = _random_lm(tmp_path, 8, 0, 2, seed=1)
    lm = b200.NGramLM(path, symbols)
    lp = _log_probs(np.random.RandomState(0), 2, 10, 8, 0).cuda()
    with pytest.raises(b200.B200CTCError):
        b200.beam_search_decode(lp[:, :, :7], [10, 10], 4, lm=lm, alpha=1.0)      # V
    with pytest.raises(b200.B200CTCError):
        b200.beam_search_decode(lp, [10, 10], 4, blank=1, lm=lm, alpha=1.0)       # blank
    with pytest.raises(b200.B200CTCError):
        b200.beam_search_decode(lp, [10, 10], 4, lm=lm, alpha=float("nan"))
    with pytest.raises(b200.B200CTCError):
        b200.beam_search_decode(lp, [10, 10], 4, lm=lm, beta=float("inf"))
    if torch.cuda.device_count() > 1:
        with pytest.raises(b200.B200CTCError):
            b200.beam_search_decode(lp.to("cuda:1"), [10, 10], 4, lm=lm, alpha=1.0)   # another device
    lm.close()
    with pytest.raises(b200.B200CTCError):
        b200.beam_search_decode(lp, [10, 10], 4, lm=lm, alpha=1.0)                # closed


def test_unaligned_workspace_gives_the_aligned_results(tmp_path):
    """A C caller's workspace may have any alignment: the beam search, with and without the LM, called with the
    queried workspace shifted by 4 bytes (and 4 bytes shorter) gives the tokens, lengths and scores of the call
    with a 256-byte aligned one."""
    import ctypes
    from pytorch_end2end_speech_recognition_b200 import _lib
    lib = _lib.load()
    B, T, V, W = 3, 24, 12, 8
    rng = np.random.RandomState(11)
    path, symbols = _random_lm(tmp_path, V, 0, 3, seed=5)
    lm = b200.NGramLM(path, symbols)
    lp = _log_probs(rng, B, T, V, 0).cuda()
    lens = torch.tensor([T, T - 5, 9], dtype=torch.int32, device="cuda")

    def run(with_lm, shift):
        n = ctypes.c_size_t()
        query = lib.b200ctc_beam_search_lm_workspace if with_lm else lib.b200ctc_beam_search_workspace
        assert query(B, T, V, W, ctypes.byref(n)) == 0
        ws = torch.empty(n.value + 256, dtype=torch.uint8, device="cuda")
        ptr, nbytes = ws.data_ptr() + shift, n.value - shift
        assert ws.data_ptr() % 256 == 0
        tokens = torch.empty((B, T), dtype=torch.int32, device="cuda")
        out_lens = torch.empty(B, dtype=torch.int32, device="cuda")
        scores = torch.empty(B, dtype=torch.float32, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream
        if with_lm:
            st = lib.b200ctc_beam_search_lm(lp.data_ptr(), 0, lp.stride(0), lp.stride(1), lens.data_ptr(), T, V, B, 0, W,
                                            lm.handle, 0.8, 0.5, tokens.data_ptr(), out_lens.data_ptr(),
                                            scores.data_ptr(), ptr, nbytes, stream)
        else:
            st = lib.b200ctc_beam_search_typed(lp.data_ptr(), 0, lp.stride(0), lp.stride(1), lens.data_ptr(), T, V, B, 0,
                                               W, tokens.data_ptr(), out_lens.data_ptr(), scores.data_ptr(), ptr, nbytes,
                                               stream)
        assert st == 0
        torch.cuda.synchronize()
        return tokens.cpu(), out_lens.cpu(), scores.cpu()

    for with_lm in (False, True):
        aligned, shifted = run(with_lm, 0), run(with_lm, 4)
        for a, s in zip(aligned, shifted):
            assert torch.equal(a, s), with_lm
    lm.close()
