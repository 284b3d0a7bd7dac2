"""GPU tests of the batched word-error call: word errors, space-free character errors and reference counts of every
pair equal to the oracle (oracle/word_ref.word_errors on top of compute_wer) on random ragged batches, adversarial
word-identity cases and long pairs; padding, strides, a poisoned workspace and CUDA-graph replay leave the results
unchanged; and evaluate_batch followed by word_errors scores the oracle decoders' hypotheses."""
import ctypes

import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from oracle import beam_lm_ref, beam_ref, ctc_ref, lm_ref, word_ref
from pytorch_end2end_speech_recognition_b200 import _lib

pytestmark = pytest.mark.gpu

S = 0          # the space id of the hand-written cases


def _pad(seqs, pad=None, rng=None, extra=0):
    """list of int sequences -> ([B, Lmax + extra] int32 CUDA tensor, [B] int32 CUDA lengths).  Entries past a length
    are 0, ``pad``, or random ids (``pad == "random"``)."""
    lens = np.array([len(s) for s in seqs], dtype=np.int32)
    width = max(int(lens.max(initial=0)), 1) + extra
    if pad == "random":
        out = rng.randint(-3, 50, size=(len(seqs), width)).astype(np.int32)
    else:
        out = np.full((len(seqs), width), 0 if pad is None else pad, dtype=np.int32)
    for b, s in enumerate(seqs):
        out[b, :len(s)] = np.asarray(s, dtype=np.int32)
    return torch.from_numpy(out).cuda(), torch.from_numpy(lens).cuda()


def _run(refs, hyps, space, **pad):
    r, rl = _pad(refs, **pad)
    h, hl = _pad(hyps, **pad)
    w, c, n = b200.word_errors(r, rl, h, hl, space)
    return w.cpu().numpy(), c.cpu().numpy(), n.cpu().numpy()


def _check(refs, hyps, space):
    w, c, n = _run(refs, hyps, space)
    assert w.shape == (len(refs), 4) and c.shape == (len(refs), 4) and n.shape == (len(refs), 2)
    for b in range(len(refs)):
        got = (tuple(int(x) for x in w[b]), tuple(int(x) for x in c[b]), tuple(int(x) for x in n[b]))
        assert got == word_ref.word_errors(refs[b], hyps[b], space), b
    return w, c, n


def _text(s):
    """'ab c' -> token ids, a = 1, b = 2, ..., ' ' = S."""
    return [S if ch == " " else ord(ch) - ord("a") + 1 for ch in s]


def _edit(rng, seq, p, alphabet):
    """seq with seeded substitutions, insertions and deletions, each at rate p."""
    out = []
    for t in seq:
        u = rng.rand()
        if u < p:
            continue                                              # deletion
        if u < 2 * p:
            out.append(int(rng.choice(alphabet)))                 # substitution
        else:
            out.append(int(t))
        if rng.rand() < p:
            out.append(int(rng.choice(alphabet)))                 # insertion
    return out


def _random_batch(rng, B, space, letters, max_len):
    alphabet = list(letters) + [space]
    refs, hyps = [], []
    for b in range(B):
        n = int(rng.randint(0, max_len + 1))
        ref = [int(t) for t in rng.choice(alphabet, size=n, p=[0.7 / len(letters)] * len(letters) + [0.3])]
        kind = b % 6
        if kind == 1:
            ref = [space] * int(rng.randint(1, 4)) + ref + [space] * int(rng.randint(1, 4))
        elif kind == 2:
            ref = [space] * int(rng.randint(0, 6))                # all spaces, or empty
        hyp = _edit(rng, ref, 0.15, alphabet)
        if kind == 3:
            hyp = [space] * int(rng.randint(0, 6))
        elif kind == 4:
            hyp = [int(t) for t in rng.choice(alphabet, size=int(rng.randint(0, max_len + 1)))]
        refs.append(ref)
        hyps.append(hyp)
    return refs, hyps


@pytest.mark.parametrize("B,space,letters,max_len,seed", [
    (300, 0, (1, 2, 3), 60, 1), (64, 5, (1, 2), 40, 2), (200, 29, tuple(range(1, 29)), 120, 3),
    (7, -4, (0, 1, 2), 30, 4)])
def test_random_ragged_batches_match_the_oracle(B, space, letters, max_len, seed):
    rng = np.random.RandomState(seed)
    refs, hyps = _random_batch(rng, B, space, letters, max_len)
    _check(refs, hyps, space)


def test_adversarial_word_identity():
    cases = [
        ("abc abd abc", "abd abc abc"),                            # equal length, one token apart
        ("ab abc a abcd", "abc ab abcd a"),                        # prefixes
        ("abc bca cab acb", "cab abc bca bac"),                    # permutations of the same tokens
        ("ab " * 500, "ab " * 499 + "ac"),                         # many copies of one word
        ("ab c", "a bc"),                                          # boundaries moved
        ("ab cd ef", "a bcd e f"),
        ("  a  b  ", "a b"),                                       # leading, trailing and repeated spaces
        ("", "a b"), ("a b", ""), ("   ", "  "), ("", ""),
        ("a" * 300, "a" * 299),                                   # one long word
    ]
    _check([_text(r) for r, _ in cases], [_text(h) for _, h in cases], S)


def test_many_distinct_and_repeated_words():
    rng = np.random.RandomState(7)
    vocab = [tuple(int(t) for t in rng.randint(1, 4, size=rng.randint(1, 6))) for _ in range(40)]
    refs, hyps = [], []
    for _ in range(16):
        words = [vocab[i] for i in rng.randint(0, len(vocab), size=200)]
        ref = [t for w in words for t in list(w) + [S]]
        hyp_words = [vocab[int(rng.randint(0, len(vocab)))] if rng.rand() < 0.1 else w for w in words]
        hyps.append([t for w in hyp_words for t in list(w) + [S]])
        refs.append(ref)
    _check(refs, hyps, S)


def test_long_pairs_and_a_space_that_never_occurs():
    rng = np.random.RandomState(11)
    alphabet = [1, 2, 3, 4, 5, 6, S]
    p = [0.14] * 6 + [0.16]
    ref_long = [int(t) for t in rng.choice(alphabet, size=17000, p=p)]
    ref_mid = [int(t) for t in rng.choice(alphabet, size=4000, p=p)]
    refs = [ref_long, ref_mid, ref_mid[:300], [t for t in ref_mid if t != S]]
    hyps = [_edit(rng, ref_long[:200], 0.1, alphabet), _edit(rng, ref_mid[:1000], 0.1, alphabet),
            _edit(rng, ref_mid, 0.1, alphabet)[:3000], _edit(rng, refs[3][:500], 0.1, alphabet)]
    _check(refs, hyps, S)
    _check(refs[2:], hyps[2:], 99)                               # no space: each non-empty sequence is one word


def test_longest_reference_against_itself_with_one_substitution():
    rng = np.random.RandomState(12)
    ref = [int(t) for t in rng.choice([1, 2, 3, 4, 5, S], size=17000, p=[0.16] * 5 + [0.2])]
    ref[0] = ref[-1] = 1
    hyp = list(ref)
    k = next(i for i in range(8000, 17000) if ref[i] != S)
    hyp[k] = 9
    n_words, n_chars = len(word_ref.split_words(ref, S)), sum(t != S for t in ref)
    w, c, n = _run([ref, ref], [ref, hyp], S)
    assert w.tolist() == [[0, 0, 0, 0], [1, 1, 0, 0]]
    assert c.tolist() == [[0, 0, 0, 0], [1, 1, 0, 0]]
    assert n.tolist() == [[n_words, n_chars]] * 2


def test_padding_past_the_lengths_is_never_read():
    rng = np.random.RandomState(13)
    refs, hyps = _random_batch(rng, 50, S, (1, 2, 3), 40)
    base = _run(refs, hyps, S)
    for pad in (S, "random"):
        got = _run(refs, hyps, S, pad=pad, rng=np.random.RandomState(14), extra=9)
        for x, y in zip(base, got):
            assert np.array_equal(x, y)


def test_row_views_of_wider_tensors_give_the_contiguous_results():
    rng = np.random.RandomState(15)
    refs, hyps = _random_batch(rng, 40, S, (1, 2, 3), 50)
    r, rl = _pad(refs)
    h, hl = _pad(hyps)
    base = b200.word_errors(r, rl, h, hl, S)
    wide_r = torch.full((r.size(0), r.size(1) + 11), 7, dtype=torch.int32, device="cuda")
    wide_h = torch.full((h.size(0), h.size(1) + 5), 7, dtype=torch.int32, device="cuda")
    wide_r[:, 3:3 + r.size(1)] = r
    wide_h[:, 2:2 + h.size(1)] = h
    view_r, view_h = wide_r[:, 3:3 + r.size(1)], wide_h[:, 2:2 + h.size(1)]
    assert not view_r.is_contiguous() and not view_h.is_contiguous()
    got = b200.word_errors(view_r, rl, view_h, hl.cpu().numpy(), S)
    for x, y in zip(base, got):
        assert torch.equal(x, y)
    got64 = b200.word_errors(r.long(), rl.cpu(), h.long(), hl, S)             # int64 ids are narrowed
    for x, y in zip(base, got64):
        assert torch.equal(x, y)


def test_poisoned_workspace_gives_the_clean_results():
    rng = np.random.RandomState(16)
    refs, hyps = _random_batch(rng, 96, S, (1, 2), 60)
    r, rl = _pad(refs)
    h, hl = _pad(hyps)
    B, R, H = r.size(0), r.size(1), h.size(1)
    lib = _lib.load()
    n = ctypes.c_size_t()
    assert lib.b200ctc_word_errors_workspace(B, R, H, ctypes.byref(n)) == 0

    def call(ws):
        out = [torch.full((B, 4), -7, dtype=torch.int32, device="cuda"),
               torch.full((B, 4), -7, dtype=torch.int32, device="cuda"),
               torch.full((B, 2), -7, dtype=torch.int32, device="cuda")]
        st = lib.b200ctc_word_errors(r.data_ptr(), R, rl.data_ptr(), h.data_ptr(), H, hl.data_ptr(), B, R, H, S,
                                     out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), ws.data_ptr(), ws.numel(),
                                     torch.cuda.current_stream().cuda_stream)
        assert st == 0
        torch.cuda.synchronize()
        return out

    clean = call(torch.zeros(n.value, dtype=torch.uint8, device="cuda"))
    g = torch.Generator(device="cuda").manual_seed(17)
    poisoned = torch.randint(0, 256, (n.value,), dtype=torch.uint8, device="cuda", generator=g)
    # the last: 4 bytes past a 256-byte boundary and 4 bytes short of the query (any alignment is accepted)
    for ws in (poisoned, poisoned, torch.full((n.value,), 0xff, dtype=torch.uint8, device="cuda"), poisoned[4:]):
        for x, y in zip(clean, call(ws)):
            assert torch.equal(x, y)
    for b in range(B):
        got = tuple(int(x) for x in clean[0][b]), tuple(int(x) for x in clean[1][b]), tuple(int(x) for x in clean[2][b])
        assert got == word_ref.word_errors(refs[b], hyps[b], S)


def test_captured_in_a_cuda_graph_and_replayed():
    rng = np.random.RandomState(18)
    refs, hyps = _random_batch(rng, 64, S, (1, 2, 3), 50)
    r, rl = _pad(refs)
    h, hl = _pad(hyps)
    eager = b200.word_errors(r, rl, h, hl, S)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        b200.word_errors(r, rl, h, hl, S)                                      # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = b200.word_errors(r, rl, h, hl, S)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(eager, static):
        assert torch.equal(x, y)
    # new inputs of the same shape, copied in place: the replay reads them, lengths included
    refs2, hyps2 = _random_batch(np.random.RandomState(19), 64, S, (1, 2, 3), 50)
    r2, rl2 = _pad([x[:r.size(1)] for x in refs2])
    h2, hl2 = _pad([x[:h.size(1)] for x in hyps2])
    r.zero_(); h.zero_()
    r[:, :r2.size(1)].copy_(r2); rl.copy_(rl2)
    h[:, :h2.size(1)].copy_(h2); hl.copy_(hl2)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(b200.word_errors(r, rl, h, hl, S), static):
        assert torch.equal(x, y)


def test_evaluate_batch_then_word_errors(tmp_path):
    """Decode on the device, score words on the device; equal to the oracle decoders' hypotheses scored by the
    oracle.  Label space: 0 .. V - 2 after the blank offset; the space is label 3."""
    rng = np.random.RandomState(20)
    B, T, V, space = 6, 90, 12, 3
    logits = (rng.randn(B, T, V) * 2).astype(np.float32)
    logits[:, :, 0] += 1.0
    logits[:, :, space + 1] += 0.5                                             # frequent spaces
    x_lens = np.array([90, 85, 70, 64, 40, 0])
    y_lens = np.array([30, 25, 22, 20, 12, 0])
    ys = np.zeros((B, 30), np.int64)
    for b in range(B):
        ys[b, :y_lens[b]] = rng.randint(0, V - 1, size=y_lens[b])
    lp_gpu = torch.log_softmax(torch.from_numpy(logits).cuda(), dim=-1, dtype=torch.float32)
    lp = lp_gpu.cpu().numpy()
    symbols = ["_"] + ["t%d" % c for c in range(1, V)]
    path = lm_ref.random_arpa(str(tmp_path / "lm.arpa"), symbols[1:-1], 3, 21, per_order=150)
    lm = b200.NGramLM(path, symbols)
    ref_lm = lm_ref.ArpaLM(path, symbols)
    oracle_hyps = {
        "greedy": ctc_ref.greedy_decode(logits, x_lens),
        "beam": [beam_ref.beam_search(lp[b], x_lens[b], 10)[0] for b in range(B)],
        "lm": [beam_lm_ref.beam_search(lp[b], x_lens[b], 10, lm=ref_lm, alpha=0.8, beta=0.5)[0] for b in range(B)],
    }
    runs = {"greedy": dict(beam_width=1), "beam": dict(beam_width=10),
            "lm": dict(beam_width=10, lm=lm, alpha=0.8, beta=0.5)}
    for name, kw in runs.items():
        _, hyps, hyp_lens = b200.evaluate_batch(torch.from_numpy(logits).cuda(), x_lens, ys, y_lens, **kw)
        w, c, n = (x.cpu().numpy() for x in b200.word_errors(torch.as_tensor(ys).cuda(), y_lens, hyps, hyp_lens,
                                                              space=space))
        for b in range(B):
            h = [int(t) - 1 for t in oracle_hyps[name][b]]
            got = tuple(int(x) for x in w[b]), tuple(int(x) for x in c[b]), tuple(int(x) for x in n[b])
            assert got == word_ref.word_errors(list(ys[b, :y_lens[b]]), h, space), (name, b)
    lm.close()
