"""Host-side tests of the n-gram LM fusion: the ABI symbols, the ARPA loader's rejections (before any CUDA call, so
on a machine without a GPU too), the oracle's LM against hand-computed values, and the LM-fused oracle search against
an exhaustive argmax over label sequences."""
import ctypes
import itertools

import numpy as np
import pytest

from oracle import beam_lm_ref, beam_ref, ctc_ref, lm_ref
from oracle.lm_ref import LN10
import pytorch_end2end_speech_recognition_b200 as b200
from pytorch_end2end_speech_recognition_b200 import _lib

NEW_SYMBOLS = ("b200ctc_ngram_lm_create", "b200ctc_ngram_lm_destroy", "b200ctc_ngram_lm_info",
               "b200ctc_beam_search_lm_workspace", "b200ctc_beam_search_lm")

# order 3; <unk>; "a zz" names a word no symbol maps to (dropped by the loader: 6 / 4 / 2 n-grams kept)
HAND_ARPA = """\\data\\
ngram 1=7
ngram 2=5
ngram 3=2

\\1-grams:
-1.0 </s>
-99 <s> -0.5
-0.7 a -0.3
-0.9 b -0.2
-1.1 c
-1.5 <unk>
-2.0 zz -0.1

\\2-grams:
-0.4 <s> a -0.25
-0.6 a b -0.15
-0.8 b a
-0.3 a zz
-0.5 a </s>

\\3-grams:
-0.2 <s> a b
-0.35 a b a

\\end\\
"""
HAND_SYMBOLS = ["_", "a", "b", "c", "d"]      # blank 0; "d" is not a unigram: <unk>


def _create(path, symbols, blank=0):
    lib = _lib.load()
    arr = (ctypes.c_char_p * len(symbols))(*[None if s is None else s.encode() for s in symbols])
    h = ctypes.c_void_p()
    st = lib.b200ctc_ngram_lm_create(str(path).encode(), arr, len(symbols), blank, 0, ctypes.byref(h))
    if st == 0:
        lib.b200ctc_ngram_lm_destroy(h)
    return st


def test_new_symbols_are_exported_and_declared():
    lib = _lib.load()
    for sym in NEW_SYMBOLS:
        assert sym in _lib.EXPORTED_SYMBOLS
        assert getattr(lib, sym).restype is ctypes.c_int and getattr(lib, sym).argtypes
    assert b200.NGramLM is not None
    n = ctypes.c_size_t()
    assert lib.b200ctc_beam_search_lm_workspace(4, 100, 30, 10, ctypes.byref(n)) == 0 and n.value > 0
    assert lib.b200ctc_beam_search_lm_workspace(4, 100, 30, 65, ctypes.byref(n)) == 1
    # no LM: rejected before anything else
    assert lib.b200ctc_beam_search_lm(None, 0, 0, 0, None, 10, 30, 1, 0, 4, None, 1.0, 0.0, None, None, None, None, 0,
                                      None) == 1
    assert lib.b200ctc_ngram_lm_info(None, ctypes.byref(ctypes.c_int()), (ctypes.c_longlong * 8)()) == 1


def _bad_files():
    ok = HAND_ARPA
    yield "no_data_header", ok.replace("\\data\\\n", "")
    yield "bad_header_line", ok.replace("ngram 2=5", "ngram 2 5")
    yield "count_mismatch", ok.replace("ngram 2=5", "ngram 2=6")
    yield "count_mismatch_short", ok.replace("ngram 3=2", "ngram 3=1")
    yield "missing_history", ok.replace("-0.35 a b a", "-0.35 b b a")
    yield "missing_bos", ok.replace("-99 <s> -0.5\n", "").replace("ngram 1=7", "ngram 1=6").replace(
        "-0.4 <s> a -0.25\n", "").replace("-0.2 <s> a b\n", "").replace("ngram 2=5", "ngram 2=4").replace(
        "ngram 3=2", "ngram 3=1")
    yield "missing_eos", ok.replace("-1.0 </s>\n", "").replace("ngram 1=7", "ngram 1=6").replace(
        "-0.5 a </s>\n", "").replace("ngram 2=5", "ngram 2=4")
    yield "uncovered_symbol", ok.replace("-1.5 <unk>\n", "").replace("ngram 1=7", "ngram 1=6")
    yield "order_above_8", ok.replace("ngram 3=2\n", "ngram 3=2\nngram 4=0\nngram 5=0\nngram 6=0\nngram 7=0\n"
                                                     "ngram 8=0\nngram 9=0\n")
    yield "bad_number", ok.replace("-0.9 b -0.2", "-0.9x b -0.2")
    yield "duplicate_ngram", ok.replace("-0.8 b a\n", "-0.8 a b\n")
    yield "no_end", ok.replace("\\end\\", "")


@pytest.mark.parametrize("name,text", list(_bad_files()))
def test_loader_rejects_malformed_files(tmp_path, name, text):
    p = tmp_path / (name + ".arpa")
    p.write_text(text)
    assert _create(p, HAND_SYMBOLS) == 1, name          # B200CTC_STATUS_INVALID_VALUE, with or without a GPU
    with pytest.raises(b200.B200CTCError, match="invalid value"):
        b200.NGramLM(str(p), HAND_SYMBOLS)


def test_loader_rejects_bad_symbols(tmp_path):
    p = tmp_path / "lm.arpa"
    p.write_text(HAND_ARPA)
    assert _create(p, HAND_SYMBOLS) != 1                 # the file itself is valid: 0 with a GPU, 2 without
    assert _create(p, ["_", "a", "b", "a"]) == 1         # duplicate symbols
    assert _create(p, ["_", "a", "<s>"]) == 1
    assert _create(p, ["_", "a", "</s>"]) == 1
    assert _create(p, ["_", "a", None]) == 1             # a non-blank symbol without a string
    assert _create(p, [None, "a", "b"], blank=0) != 1     # the blank's entry is not read
    assert _create(tmp_path / "missing.arpa", HAND_SYMBOLS) == 1


def test_oracle_lm_matches_hand_computed_values(tmp_path):
    p = tmp_path / "lm.arpa"
    p.write_text(HAND_ARPA)
    lm = lm_ref.ArpaLM(str(p), HAND_SYMBOLS)
    a, b, c, d = 1, 2, 3, 4
    assert lm.order == 3 and lm.words[d] == "<unk>"
    assert lm.log_prob([a], b) == -0.2 * LN10                              # "<s> a b"
    assert lm.log_prob([a], c) == (-0.25 + (-0.3 + -1.1)) * LN10            # backs off through two levels
    assert lm.log_prob([a, c], b) == (0.0 + -0.9) * LN10                   # "a c" is no n-gram: bo 0
    assert lm.log_prob([], d) == (-0.5 + -1.5) * LN10                       # <unk>
    assert lm.log_prob([a], lm_ref.EOS) == (-0.25 + -0.5) * LN10            # end of sentence
    assert lm.log_prob([b, a, b], a) == -0.35 * LN10                        # the history is the last two words
    assert lm.log_prob([c, b], a) == (0.0 + -0.8) * LN10                   # "c b" is no n-gram, "b a" is
    assert lm.score([a, b], 2.0, -0.5) == (0.0 + (2.0 * (-0.4 * LN10) + -0.5)) + (2.0 * (-0.2 * LN10) + -0.5)


def _ctc_log_prob(lp, y, blank):
    cost, _ = ctc_ref.ctc_cost_and_grad_single(lp, np.asarray(y, dtype=np.int64), blank)
    return -cost


@pytest.mark.parametrize("seed", range(12))
def test_oracle_search_is_the_argmax_over_all_label_sequences(tmp_path, seed):
    """With a beam wider than the number of reachable prefixes nothing is pruned, so the fused search must return
    argmax_y ln P_ctc(y|x) + S(y) + alpha * lnP(</s> | y) over every label sequence."""
    rng = np.random.RandomState(seed)
    T, V = int(rng.randint(1, 6)), int(rng.randint(2, 5))
    blank = int(rng.randint(V))
    symbols = ["w%d" % c for c in range(V)]
    order = int(rng.randint(1, 4))
    path = lm_ref.random_arpa(str(tmp_path / "lm.arpa"), [s for c, s in enumerate(symbols) if c != blank][:-1] or
                              symbols[:1], order, seed, per_order=30)
    lm = lm_ref.ArpaLM(path, symbols, blank)
    alpha, beta = float(rng.uniform(0.2, 2.0)), float(rng.uniform(-1.0, 1.0))
    x = rng.randn(T, V) * 1.5
    lp = x - np.log(np.exp(x).sum(axis=1, keepdims=True))
    hyp, score = beam_lm_ref.beam_search(lp, T, 10 ** 4, blank=blank, lm=lm, alpha=alpha, beta=beta)
    labels = [c for c in range(V) if c != blank]
    best, best_y = -np.inf, None
    for L in range(T + 1):
        for y in itertools.product(labels, repeat=L):
            if L + ctc_ref.count_repeats(y) > T:
                continue
            f = _ctc_log_prob(lp, y, blank) + lm.score(list(y), alpha, beta) + alpha * lm.log_prob(list(y), lm_ref.EOS)
            if f > best:
                best, best_y = f, list(y)
    assert hyp == best_y
    assert abs(score - best) < 1e-9 * max(1.0, abs(best))


def test_without_an_lm_alpha_and_beta_must_be_zero():
    with pytest.raises(b200.B200CTCError):
        b200.beam_search_decode(np.zeros((1, 2, 3), np.float32), [2], 2, alpha=0.5)
    with pytest.raises(b200.B200CTCError):
        b200.evaluate_batch(None, [2], np.zeros((1, 1)), [1], beta=1.0)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_with_zero_weights_is_the_lm_free_oracle(tmp_path, seed):
    rng = np.random.RandomState(100 + seed)
    T, V, W = int(rng.randint(5, 30)), int(rng.randint(3, 9)), int(rng.randint(1, 12))
    blank = int(rng.randint(V))
    symbols = ["w%d" % c for c in range(V)]
    path = lm_ref.random_arpa(str(tmp_path / "lm.arpa"), [s for c, s in enumerate(symbols) if c != blank], 3, seed)
    x = rng.randn(T, V) * 2.0
    lp = x - np.log(np.exp(x).sum(axis=1, keepdims=True))
    plain = beam_ref.beam_search(lp, T, W, blank=blank)
    assert beam_lm_ref.beam_search(lp, T, W, blank=blank) == plain
    assert beam_lm_ref.beam_search(lp, T, W, blank=blank, lm=lm_ref.ArpaLM(path, symbols, blank)) == plain
