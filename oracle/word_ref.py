"""CPU oracle for the batched word-error kernel: word and space-free character errors of character-level sequences.

TEST INFRASTRUCTURE ONLY (see oracle/ctc_ref.py): only tests/ may import it.

States the word rule on top of ``eval_ref.compute_wer`` (pinned to the reference's own function by
tests/golden/edit_distance_golden.npz): the words of a sequence are its maximal non-empty runs of tokens other than
``space`` (python's ``str.split()``, not ``str.split(sep)``: leading, trailing and repeated spaces make no empty
word), compared as tuples, so two words are equal exactly when they have the same tokens.
"""

from .eval_ref import compute_wer


def split_words(seq, space):
    """Maximal non-empty runs of tokens other than ``space``, as tuples of ints, in order."""
    words, cur = [], []
    for t in seq:
        if int(t) == space:
            if cur:
                words.append(tuple(cur))
            cur = []
        else:
            cur.append(int(t))
    if cur:
        words.append(tuple(cur))
    return words


def word_errors(ref, hyp, space):
    """(compute_wer over the words, compute_wer over the sequences without ``space``,
    (number of reference words, number of non-space reference tokens))."""
    ref_words, hyp_words = split_words(ref, space), split_words(hyp, space)
    ref_chars = [int(t) for t in ref if int(t) != space]
    hyp_chars = [int(t) for t in hyp if int(t) != space]
    return compute_wer(ref_words, hyp_words), compute_wer(ref_chars, hyp_chars), (len(ref_words), len(ref_chars))
