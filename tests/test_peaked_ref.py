"""The peaked-posterior generator and the range-check predictor of oracle/peaked_ref.py (CPU)."""
import itertools
from itertools import groupby

import numpy as np
import pytest

from oracle import ctc_ref, peaked_ref


def collapse(path, blank=0):
    return [k for k, _ in groupby(path.tolist()) if k != blank]


@pytest.mark.parametrize("L,T", [(0, 5), (1, 1), (3, 3), (5, 40), (12, 14), (40, 300)])
def test_alignments_are_valid(L, T):
    rng = np.random.RandomState(L * 100 + T)
    for rep in range(20):
        lab = rng.randint(1, 4, size=L)                  # three symbols: many repeats
        if L + ctc_ref.count_repeats(lab) > T:
            with pytest.raises(ValueError):
                peaked_ref.alignment(rng, lab, T)
            continue
        path = peaked_ref.alignment(rng, lab, T)
        assert path.shape == (T,)
        assert collapse(path) == lab.tolist()            # durations >= 1, a blank between equal labels


def test_alignments_are_uniform():
    """Every alignment of [1, 1, 2] over 7 frames equally likely (chi-square, fixed seed)."""
    lab, T = np.array([1, 1, 2]), 7
    every = [p for p in itertools.product((0, 1, 2), repeat=T) if collapse(np.array(p)) == [1, 1, 2]]
    index = {p: i for i, p in enumerate(every)}
    rng = np.random.RandomState(5)
    n = 200 * len(every)
    counts = np.zeros(len(every))
    for _ in range(n):
        counts[index[tuple(peaked_ref.alignment(rng, lab, T).tolist())]] += 1
    expected = n / len(every)
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    assert chi2 < len(every) + 5 * np.sqrt(2 * len(every)), chi2


def test_peaked_case_follows_its_target():
    rng = np.random.RandomState(3)
    T, V = 400, 30
    lab = rng.randint(1, V, size=70)
    acts, target = peaked_ref.peaked_case(rng, T, lab, V, margin=40.0, noise=0.5, err_rate=0.2, err_run=2)
    assert acts.dtype == np.float32 and acts.shape == (T, V)
    assert np.array_equal(acts.argmax(axis=1), target)
    rng2 = np.random.RandomState(3)
    rng2.randint(1, V, size=70)
    aligned = peaked_ref.alignment(rng2, lab, T)
    wrong = target != aligned
    assert collapse(aligned) == lab.tolist()
    assert 0.1 < wrong.mean() < 0.3
    assert np.all(target[wrong] != 0)                    # errors emit non-blank symbols
    clean = peaked_ref.peaked_case(np.random.RandomState(4), T, lab, V, 40.0, 0.5, 0.0, 2)[1]
    assert collapse(clean) == lab.tolist()


def test_predicted_range_bounds_every_posterior():
    """max(lane) * max(lane) >= alpha * beta' of any state of the lane: the prediction is at least log2 of the
    largest state posterior of a phase-2 frame, and that is close to 0 for a confident alignment."""
    rng = np.random.RandomState(6)
    lab = rng.randint(1, 30, size=40)
    for acts in (rng.randn(150, 30).astype(np.float32),
                 peaked_ref.peaked_case(rng, 150, lab, 30, 20.0, 1.0, 0.0, 1)[0]):
        lp = ctc_ref.log_softmax(acts.astype(np.float64), axis=1)
        ext = ctc_ref.extended_labels(lab)
        a, b, em = ctc_ref._alpha_beta(lp, ext, 0)
        ll = np.logaddexp(a[-1, -1], a[-1, -2])
        post_bits = np.max(a + b - em - ll) / np.log(2)
        bits = peaked_ref.predicted_range_bits(acts, lab)
        assert bits >= post_bits - 1e-9
        assert bits < 40
    assert peaked_ref.predicted_range_bits(acts, lab) < 1.0   # the confident one


def test_predicted_range_is_a_property_of_the_softmax():
    rng = np.random.RandomState(7)
    lab = rng.randint(1, 30, size=50)
    acts, _ = peaked_ref.peaked_case(rng, 200, lab, 30, 58.0, 0.5, 0.2, 2)
    bits = peaked_ref.predicted_range_bits(acts, lab)
    shifted = acts + rng.randn(200, 1).astype(np.float32) * 10          # row constants: same softmax
    assert abs(peaked_ref.predicted_range_bits(shifted, lab) - bits) < 1e-3
    scaled = acts * np.float32(0.5)
    assert peaked_ref.predicted_range_bits(acts, lab, logit_scale=0.5) == peaked_ref.predicted_range_bits(scaled, lab)
    assert peaked_ref.predicted_range_bits(acts[:30], lab) == -np.inf                   # infeasible


def test_misrecognised_stretches_reach_the_redo_class():
    """Recognition errors are what drives the range: the same labels and margin stay far below the threshold without
    errors and, in some of the seeds, pass it by 24 bits with them."""
    V, T, L = 30, 300, 80
    clean, errs = [], []
    for seed in range(6):
        for err, out in ((0.0, clean), (0.2, errs)):
            rng = np.random.RandomState(seed)
            lab = rng.randint(1, V, size=L)
            acts, _ = peaked_ref.peaked_case(rng, T, lab, V, 58.0, 0.5, err, 2)
            out.append(peaked_ref.predicted_range_bits(acts, lab))
    assert all(peaked_ref.range_class(b) == "must-stay-fast" for b in clean)
    assert any(peaked_ref.range_class(b) == "must-redo" for b in errs)


def test_range_classes():
    assert peaked_ref.range_class(peaked_ref.MUST_REDO_BITS) == "must-redo"
    assert peaked_ref.range_class(peaked_ref.MUST_STAY_FAST_BITS) == "must-stay-fast"
    assert peaked_ref.range_class(peaked_ref.LOST_BOUND_BITS) == "grey"
    assert peaked_ref.range_class(-np.inf) == "must-stay-fast"
