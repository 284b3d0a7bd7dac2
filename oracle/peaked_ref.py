"""Peaked posteriors: inputs shaped like the output of a trained acoustic model, and a prediction of the fast
lattice's range check on them.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package may import this module.

A trained model puts probability near one on the aligned symbol of every frame and e^-20 .. e^-60 on the others.
Where it misrecognises a stretch of frames, the forward and backward sweeps disagree about where the alignment is,
and the fast lattice's range check (lattice_fast.cuh, ``posterior_frame``) may find that a state which lost bits
could carry posterior mass; the utterance is then redone by the fp64 safe lattice (FLAG_PRECISION_LOST).
``predicted_range_bits`` evaluates the quantity that check bounds, in fp64 from the oracle's alpha / beta, so
that a test can state in advance which inputs must be redone and which must stay on the fast path.
"""

import numpy as np

from . import ctc_ref

# The range check flags an utterance when, for some phase-2 frame and lane,
#   max(fresh values of the lane) * max(stored values of the opposite side's lane) / P  >  about 2^86
# (lattice_fast.cuh: kLostBound = 127 + 110 - 24 - 2 on the biased exponent fields).  The kernel evaluates it on
# exponent fields -- the mantissas of the two maxima and of P are dropped -- so its value lies within 3 bits of
# the fp64 one; the classes below keep 24 bits away from the threshold on either side.
LOST_BOUND_BITS = 86
MUST_REDO_BITS = LOST_BOUND_BITS + 24
MUST_STAY_FAST_BITS = LOST_BOUND_BITS - 24
LANE_STATES = 8          # lattice states per lane of the fast lattice
WINDOW_MAX_L = 120       # one lattice window (256 states, less the halo) holds 2L+1 states up to this L


def alignment(rng, labels, T, blank=0):
    """A uniformly random valid CTC alignment of ``labels`` over ``T`` frames: blank gaps >= 0 (at least one
    between two equal labels), label durations >= 1.  Returns int64 [T]."""
    labels = np.asarray(labels, dtype=np.int64)
    L = len(labels)
    need = L + ctc_ref.count_repeats(labels)
    if need > T:
        raise ValueError("no alignment of %d labels (+%d repeats) in %d frames" % (L, need - L, T))
    extra = T - need
    # stars and bars: the extra frames over 2L+1 slots (L+1 blank gaps, L label durations), every composition
    # equally likely -- and compositions are in one-to-one correspondence with alignments
    n_slots = 2 * L + 1
    bars = np.sort(rng.choice(extra + n_slots - 1, size=n_slots - 1, replace=False))
    parts = np.diff(np.concatenate([[-1], bars, [extra + n_slots - 1]])) - 1
    seq = []
    for i in range(L):
        forced = 1 if i > 0 and labels[i] == labels[i - 1] else 0
        seq += [blank] * (parts[2 * i] + forced) + [int(labels[i])] * (1 + parts[2 * i + 1])
    seq += [blank] * parts[2 * L]
    return np.array(seq, dtype=np.int64)


def peaked_case(rng, T, labels, V, margin, noise, err_rate, err_run, blank=0):
    """Logits ``acts[T, V] = noise * N(0,1) + margin * onehot(target_t)`` (float32) and ``target[T]``.

    ``target`` is a random alignment of ``labels``, corrupted by recognition errors: every frame starts a run of
    ``err_run`` wrong frames with probability ``err_rate / err_run`` (about ``err_rate`` of the frames end up
    wrong); a run emits one random non-blank symbol that differs from the aligned symbol of each of its frames."""
    target = alignment(rng, labels, T, blank)
    aligned = target.copy()
    non_blank = np.array([k for k in range(V) if k != blank])
    starts = np.nonzero(rng.rand(T) < err_rate / err_run)[0] if err_rate > 0 else []
    for t0 in starts:
        span = slice(t0, min(T, t0 + err_run))
        while True:
            sym = int(rng.choice(non_blank))
            if not np.any(aligned[span] == sym):
                break
        target[span] = sym
    acts = noise * rng.randn(T, V)
    acts[np.arange(T), target] += margin
    return acts.astype(np.float32), target


def predicted_range_bits(acts_b, labels_b, blank=0, logit_scale=1.0):
    """log2 of the largest quantity the fast lattice's range check bounds, for one utterance (fp64).

    For every phase-2 frame t and lane (LANE_STATES consecutive lattice states):
      max_{s in lane} fresh_t(s) * max_{s in lane} stored_t(s) / P.
    The forward sweep owns the frames t >= T - floor(T/2) in phase 2 (lattice_fast.cuh, side_plan: it covers
    T - floor(T/2) frames in phase 1), its lanes are s // 8, fresh = alpha_t (emission included) and stored =
    beta_t / y_t (the backward side's pre-emission record).  The backward sweep runs on the reversed label
    sequence: its phase-2 frames are t < T - floor(T/2), its lanes (S-1-s) // 8, fresh = beta_t and stored =
    alpha_t / y_t.  The record a lane reads holds the states of its own group (the writer stores in the reader's
    group order), so both maxima run over the same states.

    Valid for one lattice window (L <= WINDOW_MAX_L): with several windows the halo lanes are not checked.
    The kernel evaluates the bound on exponent fields of fp32 values (within 3 bits of this), and only at
    frames where its dexp could matter; neither changes which side of a 24-bit margin a case is on.
    Returns -inf when the utterance is infeasible or empty."""
    acts_b = np.asarray(acts_b, dtype=np.float32)
    labels_b = np.asarray(labels_b, dtype=np.int64)
    T = acts_b.shape[0]
    if T == 0 or len(labels_b) + ctc_ref.count_repeats(labels_b) > T:
        return -np.inf
    z = (acts_b * np.float32(logit_scale)).astype(np.float64)       # the kernel scales in fp32
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        lp = ctc_ref.log_softmax(z, axis=1)
        ext = ctc_ref.extended_labels(labels_b, blank)
        alpha, beta, em = ctc_ref._alpha_beta(lp, ext, blank)
        S = len(ext)
        ll = alpha[T - 1, S - 1] if S == 1 else np.logaddexp(alpha[T - 1, S - 1], alpha[T - 1, S - 2])
        if not np.isfinite(ll):
            return -np.inf
        split = T - T // 2
        s = np.arange(S)
        out = -np.inf
        for lanes, fresh, stored, frames in ((s // LANE_STATES, alpha, beta - em, slice(split, T)),
                                             ((S - 1 - s) // LANE_STATES, beta, alpha - em, slice(0, split))):
            for g in np.unique(lanes):
                sel = lanes == g
                q = fresh[frames][:, sel].max(axis=1) + stored[frames][:, sel].max(axis=1) - ll
                q = q[np.isfinite(q)]
                if q.size:
                    out = max(out, float(q.max()))
    return out / np.log(2.0)


def range_class(bits):
    """'must-redo', 'must-stay-fast' or 'grey' (parity only) for a predicted range in bits."""
    if bits >= MUST_REDO_BITS:
        return "must-redo"
    if bits <= MUST_STAY_FAST_BITS:
        return "must-stay-fast"
    return "grey"


def min_log_prob(acts_b, logit_scale=1.0):
    """Smallest natural-log softmax probability of the rows (fp64): K1 flags a row when it is below -69."""
    z = (np.asarray(acts_b, dtype=np.float32) * np.float32(logit_scale)).astype(np.float64)
    return float(ctc_ref.log_softmax(z, axis=1).min()) if z.size else np.inf
