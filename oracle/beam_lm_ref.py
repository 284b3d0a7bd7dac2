"""CPU oracle for the CTC prefix beam search with an n-gram language model fused in (TEST INFRASTRUCTURE ONLY; see
oracle/ctc_ref.py), the definition of include/b200ctc.h, b200ctc_beam_search_lm.

oracle/beam_ref.py's search (the reference's decoder restated, tuple-keyed insertion-ordered dict, stable sort) with
``lm`` (an oracle.lm_ref.ArpaLM): every prefix carries S(prefix + c) = S(prefix) + (alpha * lnP(c | prefix) + beta),
the stable sort is by logaddexp(p_blank, p_non_blank) + S, and the hypothesis is the entry of the last beam with the
largest (logaddexp(p_blank, p_non_blank) + S) + alpha * lnP(</s> | prefix), ties to the earlier entry.  Each python
float operation is rounded on its own, as the kernel's __dmul_rn / __dadd_rn.
"""

import numpy as np

from . import beam_ref

LOG_0 = beam_ref.LOG_0


def beam_search(log_probs, n_frames, beam_width, blank=0, lm=None, alpha=0.0, beta=0.0):
    """log_probs [T, V]; returns (hypothesis as a list of ints, its score).  lm: an oracle.lm_ref.ArpaLM; without one
    this is oracle.beam_ref.beam_search."""
    if lm is None:
        return beam_ref.beam_search(log_probs, n_frames, beam_width, blank)
    lp = np.asarray(log_probs, dtype=np.float64)
    V = lp.shape[1]
    S = {(): 0.0}                                 # S depends on the prefix alone

    def extend(prefix, c):
        new_prefix = prefix + (c,)
        if new_prefix not in S:
            S[new_prefix] = S[prefix] + (alpha * lm.log_prob(prefix, c) + beta)
        return new_prefix

    beam = [((), (0.0, LOG_0))]
    with np.errstate(all="ignore"):
        for t in range(int(n_frames)):
            nxt = {}
            for c in range(V):
                p_t = lp[t, c]
                for prefix, (p_b, p_nb) in beam:
                    if c == blank:
                        n_b, n_nb = nxt.get(prefix, (LOG_0, LOG_0))
                        nxt[prefix] = (np.logaddexp(n_b, np.logaddexp(p_b + p_t, p_nb + p_t)), n_nb)
                        continue
                    end = prefix[-1] if prefix else None
                    new_prefix = extend(prefix, c)
                    n_b, n_nb = nxt.get(new_prefix, (LOG_0, LOG_0))
                    if c != end:
                        n_nb = np.logaddexp(n_nb, np.logaddexp(p_b + p_t, p_nb + p_t))
                    else:
                        n_nb = np.logaddexp(n_nb, p_b + p_t)
                    nxt[new_prefix] = (n_b, n_nb)
                    if c == end:
                        n_b, n_nb = nxt.get(prefix, (LOG_0, LOG_0))
                        nxt[prefix] = (n_b, np.logaddexp(n_nb, p_nb + p_t))
            beam = sorted(nxt.items(), key=lambda x: np.logaddexp(*x[1]) + S[x[0]], reverse=True)[:beam_width]
        best, best_score = None, None
        for prefix, (p_b, p_nb) in beam:
            f = (np.logaddexp(p_b, p_nb) + S[prefix]) + alpha * lm.log_prob(prefix, None)
            if best is None or f > best_score:
                best, best_score = prefix, f
    return list(best), float(best_score)
