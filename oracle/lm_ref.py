"""CPU oracle of the n-gram language model fused into the prefix beam search (TEST INFRASTRUCTURE ONLY).

A dict-based ARPA reader and ``log_prob`` written directly from the definition (include/b200ctc.h,
b200ctc_beam_search_lm), independent of the library's loader (csrc/ngram_lm.cu):

    h = the last min(N-1, len) words of <s> followed by the prefix's words
    log10P(c | h) = p(h c)                                   if "h c" is an n-gram
                  = bo(h) + log10P(c | h minus its first word)   otherwise;   bo(h) = 0 when h is not an n-gram
    lnP(c | h) = log10P(c | h) * LN10

Numbers are read with python's float() (correctly rounded, as the library's strtod).  A decoder id maps to its
symbol when that is a unigram, else to <unk>.  Also: seeded writers of history-closed ARPA files for the tests.
"""

import math

import numpy as np

LN10 = 2.302585092994045684017991454684364208   # the double nearest ln 10, the literal of csrc/ngram_lm.cuh
EOS = None                                       # log_prob(history, EOS): ln P(</s> | history)


class ArpaLM(object):
    def __init__(self, path, symbols, blank=0):
        self.ngrams = {}            # tuple of words -> (log10 p, log10 bo)
        self.order = 0
        section = 0
        with open(path, encoding="utf-8") as f:
            for raw in f:
                line = raw.strip()
                if not line:
                    continue
                if line.startswith("\\"):
                    section = int(line[1:line.index("-")]) if line.endswith("-grams:") else 0
                    continue
                if section == 0:
                    continue
                tok = line.split()
                words = tuple(tok[1:section + 1])
                bo = float(tok[section + 1]) if len(tok) == section + 2 else 0.0
                self.ngrams[words] = (float(tok[0]), bo)
                self.order = max(self.order, section)
        self.words = {}
        for c, s in enumerate(symbols):
            if c != blank:
                self.words[c] = s if (s,) in self.ngrams else "<unk>"

    def log10_prob(self, h, w):
        h = tuple(h)
        if h + (w,) in self.ngrams:
            return self.ngrams[h + (w,)][0]
        bo = self.ngrams[h][1] if h in self.ngrams else 0.0
        return bo + self.log10_prob(h[1:], w)

    def log_prob(self, history, c):
        """ln P(c | history): history a sequence of decoder ids, c a decoder id or EOS."""
        words = ["<s>"] + [self.words[x] for x in history]
        n = min(self.order - 1, len(words))
        h = words[len(words) - n:] if n > 0 else []
        return self.log10_prob(h, "</s>" if c is EOS else self.words[c]) * LN10

    def score(self, seq, alpha, beta):
        """S(seq) = sum over its tokens of (alpha * lnP + beta), in order, each operation rounded."""
        S = 0.0
        for i in range(len(seq)):
            S = S + (alpha * self.log_prob(seq[:i], seq[i]) + beta)
        return S


def _write(path, grams, order):
    with open(path, "w", encoding="utf-8") as f:
        f.write("\\data\\\n")
        for k in range(1, order + 1):
            f.write("ngram %d=%d\n" % (k, len(grams[k])))
        for k in range(1, order + 1):
            f.write("\n\\%d-grams:\n" % k)
            for g, (p, bo) in grams[k]:
                f.write("%s\t%s" % (p, " ".join(g)) + ("\t%s" % bo if bo is not None else "") + "\n")
        f.write("\n\\end\\\n")


def random_arpa(path, words, order, seed, per_order=200, extra_words=("zz_unmapped",)):
    """A history-closed ARPA file of the given order over ``words`` + <s>, </s>, <unk> + ``extra_words``, with random
    probabilities and back-off weights (some histories without one)."""
    rng = np.random.RandomState(seed)
    vocab = list(words) + ["</s>", "<unk>"] + list(extra_words)
    levels = {1: [(w,) for w in vocab] + [("<s>",)]}
    for k in range(2, order + 1):
        hist = [g for g in levels[k - 1] if g[-1] != "</s>"]
        want = min(per_order, len(hist) * len(vocab) // 2)
        seen = set()
        while len(seen) < want:
            seen.add(hist[rng.randint(len(hist))] + (vocab[rng.randint(len(vocab))],))
        levels[k] = sorted(seen)
    grams = {}
    for k in range(1, order + 1):
        rows = []
        for g in levels[k]:
            p = "-99" if g == ("<s>",) else "%.6f" % rng.uniform(-3.0, -0.05)
            bo = "%.6f" % rng.uniform(-1.0, 0.3) if k < order and rng.uniform() < 0.8 else None
            rows.append((g, (p, bo)))
        grams[k] = rows
    _write(path, grams, order)
    return path


def counted_arpa(path, corpus, order, discount=0.5):
    """An absolute-discounting back-off model counted from ``corpus`` (a list of token-string sentences)."""
    counts = [dict() for _ in range(order + 1)]
    for sent in corpus:
        s = ["<s>"] + list(sent) + ["</s>"]
        for k in range(1, order + 1):
            for i in range(len(s) - k + 1):
                g = tuple(s[i:i + k])
                if g == ("<s>",):
                    continue
                counts[k][g] = counts[k].get(g, 0) + 1
    vocab = sorted(set(w for (w,) in counts[1]) | {"<s>"})
    total = sum(counts[1].values())
    prob = {}                                     # tuple -> linear probability (for the back-off weights)
    for (w,), n in counts[1].items():
        prob[(w,)] = n / total
    grams = {1: [(("<s>",), ("-99", None))]}
    grams[1] += [((w,), ("%.7f" % math.log10(prob[(w,)]), None)) for w in vocab if w != "<s>"]

    def lower(g):                                 # back-off probability of g's last word given g's history
        for j in range(1, len(g)):
            if g[j:] in prob:
                return prob[g[j:]]
        return prob.get(g[-1:], 1e-7)

    for k in range(2, order + 1):
        hist_tot = {}
        for g, n in counts[k].items():
            hist_tot[g[:-1]] = hist_tot.get(g[:-1], 0) + n
        rows = []
        for g, n in sorted(counts[k].items()):
            prob[g] = (n - discount) / hist_tot[g[:-1]]
            rows.append((g, ["%.7f" % math.log10(prob[g]), None]))
        grams[k] = rows
    bo = {}
    for k in range(2, order + 1):
        left, low = {}, {}
        for g, _ in grams[k]:
            h = g[:-1]
            left[h] = left.get(h, 1.0) - prob[g]
            low[h] = low.get(h, 1.0) - lower(g)
        for h in left:
            bo[h] = "%.7f" % math.log10(max(left[h], 1e-9) / max(low[h], 1e-9))
    for k in range(1, order):
        grams[k] = [(g, (p, bo.get(g))) for g, (p, _) in grams[k]]
    grams[order] = [(g, (p, None)) for g, (p, _) in grams[order]]
    _write(path, grams, order)
    return path
