"""Time of the batched word-error call on a C3-shaped batch (B = 128 character references of up to 400 symbols,
V = 30) against the two ways of getting the same numbers per utterance: the ``b200.compute_wer`` loop over word
lists on the host, and the host oracle (oracle/word_ref.word_errors).

    python tools/word_errors_probe.py [--steps N] [--oracle-pairs N]

References are drawn from a seeded list of 500 words of 1 to 10 symbols over the V - 2 symbols that are neither the
blank nor the space; hypotheses are the references with seeded substitutions, insertions and deletions (5 % each,
spaces included).  Label space: symbols 0 .. 27, space 28, as ``evaluate_batch`` returns hypotheses.

``word_errors``: CUDA events around N calls (inputs and lengths already on the device), and the kernel's own time
from a profiler run of its own.  ``compute_wer`` loop: what a user runs today -- copy the hypotheses to the host,
split each pair at the space, one ``b200.compute_wer`` call per utterance; host clock, which ends synchronised
because every call copies its result back.  Oracle: host clock over the first ``--oracle-pairs`` pairs (all by
default).  Every result is checked against the oracle on those pairs and against the ``compute_wer`` loop on all of
them.  The card's name and power limit are printed with the numbers."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytorch_end2end_speech_recognition_b200 as b200  # noqa: E402
from oracle import word_ref  # noqa: E402

B, V, MAX_REF, SPACE = 128, 30, 400, 28


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def make_batch(seed=1623):
    rng = np.random.RandomState(seed)
    letters = np.arange(V - 2)
    words = [list(rng.choice(letters, size=rng.randint(1, 11))) for _ in range(500)]
    refs, hyps = [], []
    for _ in range(B):
        target, ref = rng.randint(MAX_REF // 2, MAX_REF + 1), []
        while True:
            w = words[rng.randint(len(words))]
            if len(ref) + len(w) + (1 if ref else 0) > target:
                break
            ref += ([SPACE] if ref else []) + w
        hyp = []
        for t in ref:
            u = rng.rand()
            if u < 0.05:
                continue                                                  # deletion
            hyp.append(int(rng.choice(letters)) if u < 0.10 else int(t))  # substitution
            if rng.rand() < 0.05:
                hyp.append(int(rng.randint(V - 1)))                       # insertion (the space included)
        refs.append([int(t) for t in ref])
        hyps.append(hyp)
    return refs, hyps


def padded(seqs):
    lens = np.array([len(s) for s in seqs], dtype=np.int32)
    out = np.zeros((len(seqs), int(lens.max())), dtype=np.int32)
    for b, s in enumerate(seqs):
        out[b, :len(s)] = s
    return torch.from_numpy(out).cuda(), torch.from_numpy(lens).cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--oracle-pairs", type=int, default=B)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    print("card: %s" % card())
    refs, hyps = make_batch()
    r, rl = padded(refs)
    h, hl = padded(hyps)
    print("batch: B = %d, reference symbols %d..%d (mean %.0f), %d reference words, hypotheses up to %d symbols" % (
        B, min(map(len, refs)), max(map(len, refs)), np.mean([len(x) for x in refs]),
        sum(len(word_ref.split_words(x, SPACE)) for x in refs), h.size(1)))

    def call():
        return b200.word_errors(r, rl, h, hl, SPACE)

    w, c, n = (x.cpu().numpy() for x in call())
    for _ in range(3):
        call()
    best = float("inf")
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            call()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / args.steps)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            call()
        torch.cuda.synchronize()
    ktimes = sorted(e.device_time / 1e3 for e in prof.events() if "word_errors_kernel" in e.name)
    kernel = ktimes[len(ktimes) // 2] if ktimes else float("nan")

    # the per-utterance loop of today: hypotheses to the host, split at the space, one compute_wer per utterance
    b200.compute_wer([(1,)], [(1,)])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    hyp_host, hyp_lens = h.cpu().numpy(), hl.cpu().numpy()
    loop = [b200.compute_wer(word_ref.split_words(refs[b], SPACE),
                             word_ref.split_words(hyp_host[b, :hyp_lens[b]], SPACE)) for b in range(B)]
    t_loop = (time.perf_counter() - t0) * 1e3
    for b in range(B):
        assert tuple(loop[b]) == tuple(int(x) for x in w[b]), b

    k = min(args.oracle_pairs, B)
    t0 = time.perf_counter()
    oracle = [word_ref.word_errors(refs[b], hyps[b], SPACE) for b in range(k)]
    t_oracle = (time.perf_counter() - t0) * 1e3
    for b in range(k):
        assert oracle[b] == (tuple(int(x) for x in w[b]), tuple(int(x) for x in c[b]), tuple(int(x) for x in n[b])), b

    wer = w[:, 0].sum() / n[:, 0].sum()
    cer = c[:, 0].sum() / n[:, 1].sum()
    print("WER %.4f, CER %.4f (equal to the compute_wer loop on all %d pairs and to the oracle on %d)" % (wer, cer, B, k))
    print("word_errors: %.3f ms/call (events, best of 3 x %d calls), kernel %.3f ms (median of %d)" % (
        best, args.steps, kernel, len(ktimes)))
    print("compute_wer loop (words only): %.1f ms for %d utterances (host clock, incl. the hypothesis copy)" % (t_loop, B))
    print("host oracle (words + characters): %.1f ms for %d pairs, %.1f ms/pair" % (t_oracle, k, t_oracle / k))
    print("card: %s" % card())


if __name__ == "__main__":
    main()
