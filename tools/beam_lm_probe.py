"""Time of the prefix beam search with and without an n-gram LM fused in, at beam 10, on the C1 (V = 62), C3 (V = 30)
and C4 (V = 3386) shapes, the LM-fused kernel's own time from a profiler run of its own, and the host load time of
the LM.

    python tools/beam_lm_probe.py [C1 C3 C4 ...] [--beam 10] [--steps N]

Log-probabilities are ``log_softmax`` of the configs' seeded logits, batch-major [B, T, V].  The LMs are seeded,
history-closed random trigram models (oracle/lm_ref.random_arpa) written to a temporary directory: C1 / C3 with up
to 20 000 n-grams per order, C4 with about 400 000 bigrams and 400 000 trigrams.  The card's name and power limit are
printed with the numbers."""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytorch_end2end_speech_recognition_b200 as b200  # noqa: E402
from pytorch_end2end_speech_recognition_b200 import workloads  # noqa: E402
from oracle import lm_ref  # noqa: E402

PER_ORDER = {"C4": 400000}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def time_calls(call, steps, reps=3):
    call()
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            call()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps)
    return best


def kernel_ms(call, tag, n=3):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            call()
        torch.cuda.synchronize()
    times = [e.device_time / 1e3 for e in prof.events() if "beam_search_kernel" in e.name and tag in e.name]
    return (sorted(times)[len(times) // 2], len(times)) if times else (float("nan"), 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=["C1", "C3", "C4"])
    ap.add_argument("--beam", type=int, default=10)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    print("card: %s" % card())
    tmp = tempfile.mkdtemp(prefix="beam_lm_probe_")
    for key in args.configs:
        wl = workloads.make_lengths_and_labels(key)
        lp = torch.log_softmax(workloads.make_acts(wl).transpose(0, 1).contiguous(), dim=-1).cuda()
        lens = torch.from_numpy(wl.act_lens.astype(np.int32)).cuda()
        symbols = ["_"] + ["s%d" % c for c in range(1, wl.V)]
        path = lm_ref.random_arpa(os.path.join(tmp, key + ".arpa"), symbols[1:], 3, 1623,
                                  per_order=PER_ORDER.get(key, 20000))
        t0 = time.perf_counter()
        lm = b200.NGramLM(path, symbols)
        load_s = time.perf_counter() - t0
        os.remove(path)

        def plain():
            return b200.beam_search_decode(lp, lens, args.beam)

        def fused():
            return b200.beam_search_decode(lp, lens, args.beam, lm=lm, alpha=0.8, beta=1.0)

        t_plain = time_calls(plain, args.steps)
        t_fused = time_calls(fused, args.steps)
        k_plain, _ = kernel_ms(plain, ", false>")
        k_fused, cnt = kernel_ms(fused, ", true>")
        print("%s (%s), beam %d, LM order %d with %s n-grams (loaded in %.3f s on the host, incl. the copy to the GPU): "
              "beam_search_decode %.3f ms/call without the LM, %.3f ms/call with it (x%.2f); kernels %.3f / %.3f ms "
              "(median of %d)" % (key, wl.name, args.beam, lm.order, "+".join(str(c) for c in lm.counts), load_s,
                                  t_plain, t_fused, t_fused / t_plain, k_plain, k_fused, cnt))
        lm.close()
        del lp
        torch.cuda.empty_cache()
    os.rmdir(tmp)
    print("card: %s" % card())


if __name__ == "__main__":
    main()
