"""Time of the greedy decoder, the posterior softmax and ``evaluate_batch`` on fp32, bfloat16 and float16 logits, and
of the composition a 16-bit call replaces (``greedy_decode(logits.float())``, the cast inside the timed region).
Also the arg-max kernel's own time, from a profiler run of its own, and its achieved bandwidth on algorithmic bytes:
``elem_size * V`` read per valid frame plus 4 bytes written per frame.

    python tools/decode_precision_probe.py [C3 C4 ...] [--steps N]

Inputs are the configs' batch-major [B, T, V] logits.  Each variant cycles through enough copies to keep more than
300 MB in flight, so no call reads its input from the 126 MB L2.  The card's name and power limit are printed with
the numbers."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytorch_end2end_speech_recognition_b200 as b200  # noqa: E402
from pytorch_end2end_speech_recognition_b200 import workloads  # noqa: E402

ROTATE_BYTES = 300e6
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def time_calls(call, n_sets, steps, reps=5):
    for i in range(max(3, n_sets)):
        call(i)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(steps):
            call(i)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps)
    return best


def argmax_kernel_us(call, n_sets):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for i in range(4 * n_sets + 8):
            call(i)
        torch.cuda.synchronize()
    times = [e.device_time for e in prof.events() if "frame_argmax" in e.name]
    return (sorted(times)[len(times) // 2], len(times)) if times else (float("nan"), 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=["C3", "C4"])
    ap.add_argument("--steps", type=int, default=40)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    print("card: %s" % card())
    for key in args.configs:
        wl = workloads.make_lengths_and_labels(key)
        n = wl.T * wl.B * wl.V
        n_sets = max(2, int(-(-ROTATE_BYTES // (2 * n))))
        base = [workloads.make_acts(wl, copy_index=i).transpose(0, 1).contiguous() for i in range(n_sets)]   # [B, T, V]
        sets = {name: [a.to(dt).cuda() for a in base] for name, dt in DTYPES.items()}
        del base
        lens = torch.from_numpy(wl.act_lens.astype(np.int32)).cuda()
        frames = int(np.minimum(wl.act_lens, wl.T).sum())
        ys = torch.randint(0, wl.V - 1, (wl.B, int(wl.label_lens.max())), device="cuda")
        y_lens = torch.from_numpy(wl.label_lens.astype(np.int32)).cuda()
        print("%s (%s), %d logit sets per type" % (key, wl.name, n_sets))
        for name, xs in sets.items():
            elem = xs[0].element_size()

            def greedy(i, xs=xs):
                return b200.greedy_decode(xs[i % n_sets], lens)

            def posteriors(i, xs=xs):
                return b200.posteriors(xs[i % n_sets])

            def evaluate(i, xs=xs):
                return b200.evaluate_batch(xs[i % n_sets], lens, ys, y_lens, beam_width=1)

            t_greedy = time_calls(greedy, n_sets, args.steps)
            t_post = time_calls(posteriors, n_sets, args.steps)
            t_eval = time_calls(evaluate, n_sets, args.steps)
            us, cnt = argmax_kernel_us(greedy, n_sets)
            nbytes = elem * wl.V * frames + 4 * frames
            line = ("%s %s: greedy_decode %.4f ms/call, posteriors %.4f ms/call, evaluate_batch(beam_width=1) %.4f "
                    "ms/call; arg-max kernel %.1f us (median of %d) = %.0f GB/s on %d algorithmic bytes"
                    % (key, name, t_greedy, t_post, t_eval, us, cnt, nbytes / (us * 1e-6) / 1e9, nbytes))
            if name != "fp32":
                t_comp = time_calls(lambda i, xs=xs: b200.greedy_decode(xs[i % n_sets].float(), lens), n_sets, args.steps)
                line += "; greedy_decode(logits.float()) %.4f ms/call" % t_comp
            print(line)
        del sets
        torch.cuda.empty_cache()
    print("card: %s" % card())


if __name__ == "__main__":
    main()
