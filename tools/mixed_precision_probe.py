"""Step time of the device-resident loss on bfloat16 logits, against the fp32 engine on fp32 logits and against the
composition it replaces (``acts.float()``, the fp32 engine, ``grads.to(bfloat16)``): the forward call
``ctc_loss_and_grad``, and forward + backward of ``ctc_loss_from_padded`` (the training step's loss) into
batch-major logits.  Also the time and achieved bandwidth of the kernel that rounds the staged fp32 gradient into
the bfloat16 buffer and of the backward kernel that multiplies it by grad_output.

    python tools/mixed_precision_probe.py [C3 C4 ...] [--steps N]

Each variant cycles through enough copies of the logits to keep more than 300 MB in flight, so no step reads its
inputs from the 126 MB L2.  The card's name and power limit are printed with the numbers."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytorch_end2end_speech_recognition_b200 as b200  # noqa: E402
from pytorch_end2end_speech_recognition_b200 import workloads  # noqa: E402

ROTATE_BYTES = 300e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def device_labels(wl):
    Lmax = int(wl.label_lens.max())
    ys = torch.zeros(wl.B, Lmax, dtype=torch.int32)
    off = 0
    for b, L in enumerate(wl.label_lens):
        ys[b, :L] = torch.from_numpy(wl.labels[off:off + L])
        off += L
    return ys.cuda(), torch.from_numpy(wl.act_lens).cuda(), torch.from_numpy(wl.label_lens).cuda()


def time_steps(step, n_sets, steps, reps=5):
    for i in range(max(3, n_sets)):
        step(i)
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(steps):
            step(i)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / steps)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=["C3", "C4"])
    ap.add_argument("--steps", type=int, default=40)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    print("card: %s" % card())
    for key in args.configs:
        wl = workloads.make_lengths_and_labels(key)
        dev = device_labels(wl)
        n = wl.T * wl.B * wl.V
        n_sets = max(2, int(-(-ROTATE_BYTES // (2 * n))))
        a32 = [workloads.make_acts(wl, copy_index=i).cuda() for i in range(n_sets)]
        a16 = [a.to(torch.bfloat16) for a in a32]

        def fp32(i):
            return b200.ctc_loss_and_grad(a32[i % n_sets], *dev)

        def bf16(i):
            return b200.ctc_loss_and_grad(a16[i % n_sets], *dev)

        def composition(i):
            c, l, g = b200.ctc_loss_and_grad(a16[i % n_sets].float(), *dev)
            return c, l, g.to(torch.bfloat16)

        ys, x_lens, y_lens = dev[0] - 1, dev[1], dev[2]             # from_padded adds the blank offset back

        def train(sets, widen):
            def step(i):
                lg = sets[i % n_sets].transpose(0, 1).detach().requires_grad_(True)    # [B, T, V] leaf
                loss = b200.ctc_loss_from_padded(lg.float() if widen else lg, ys, x_lens, y_lens)
                loss.backward()
                return lg.grad
            return step

        t = {name: time_steps(f, n_sets, args.steps) for name, f in
             (("fp32", fp32), ("bf16", bf16), ("composition", composition))}
        print("%s (%s), %d logit sets: fp32 engine %.4f ms/step, bf16 %.4f ms/step, composition %.4f ms/step"
              % (key, wl.name, n_sets, t["fp32"], t["bf16"], t["composition"]))
        t = {name: time_steps(f, n_sets, args.steps) for name, f in
             (("fp32", train(a32, False)), ("bf16", train(a16, False)), ("composition", train(a16, True)))}
        print("%s forward + backward of ctc_loss_from_padded: fp32 logits %.4f ms/step, bf16 logits %.4f ms/step, "
              "bf16 logits through .float() %.4f ms/step" % (key, t["fp32"], t["bf16"], t["composition"]))
        # the narrowing and scaling kernels alone, from a profiler run of its own
        step = train(a16, False)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for i in range(10):
                step(i)
            torch.cuda.synchronize()
        for kernel, nbytes in (("narrow_grads_kernel", 6), ("scale_grads_kernel", 4)):
            times = [e.device_time for e in prof.events() if kernel in e.name]
            if times:
                us = sorted(times)[len(times) // 2]
                print("%s %s: %.1f us median of %d, %.0f GB/s (%d elements, %d bytes each)"
                      % (key, kernel, us, len(times), nbytes * n / (us * 1e-6) / 1e9, n, nbytes))
            else:
                print("%s %s: not found in the profile" % (key, kernel))
        del a32, a16
        b200.ctc.release_workspaces()
        torch.cuda.empty_cache()
    print("card: %s" % card())


if __name__ == "__main__":
    main()
