"""Developer aid (GPU box): where does a step's time go?  Per-step device time of the host-label call (with the
same labels every step, and with two label sets in turn, as in training, where every mini-batch brings new
transcripts), the device-resident call issued eagerly, and the device-resident call replayed from a CUDA graph,
next to the kernel times the library measures with its own events.   python tools/step_probe.py C1 C3"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pytorch_end2end_speech_recognition_b200 import ctc as ctc_mod, workloads  # noqa: E402
import pytorch_end2end_speech_recognition_b200 as b200  # noqa: E402


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    fn(n)
    e1.record()
    host = (time.perf_counter() - t0) * 1e3 / n
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, host


for key in (sys.argv[1:] or ["C1", "C3"]):
    wl = workloads.make_lengths_and_labels(key)
    dev = torch.device("cuda", 0)
    r = bench.Runner(wl, dev, 1, 0)
    slot = r.loss_groups[0][0:1]

    # every symbol moved to the next one: other labels with the same lengths and repeats
    label_sets = (wl.labels, (wl.labels % (wl.V - 1) + 1).astype(np.int32))

    def host_path(n, n_sets=1):
        for i in range(n):
            b200.ctc_loss_and_grad(r.acts_dev[i % r.n_rot], label_sets[i % n_sets], wl.act_lens, wl.label_lens,
                                   grads=r.grads_dev[i % r.n_rot], costs=r.costs, loss_sum=slot)

    def host_path_alternating(n):
        host_path(n, 2)

    def dev_eager(n):
        for i in range(n):
            r.one(i % r.n_rot, slot)

    for fn in (host_path, host_path_alternating, dev_eager):
        fn(8)
    res = {"host-label call, eager": timed(host_path, 48),
           "host-label call, two label sets": timed(host_path_alternating, 48),
           "device-resident call, eager": timed(dev_eager, 48),
           "device-resident call, graph of %d" % r.group: timed(lambda n: r.run(n), 48)}
    for grp in (8, 16):
        bench.GROUP = grp
        r2 = bench.Runner(wl, dev, 1, 0, acts_dev=r.acts_dev)
        r2.run(2 * grp)
        res["device-resident call, graph of %d" % r2.group] = timed(lambda n: r2.run(n), 48)
        del r2
    bench.GROUP = 8
    k = bench.kernel_times(r, ctc_mod, 8)
    print(key, "kernels (library events, eager): softmax %.4f lattice %.4f third %.4f ms" % tuple(k))
    for name, (d, h) in res.items():
        print("   %-34s device %.4f ms/step   host %.4f ms/step" % (name, d, h))
    del r
    ctc_mod.release_workspaces()
