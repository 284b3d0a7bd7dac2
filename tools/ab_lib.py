"""Developer aid (GPU box): A/B two builds of the library on the host-label call (whose C signature has not
changed since round 1), bypassing the Python package.   python tools/ab_lib.py libA.so libB.so C1 C3"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pytorch_end2end_speech_recognition_b200 import _lib, workloads  # noqa: E402

libs = [a for a in sys.argv[1:] if a.endswith(".so")]
keys = [a for a in sys.argv[1:] if not a.endswith(".so")] or ["C1", "C3"]
ip = ctypes.POINTER(ctypes.c_int)
for key in keys:
    wl = workloads.make_lengths_and_labels(key)
    n_rot = 8
    acts = [workloads.make_acts(wl, copy_index=i).cuda() for i in range(n_rot)]
    grads = [torch.empty_like(a) for a in acts]
    costs, loss = torch.empty(wl.B, device="cuda"), torch.empty(1, device="cuda")
    for path in libs:
        lib = _lib.declare(ctypes.CDLL(path))
        h = ctypes.c_void_p()
        assert lib.b200ctc_create(ctypes.byref(h), 0) == 0
        n = ctypes.c_size_t()
        ll, al, lab = wl.label_lens.ctypes.data_as(ip), wl.act_lens.ctypes.data_as(ip), wl.labels.ctypes.data_as(ip)
        assert lib.b200ctc_get_workspace_size(ll, al, wl.T, wl.V, wl.B, ctypes.byref(n)) == 0
        ws = torch.empty(n.value, dtype=torch.uint8, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream

        def step(i):
            a = acts[i % n_rot]
            st = lib.b200ctc_loss_and_grad(h, a.data_ptr(), a.stride(0), a.stride(1), grads[i % n_rot].data_ptr(), lab, ll, al,
                                           wl.T, wl.V, wl.B, 0, costs.data_ptr(), loss.data_ptr(), ws.data_ptr(), n.value, stream)
            assert st == 0
        for i in range(10):
            step(i)
        best = 1e9
        for rep in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(64):
                step(i)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / 64)
        print("%s %-28s %.4f ms/step   loss %.3f" % (key, os.path.basename(path), best, float(loss.cpu()[0])))
