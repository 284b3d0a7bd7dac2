"""Developer aid (GPU box): race hunt.  Repeats the host-label call on fixed inputs and compares costs and
gradients bit for bit with the first result (the engine is bit-reproducible by design).
   python tools/stress_repro.py lib.so [more.so] KEY [KEY ...] [--n=40]"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pytorch_end2end_speech_recognition_b200 import _lib, workloads  # noqa: E402

libs = [a for a in sys.argv[1:] if a.endswith(".so")]
keys = [a for a in sys.argv[1:] if not a.endswith(".so") and not a.startswith("--")] or ["C5"]
n_rep = next((int(a[4:]) for a in sys.argv[1:] if a.startswith("--n=")), 40)
alt_key = next((a[6:] for a in sys.argv[1:] if a.startswith("--alt=")), None)   # a call of this workload (same handle, same workspace) before every repeat
poison = "--poison" in sys.argv                                                   # fill the workspace with NaN bit patterns before every repeat
ip = ctypes.POINTER(ctypes.c_int)
for key in keys:
    wl = workloads.make_lengths_and_labels(key)
    acts = workloads.make_acts(wl).cuda()
    for path in libs:
        lib = _lib.declare(ctypes.CDLL(path))
        h = ctypes.c_void_p()
        assert lib.b200ctc_create(ctypes.byref(h), 0) == 0
        n = ctypes.c_size_t()
        ll, al, lab = wl.label_lens.ctypes.data_as(ip), wl.act_lens.ctypes.data_as(ip), wl.labels.ctypes.data_as(ip)
        assert lib.b200ctc_get_workspace_size(ll, al, wl.T, wl.V, wl.B, ctypes.byref(n)) == 0
        size = n.value
        if alt_key:
            awl = workloads.make_lengths_and_labels(alt_key)
            aacts = workloads.make_acts(awl).cuda()
            agr = torch.empty_like(aacts)
            all_, aal, alab = awl.label_lens.ctypes.data_as(ip), awl.act_lens.ctypes.data_as(ip), awl.labels.ctypes.data_as(ip)
            n2 = ctypes.c_size_t()
            assert lib.b200ctc_get_workspace_size(all_, aal, awl.T, awl.V, awl.B, ctypes.byref(n2)) == 0
            size = max(size, n2.value)
            acost, aloss = torch.empty(awl.B, device="cuda"), torch.empty(1, device="cuda")
        ws = torch.empty(size, dtype=torch.uint8, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream
        ref_g = ref_c = None
        bad = 0
        worst = 0.0
        for it in range(n_rep):
            if poison:
                ws.fill_(0xff)
            if alt_key:
                st = lib.b200ctc_loss_and_grad(h, aacts.data_ptr(), aacts.stride(0), aacts.stride(1), agr.data_ptr(), alab, all_, aal,
                                               awl.T, awl.V, awl.B, 0, acost.data_ptr(), aloss.data_ptr(), ws.data_ptr(), size, stream)
                assert st == 0
            grads = torch.full_like(acts, float("nan"))
            costs, loss = torch.empty(wl.B, device="cuda"), torch.empty(1, device="cuda")
            st = lib.b200ctc_loss_and_grad(h, acts.data_ptr(), acts.stride(0), acts.stride(1), grads.data_ptr(), lab, ll, al,
                                           wl.T, wl.V, wl.B, 0, costs.data_ptr(), loss.data_ptr(), ws.data_ptr(), size, stream)
            assert st == 0
            torch.cuda.synchronize()
            if ref_g is None:
                ref_g, ref_c = grads.clone(), costs.clone()
                continue
            same = torch.equal(grads, ref_g) and torch.equal(costs, ref_c)
            if not same:
                bad += 1
                d = (grads - ref_g).abs()
                d[torch.isnan(d)] = 1e9
                worst = max(worst, float(d.max()))
                idx = torch.nonzero(d > 0)
                if bad <= 3:
                    print("   mismatch at iteration %d: %d entries differ, max |diff| %.3g, first (t,b,v) = %s, utterances %s" % (
                        it, idx.shape[0], float(d.max()), idx[0].tolist(), sorted(set(idx[:, 1].tolist()))[:8]))
        print("%s %-26s %d/%d repeats differ from the first result (max |diff| %.3g)" % (key, os.path.basename(path), bad, n_rep - 1, worst))
