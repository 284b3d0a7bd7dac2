"""ctypes wrapper + build recipe for the C++/OpenMP CPU restatement (oracle/ctc_cpu.cpp).

TEST / BASELINE INFRASTRUCTURE ONLY (see the header of ctc_cpu.cpp).  The shared object is
compiled with the host compiler: ``g++ -O3 -march=native -fopenmp -shared -fPIC``.
"""

import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_DIR = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_DIR, "ctc_cpu.cpp")
LIB = os.path.join(_DIR, "liboracle_ctc.so")
_lib = None


def _stale(path):
    return not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(SRC)


def build(force=False, out=LIB):
    if force or _stale(out):
        subprocess.run(["g++", "-O3", "-march=native", "-std=c++17", "-fopenmp", "-shared", "-fPIC",
                        SRC, "-o", out], check=True)
    return out


def load():
    global _lib
    if _lib is None:
        # -march=native code built elsewhere may not run here: rebuild when the host differs
        if _stale(LIB):
            # only build() writes into the source tree: a missing or stale library is compiled into a
            # temporary directory (the tree may be read-only), loaded, and the directory removed
            tmp = tempfile.mkdtemp(prefix="oracle_ctc_")
            try:
                lib = ctypes.CDLL(build(out=os.path.join(tmp, "liboracle_ctc.so")))
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
        else:
            lib = ctypes.CDLL(LIB)
        fp = ctypes.POINTER(ctypes.c_float)
        ip = ctypes.POINTER(ctypes.c_int)
        for name in ("oracle_ctc_cpu_f32", "oracle_ctc_cpu_f64"):
            fn = getattr(lib, name)
            fn.restype = ctypes.c_int
            fn.argtypes = [fp, fp, ip, ip, ip, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, fp,
                           ctypes.c_int]
        lib.oracle_ctc_max_threads.restype = ctypes.c_int
        _lib = lib
    return _lib


def max_threads():
    return load().oracle_ctc_max_threads()


def ctc_cpu(acts, labels, act_lens, label_lens, blank=0, precision="f32", num_threads=None, need_grad=True):
    """acts: float32 [T,B,V] numpy (contiguous).  Returns (costs[B] f32, grads[T,B,V] f32 or None)."""
    lib = load()
    acts = np.ascontiguousarray(acts, dtype=np.float32)
    T, B, V = acts.shape
    labels = np.ascontiguousarray(labels, dtype=np.int32)
    act_lens = np.ascontiguousarray(act_lens, dtype=np.int32)
    label_lens = np.ascontiguousarray(label_lens, dtype=np.int32)
    costs = np.empty(B, dtype=np.float32)
    grads = np.empty_like(acts) if need_grad else None
    fp = ctypes.POINTER(ctypes.c_float)
    ip = ctypes.POINTER(ctypes.c_int)
    fn = lib.oracle_ctc_cpu_f32 if precision == "f32" else lib.oracle_ctc_cpu_f64
    nt = int(num_threads) if num_threads else max_threads()
    fn(acts.ctypes.data_as(fp), grads.ctypes.data_as(fp) if need_grad else None,
       labels.ctypes.data_as(ip), label_lens.ctypes.data_as(ip), act_lens.ctypes.data_as(ip),
       T, B, V, int(blank), costs.ctypes.data_as(fp), nt)
    return costs, grads
