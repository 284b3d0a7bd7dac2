"""ctypes binding of the C-ABI library (include/b200ctc.h) for the decoders, evaluation and diagnostics; the
loss goes through the PyTorch extension (csrc/torch_binding.cpp).

The shared library is built in-tree by ``build.py`` (``lib/libb200ctc.so``).  There is no
fallback implementation: if the library cannot be loaded every product entry point raises.
"""

import ctypes
import os
import threading

from . import build as _build

_LOCK = threading.Lock()
_LIB = None

STATUS_SUCCESS = 0
FLOAT32, BFLOAT16, FLOAT16 = 0, 1, 2     # b200ctc_dtype_t

# every symbol include/b200ctc.h declares (tests check that the library exports all of them)
EXPORTED_SYMBOLS = (
    "b200ctc_version",
    "b200ctc_status_string",
    "b200ctc_create",
    "b200ctc_destroy",
    "b200ctc_get_workspace_size",
    "b200ctc_get_workspace_bound",
    "b200ctc_loss_and_grad",
    "b200ctc_loss_and_grad_dev",
    "b200ctc_loss_and_grad_dev_typed",
    "b200ctc_get_workspace_bound_typed",
    "b200ctc_scale_grads",
    "b200ctc_greedy_decode",
    "b200ctc_greedy_decode_typed",
    "b200ctc_beam_search_workspace",
    "b200ctc_beam_search",
    "b200ctc_beam_search_typed",
    "b200ctc_edit_distance_workspace",
    "b200ctc_edit_distance",
    "b200ctc_softmax_temperature",
    "b200ctc_softmax_temperature_typed",
    "b200ctc_set_profiling",
    "b200ctc_get_last_kernel_ms",
    "b200ctc_get_last_fallbacks",
    "b200ctc_get_plan_cache_stats",
)


class B200CTCError(RuntimeError):
    """Raised for every non-zero status of the C ABI (a RuntimeError, so the reference's
    skip-mini-batch guard, utils/training/training_loop.py:69-76, keeps working)."""


def declare(lib):
    """Set the ctypes signatures of ``lib``'s entry points (any build of the library, variants included) and
    return it.  b200ctc_loss_and_grad_dev is left undeclared: only the PyTorch extension calls it."""
    c_int_p = ctypes.POINTER(ctypes.c_int)
    lib.b200ctc_version.restype = ctypes.c_int
    lib.b200ctc_version.argtypes = []
    lib.b200ctc_status_string.restype = ctypes.c_char_p
    lib.b200ctc_status_string.argtypes = [ctypes.c_int]
    lib.b200ctc_create.restype = ctypes.c_int
    lib.b200ctc_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int]
    lib.b200ctc_destroy.restype = ctypes.c_int
    lib.b200ctc_destroy.argtypes = [ctypes.c_void_p]
    lib.b200ctc_get_workspace_size.restype = ctypes.c_int
    lib.b200ctc_get_workspace_size.argtypes = [c_int_p, c_int_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.POINTER(ctypes.c_size_t)]
    lib.b200ctc_loss_and_grad.restype = ctypes.c_int
    lib.b200ctc_loss_and_grad.argtypes = [
        ctypes.c_void_p,                                   # handle
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64,   # acts, stride_t, stride_b
        ctypes.c_void_p,                                   # grads
        c_int_p, c_int_p, c_int_p,                         # flat_labels, label_lens, act_lens (host)
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,  # T, V, B, blank
        ctypes.c_void_p, ctypes.c_void_p,                  # costs, loss_sum (device)
        ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p  # workspace, bytes, stream
    ]
    lib.b200ctc_get_workspace_bound.restype = ctypes.c_int
    lib.b200ctc_get_workspace_bound.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.POINTER(ctypes.c_size_t)]
    lib.b200ctc_get_workspace_bound_typed.restype = ctypes.c_int
    lib.b200ctc_get_workspace_bound_typed.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                      ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_size_t)]
    lib.b200ctc_loss_and_grad_dev_typed.restype = ctypes.c_int
    lib.b200ctc_loss_and_grad_dev_typed.argtypes = [
        ctypes.c_void_p,                                                 # handle
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int,   # acts, stride_t, stride_b, acts_dtype
        ctypes.c_void_p,                                                 # grads (acts_dtype)
        ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,   # labels, label_stride, label_lens, act_lens
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,  # T, V, B, max_label_len, blank
        ctypes.c_void_p,                                                 # options or NULL
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,               # costs, loss_sum, ls_costs (device fp32)
        ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p                # workspace, bytes, stream
    ]
    lib.b200ctc_scale_grads.restype = ctypes.c_int
    lib.b200ctc_scale_grads.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    lib.b200ctc_get_plan_cache_stats.restype = ctypes.c_int
    lib.b200ctc_get_plan_cache_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_longlong),
                                                 ctypes.POINTER(ctypes.c_longlong)]
    lib.b200ctc_greedy_decode.restype = ctypes.c_int
    lib.b200ctc_greedy_decode.argtypes = [
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.b200ctc_greedy_decode_typed.restype = ctypes.c_int
    lib.b200ctc_greedy_decode_typed.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.b200ctc_beam_search_workspace.restype = ctypes.c_int
    lib.b200ctc_beam_search_workspace.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                  ctypes.POINTER(ctypes.c_size_t)]
    lib.b200ctc_beam_search.restype = ctypes.c_int
    lib.b200ctc_beam_search.argtypes = [
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
        ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_size_t, ctypes.c_void_p]
    lib.b200ctc_beam_search_typed.restype = ctypes.c_int
    lib.b200ctc_beam_search_typed.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
        ctypes.c_size_t, ctypes.c_void_p]
    lib.b200ctc_edit_distance_workspace.restype = ctypes.c_int
    lib.b200ctc_edit_distance_workspace.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_size_t)]
    lib.b200ctc_edit_distance.restype = ctypes.c_int
    lib.b200ctc_edit_distance.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
        ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    lib.b200ctc_softmax_temperature.restype = ctypes.c_int
    lib.b200ctc_softmax_temperature.argtypes = [
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
        ctypes.c_void_p, ctypes.c_void_p]
    lib.b200ctc_softmax_temperature_typed.restype = ctypes.c_int
    lib.b200ctc_softmax_temperature_typed.argtypes = [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
        ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]
    lib.b200ctc_set_profiling.restype = ctypes.c_int
    lib.b200ctc_set_profiling.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.b200ctc_get_last_kernel_ms.restype = ctypes.c_int
    lib.b200ctc_get_last_kernel_ms.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]
    lib.b200ctc_get_last_fallbacks.restype = ctypes.c_int
    lib.b200ctc_get_last_fallbacks.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_void_p]
    return lib


def library_path():
    return _build.LIB_PATH


def load(build_if_missing=True):
    """Load (and if necessary build) libb200ctc.so.  Raises B200CTCError when impossible."""
    global _LIB
    with _LOCK:
        if _LIB is not None:
            return _LIB
        path = _build.LIB_PATH
        if not os.path.exists(path) and not build_if_missing:
            raise B200CTCError("libb200ctc.so is not built (%s); run __graft_entry__.build()" % path)
        if build_if_missing and not os.environ.get("B200CTC_LIB"):
            # a no-op when the library is newer than every source; rebuilds a stale library after csrc edits
            # (lib/ is git-ignored but travels with the repo snapshot).  Without nvcc a library that exists is used.
            try:
                _build.build_library()
            except Exception as exc:  # nvcc missing or compile error
                if not os.path.exists(path):
                    raise B200CTCError("cannot build libb200ctc.so: %s" % exc)
        try:
            _LIB = declare(ctypes.CDLL(path))
        except OSError as exc:
            raise B200CTCError("cannot load %s: %s" % (path, exc))
        return _LIB


def check(status, what):
    if status != STATUS_SUCCESS:
        msg = load().b200ctc_status_string(status).decode()
        raise B200CTCError("%s failed: %s (status %d)" % (what, msg, status))
