"""Host-side mirror of the ``warpctc_pytorch`` call surface used by the reference
(models/pytorch_v3/ctc/ctc.py:30-69, identical in models/pytorch/ctc/ctc.py), on top of the
C ABI in include/b200ctc.h.

Surface kept (same names, argument order and meaning):
  * ``gpu_ctc(acts, grads, labels, label_lens, act_lens, minibatch_size, costs[, blank])``
        fills ``grads`` (CUDA) and ``costs`` (CPU, per utterance) in place; note the order
        label_lens BEFORE act_lens (reference call, ctc.py:39-45).
  * ``cpu_ctc(...)``   raises: the product has no CPU path (the CPU restatement lives in oracle/).
  * ``_CTC``           autograd.Function; ``forward`` may be overridden by a subclass that only
        stashes ``ctx.grads`` (exactly what the reference does, ctc.py:30-52) while ``backward``
        is inherited from here.
  * ``CTCLoss(size_average=False, length_average=False, blank=0)``  nn.Module front end.
Native additions: ``ctc_loss_and_grad`` (device-resident results, no host sync) and
``ctc_loss`` (autograd, device scalar).  With device-resident labels these, and ``ctc_loss_from_padded``, also take
bfloat16 and float16 logits (``torch.autocast``): the gradient comes back in the logits' dtype, the costs in fp32.
"""

import ctypes
import importlib.util
import os

import numpy as np
import torch

from . import _lib
from . import build as _build
from ._lib import B200CTCError

_HANDLES = {}
_EXT = None          # the PyTorch C++ extension over the C ABI (csrc/torch_binding.cpp), once loaded


def _ext():
    """The thin PyTorch C++ extension (north_star: "a thin PyTorch C++/CUDA extension over a C-ABI"): the one
    binding of the loss.  Built in-tree by ``__graft_entry__.build()``, and here when it is missing or stale, as
    ``_lib.load()`` builds the library -- unless ``B200CTC_LIB`` selects a developer variant of the library, in
    which case nothing is built on demand.  Raises B200CTCError when the extension cannot be built or imported."""
    global _EXT
    if _EXT is None:
        # The library first: every build of it is named libb200ctc.so, so the extension's dependency on that name
        # resolves to the copy already loaded (B200CTC_LIB's variant included) and the loss and the ctypes
        # diagnostics share one library, and one set of handles, per process.
        _lib.load()
        path = _build.extension_path()
        if not os.environ.get("B200CTC_LIB"):
            try:
                _build.build_extension()
            except Exception as exc:      # no host compiler: an extension that exists is used, as for the library
                if not os.path.exists(path):
                    raise B200CTCError("cannot build the PyTorch extension %s: %s" % (path, exc)) from exc
        try:
            spec = importlib.util.spec_from_file_location(_build.EXT_NAME, path)
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
        except Exception as exc:          # missing, or built for another torch / python
            raise B200CTCError("cannot import the PyTorch extension %s: %s" % (path, exc)) from exc
        _EXT = mod
    return _EXT


def _handle(device_index):
    """One library handle per device (the handle serialises its calls with a mutex, include/b200ctc.h), created
    by the extension and shared with the ctypes entry points (diagnostics, decoders)."""
    h = _HANDLES.get(device_index)
    if h is None:
        h = _HANDLES[device_index] = ctypes.c_void_p(_ext().handle_address(int(device_index)))
    return h


def release_workspaces():
    """Drop the cached workspaces (they are re-allocated on the next call)."""
    _ext().release_workspaces()


def set_profiling(enable, device_index=None):
    """Bracket each kernel of the following ctc_loss_and_grad calls with CUDA events (bench only)."""
    if device_index is None:
        device_index = torch.cuda.current_device()
    _lib.check(_lib.load().b200ctc_set_profiling(_handle(device_index), 1 if enable else 0), "b200ctc_set_profiling")


def last_kernel_ms(device_index=None):
    """Device time (ms) of the last call's kernels: (softmax rows, lattice, cost sum)."""
    if device_index is None:
        device_index = torch.cuda.current_device()
    ms = (ctypes.c_float * 3)()
    _lib.check(_lib.load().b200ctc_get_last_kernel_ms(_handle(device_index), ms), "b200ctc_get_last_kernel_ms")
    return tuple(float(x) for x in ms)


def last_fallbacks(device_index=None, with_invalid=False):
    """(extreme_rows, range_lost): utterances of the last call that took the fp64 safe lattice;
    with_invalid=True appends the number of utterances a device-resident call rejected (cost NaN)."""
    if device_index is None:
        device_index = torch.cuda.current_device()
    c = (ctypes.c_int * 3)()
    _lib.check(_lib.load().b200ctc_get_last_fallbacks(_handle(device_index), c,
                                                      torch.cuda.current_stream().cuda_stream),
               "b200ctc_get_last_fallbacks")
    return (int(c[0]), int(c[1]), int(c[2])) if with_invalid else (int(c[0]), int(c[1]))


def plan_cache_stats(device_index=None):
    """(hits, misses) of the host-label call's plan cache on this device's handle."""
    if device_index is None:
        device_index = torch.cuda.current_device()
    h, m = ctypes.c_longlong(), ctypes.c_longlong()
    _lib.check(_lib.load().b200ctc_get_plan_cache_stats(_handle(device_index), ctypes.byref(h), ctypes.byref(m)),
               "b200ctc_get_plan_cache_stats")
    return int(h.value), int(m.value)


def _host_i32(x, name):
    """labels / lengths arrive as CPU int32 tensors in the reference (ctc.py:295-297,321);
    numpy arrays and lists are accepted too.  Returns a C-contiguous int32 numpy array."""
    if isinstance(x, np.ndarray) and x.dtype == np.int32 and x.ndim == 1 and x.flags.c_contiguous:
        return x
    if isinstance(x, torch.Tensor):
        if x.is_cuda:
            x = x.cpu()  # the warp-ctc contract keeps these on the host; tolerate device tensors
        x = x.detach().numpy()
    arr = np.ascontiguousarray(np.asarray(x), dtype=np.int32)
    if arr.ndim != 1:
        raise B200CTCError("%s must be 1-dimensional" % name)
    return arr


def _as_cpu_tensor(x):
    """labels / lengths for the extension's host-label entry point: a 1-D CPU int32 tensor (no copy for int32 numpy)."""
    if isinstance(x, torch.Tensor):
        return x
    return torch.from_numpy(np.ascontiguousarray(np.asarray(x), dtype=np.int32))


def _i32_ptr(arr):
    return arr.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


_REDUCED = (torch.bfloat16, torch.float16)


def _require_cuda(acts, reduced=False):
    """``reduced``: bfloat16 / float16 logits are accepted too (the device-resident loss)."""
    if not isinstance(acts, torch.Tensor) or not acts.is_cuda:
        raise B200CTCError("acts must be a CUDA tensor: this engine has no CPU path "
                           "(the CPU restatement lives in oracle/ for tests only)")
    if acts.dtype != torch.float32 and not (reduced and acts.dtype in _REDUCED):
        raise B200CTCError("acts must be %s, got %s" % ("float32, bfloat16 or float16" if reduced else "float32",
                                                        acts.dtype))
    if acts.dim() != 3:
        raise B200CTCError("acts must be [T, B, V]")


def workspace_bytes(label_lens, act_lens, T, V):
    lib = _lib.load()
    label_lens = _host_i32(label_lens, "label_lens")
    act_lens = _host_i32(act_lens, "act_lens")
    n = ctypes.c_size_t()
    _lib.check(lib.b200ctc_get_workspace_size(_i32_ptr(label_lens), _i32_ptr(act_lens), int(T), int(V),
                                              len(act_lens), ctypes.byref(n)), "b200ctc_get_workspace_size")
    return n.value


def workspace_bound(T, V, B, max_label_len):
    """Workspace size from the shape alone (what the device-resident call uses)."""
    n = ctypes.c_size_t()
    _lib.check(_lib.load().b200ctc_get_workspace_bound(int(T), int(V), int(B), int(max_label_len), ctypes.byref(n)),
               "b200ctc_get_workspace_bound")
    return n.value


def _scale_grads(grads, scale):
    """``grads * scale`` for backward; ``scale`` is grad_output: a 0-dim tensor, or ``[B]`` (one per utterance).  A
    bfloat16 / float16 gradient is multiplied in fp32 and rounded once, in one pass of b200ctc_scale_grads: a plain
    ``grads * scale`` would round the fp32 ``scale`` to the gradient's dtype first (a GradScaler's 2^16 is inf in
    float16)."""
    if grads.dtype == torch.float32:
        return grads * (scale.reshape(1, -1, 1) if scale.dim() else scale)
    try:
        return _ext().scale_grads(grads, scale)
    except RuntimeError as exc:
        raise B200CTCError(str(exc).split("\n")[0])


def ctc_loss_and_grad(acts, labels, act_lens, label_lens, blank=0, grads=None, need_grad=True,
                      costs=None, loss_sum=None, max_label_len=None, logit_scale=1.0, label_smoothing=0.0,
                      loss_scale=1.0, grad_scale=1.0, ls_costs=None):
    """One fused cost-and-gradient evaluation on the current CUDA stream.

    acts [T,B,V] CUDA fp32 logits (any strides with a unit vocabulary stride, e.g. the
    ``logits.transpose(0, 1)`` view the reference passes, ctc.py:319 -- no copy is made).  With device-resident
    labels bfloat16 and float16 logits are accepted as well: they are widened to fp32 as they are loaded, the
    gradient is formed in fp32 and rounded once into a tensor of their dtype, and the costs stay fp32.  The result
    is the fp32 evaluation of ``acts.float()`` with its gradient cast by ``.to(acts.dtype)``.
    Two forms of labels / lengths:
      * host-resident (the warp-ctc contract, ctc.py:295-297,321): flat int32 ``labels`` and ``act_lens`` /
        ``label_lens`` as CPU tensors, numpy arrays or lists -- planned on the host, tables copied by the call;
      * device-resident: ``labels`` a CUDA int32 tensor ``[B, Lmax]`` (padded; entries past ``label_lens[b]`` are
        ignored) with CUDA int32 ``act_lens`` / ``label_lens`` -- planned by a kernel, the call is kernel
        launches only and can be captured into a CUDA graph (``max_label_len`` defaults to ``Lmax``).
    ``logit_scale`` / ``label_smoothing`` / ``loss_scale`` / ``grad_scale`` (device-resident form only) fuse the
    arithmetic of the reference's call site into the kernels (b200ctc_options, include/b200ctc.h):
    logits * logit_scale (1/temperature, ctc.py:306-307), loss_sum = loss_scale * sum_b[(1-ls) cost_b + ls/V * XE_b]
    (ctc.py:323,329-337), grads = grad_scale * d(loss_sum/loss_scale)/d(scaled logits).
    Returns device tensors ``(costs[B], loss_sum[1], grads[T,B,V] or None)``; nothing synchronises the host.
    """
    _require_cuda(acts, reduced=True)
    ext = _ext()
    try:
        if isinstance(labels, torch.Tensor) and labels.is_cuda:
            return ext.loss_and_grad_dev(acts, labels, act_lens, label_lens, int(blank), grads, bool(need_grad), costs,
                                         loss_sum, -1 if max_label_len is None else int(max_label_len),
                                         float(logit_scale), float(label_smoothing), float(loss_scale),
                                         float(grad_scale), ls_costs)
        if logit_scale != 1.0 or label_smoothing != 0.0 or loss_scale != 1.0 or grad_scale != 1.0:
            raise B200CTCError("logit_scale / label_smoothing / loss_scale / grad_scale need device-resident labels "
                               "(the warp-ctc style call has no such arguments); see ctc_loss_from_padded")
        if acts.dtype != torch.float32:
            raise B200CTCError("%s logits need device-resident labels (CUDA tensors); the warp-ctc style call with "
                               "host labels takes float32 only" % acts.dtype)
        return ext.loss_and_grad_host(acts, _as_cpu_tensor(labels), _as_cpu_tensor(act_lens), _as_cpu_tensor(label_lens),
                                      int(blank), grads, bool(need_grad), costs, loss_sum)
    except B200CTCError:
        raise
    except (RuntimeError, TypeError) as exc:
        raise B200CTCError(str(exc).split("\n")[0])


# ------------------------------------------------------------------------------------------------
# warpctc_pytorch surface
# ------------------------------------------------------------------------------------------------

def gpu_ctc(acts, grads, labels, label_lens, act_lens, minibatch_size, costs, blank=0):
    """Drop-in for ``warpctc_pytorch.gpu_ctc`` (reference call: ctc.py:35,39-45).
    ``grads`` (CUDA, same shape as acts) and ``costs`` (CPU float32 [B]) are filled in place."""
    _require_cuda(acts)
    if int(minibatch_size) != acts.size(1):
        raise B200CTCError("minibatch_size=%d does not match acts.size(1)=%d" % (minibatch_size, acts.size(1)))
    dev_costs, _, _ = ctc_loss_and_grad(acts, labels, act_lens, label_lens, blank=blank, grads=grads)
    costs.copy_(dev_costs)  # device -> host: the legacy surface returns per-utterance costs on the CPU
    return 0


def cpu_ctc(*_args, **_kwargs):
    raise B200CTCError("cpu_ctc: this engine is CUDA-only (sm_100a); there is no CPU fallback")


class _CTC(torch.autograd.Function):
    """``warpctc_pytorch._CTC``: cost in forward, gradient stashed on ``ctx.grads``."""

    # True reproduces the oldest upstream revision, which ignored grad_output (SURVEY 3.2)
    legacy_ignore_grad_output = False

    @staticmethod
    def forward(ctx, acts, labels, act_lens, label_lens, size_average=False, length_average=False, blank=0):
        if not acts.is_cuda:
            cpu_ctc()
        minibatch_size = acts.size(1)
        costs, loss_sum, grads = ctc_loss_and_grad(acts, labels, act_lens, label_lens, blank=blank)
        loss = loss_sum.cpu()  # FloatTensor[1] on the host, as upstream returns it
        if length_average:
            total_length = float(_host_i32(act_lens, "act_lens").sum())
            grads = grads / total_length
            loss = loss / total_length
        elif size_average:
            grads = grads / minibatch_size
            loss = loss / minibatch_size
        ctx.grads = grads
        return loss

    @staticmethod
    def backward(ctx, grad_output):
        grads = ctx.grads
        if isinstance(grads, torch.Tensor) and not _CTC.legacy_ignore_grad_output:
            grads = grads * grad_output.to(grads.device).reshape(-1)[0]
        # one slot per forward input: 7 here, 5 for the reference's override (ctc.py:32)
        return (grads,) + (None,) * (len(ctx.needs_input_grad) - 1)


class CTCLoss(torch.nn.Module):
    """``warpctc_pytorch.CTCLoss`` (instantiated by the reference at ctc.py:69).

    size_average: divide cost and gradient by the mini-batch size;
    length_average: divide by the total number of frames; blank: blank symbol index.
    """

    def __init__(self, size_average=False, length_average=False, blank=0):
        super().__init__()
        self.ctc = _CTC.apply
        self.size_average = size_average
        self.length_average = length_average
        self.blank = blank

    def forward(self, acts, labels, act_lens, label_lens):
        if labels.dim() != 1:
            raise B200CTCError("labels must be 1 dimensional")
        for name, x in (("labels", labels), ("act_lens", act_lens), ("label_lens", label_lens)):
            if isinstance(x, torch.Tensor) and x.requires_grad:
                raise B200CTCError("%s must not require gradients" % name)
        return self.ctc(acts, labels, act_lens, label_lens, self.size_average, self.length_average, self.blank)


# ------------------------------------------------------------------------------------------------
# native API: device-resident loss, no host synchronisation
# ------------------------------------------------------------------------------------------------

class _CTCDevice(torch.autograd.Function):
    @staticmethod
    def forward(ctx, acts, labels, act_lens, label_lens, blank, reduction):
        costs, loss_sum, grads = ctc_loss_and_grad(acts, labels, act_lens, label_lens, blank=blank,
                                                   need_grad=acts.requires_grad)
        ctx.grads = grads
        ctx.reduction = reduction
        if reduction == "none":
            return costs
        if reduction == "mean":
            return loss_sum / acts.size(1)
        return loss_sum

    @staticmethod
    def backward(ctx, grad_output):
        if ctx.reduction == "none":
            g = _scale_grads(ctx.grads, grad_output.reshape(-1))
        elif ctx.reduction == "mean":
            g = _scale_grads(ctx.grads, grad_output.reshape(-1)[0] / ctx.grads.size(1))
        else:
            g = _scale_grads(ctx.grads, grad_output.reshape(-1)[0])
        return g, None, None, None, None, None


def ctc_loss(acts, labels, act_lens, label_lens, blank=0, reduction="sum"):
    """Device-resident CTC loss: returns a CUDA tensor ([1] for 'sum'/'mean', [B] for 'none').  ``acts`` may be
    fp32, bfloat16 or float16; the loss is fp32 and the gradient has the dtype of ``acts``."""
    if reduction not in ("sum", "mean", "none"):
        raise B200CTCError("reduction must be 'sum', 'mean' or 'none'")
    return _CTCDevice.apply(acts, labels, act_lens, label_lens, blank, reduction)


# ------------------------------------------------------------------------------------------------
# call-site helpers (SURVEY 8(f) rank 1): what CTC.forward does around the op, without the python loop,
# the transpose copy and the host round trips
# ------------------------------------------------------------------------------------------------

def concatenate_labels(ys, y_lens):
    """Vectorised ``_concatenate_labels`` (reference: models/pytorch_v3/ctc/ctc.py:532-549, a python loop
    over the mini-batch): padded ``ys[B, Lmax]`` + ``y_lens[B]`` -> flat int32 ``[sum(y_lens)]`` on the host."""
    ys = ys.detach().cpu().numpy() if isinstance(ys, torch.Tensor) else np.asarray(ys)
    y_lens = _host_i32(y_lens, "y_lens")
    if ys.ndim != 2 or ys.shape[0] != len(y_lens):
        raise B200CTCError("ys must be [B, Lmax] with one length per row")
    if len(y_lens) and int(y_lens.max(initial=0)) > ys.shape[1]:
        raise B200CTCError("y_lens exceeds the padded label width")
    mask = np.arange(ys.shape[1])[None, :] < y_lens[:, None]
    return np.ascontiguousarray(ys[mask], dtype=np.int32)


class _CTCFromPadded(torch.autograd.Function):
    """The whole loss computation of ``CTC.forward`` as ONE device-resident call: temperature, ``/ len(xs)`` and
    the label-smoothing cross entropy are evaluated inside the kernels (b200ctc_options)."""

    @staticmethod
    def forward(ctx, logits, ys, x_lens, y_lens, inv_temperature, label_smoothing, loss_scale):
        need_grad = logits.requires_grad
        _, loss, grads = ctc_loss_and_grad(
            logits.transpose(0, 1), ys, x_lens, y_lens, blank=0, need_grad=need_grad,
            logit_scale=inv_temperature, label_smoothing=label_smoothing, loss_scale=loss_scale,
            grad_scale=loss_scale * inv_temperature)      # d loss / d (unscaled, batch-major) logits
        ctx.grads = grads
        return loss

    @staticmethod
    def backward(ctx, grad_output):
        g = _scale_grads(ctx.grads, grad_output.reshape(-1)[0])        # [T, B, V]
        return g.transpose(0, 1), None, None, None, None, None, None


def _dev_padded_labels(ys, y_lens, dev, label_offset):
    """Padded ``ys[B, Lmax]`` (+ ``label_offset``) and ``y_lens[B]`` as CUDA int32 tensors (the reference keeps
    them on the host, ctc.py:295-297: they are uploaded here, a few kilobytes)."""
    ys = torch.as_tensor(ys) if not isinstance(ys, torch.Tensor) else ys
    y_lens = torch.as_tensor(y_lens) if not isinstance(y_lens, torch.Tensor) else y_lens
    if ys.dim() != 2 or ys.size(0) != y_lens.numel():
        raise B200CTCError("ys must be [B, Lmax] with one length per row")
    ys = ys.to(device=dev, dtype=torch.int32)
    if label_offset:
        ys = ys + int(label_offset)
    return ys.contiguous(), y_lens.to(device=dev, dtype=torch.int32).contiguous()


def ctc_loss_from_padded(logits, ys, x_lens, y_lens, label_offset=1, logits_temperature=1.0, average=True,
                         label_smoothing=0.0):
    """The loss computation of ``CTC.forward`` (reference: ctc.py:299-337) as one call, device resident.

    logits ``[B, T, V]`` CUDA (batch-major, as the encoder returns them; consumed through a strided view,
    no ``transpose().contiguous()`` copy), ys ``[B, Lmax]`` padded labels WITHOUT the blank offset
    (``label_offset=1`` reproduces ``ys = ys + 1``, ctc.py:300: index 0 is the blank), x_lens / y_lens ``[B]``
    (host or device).  ``logits_temperature`` is the reference's "output smoothing" (ctc.py:306-307),
    ``average=True`` its ``/ len(xs)`` (ctc.py:323), ``label_smoothing`` its ``ls_prob`` (ctc.py:329-337 with
    models/pytorch_v3/criterion.py:51-80): all three are evaluated inside the kernels, not as tensor passes.
    Returns a CUDA tensor ``[1]``:  ``(1-ls) * sum_b cost_b / B + ls/V * sum_b sum_{t<x_lens[b]} sum_k -lp[b,t,k] / B``
    that back-propagates into ``logits``.  ``logits`` may be fp32, bfloat16 or float16 (the output of a projection
    under ``torch.autocast``): the loss is fp32 and the gradient has the dtype of ``logits``.
    """
    if logits.dim() != 3:
        raise B200CTCError("logits must be [B, T, V]")
    _require_cuda(logits, reduced=True)
    dev = logits.device
    ys_d, y_lens_d = _dev_padded_labels(ys, y_lens, dev, label_offset)
    x_lens_d = (x_lens if isinstance(x_lens, torch.Tensor) else torch.as_tensor(np.asarray(x_lens))).to(
        device=dev, dtype=torch.int32).contiguous()
    B = logits.size(0)
    loss_scale = 1.0 / B if (average and B > 0) else 1.0
    return _CTCFromPadded.apply(logits, ys_d, x_lens_d, y_lens_d, 1.0 / float(logits_temperature),
                                float(label_smoothing), loss_scale)
