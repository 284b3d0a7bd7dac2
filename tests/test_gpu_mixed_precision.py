"""bfloat16 / float16 logits in the device-resident CTC loss.

Every result is compared with the composition it replaces: the fp32 engine on the widened logits,
``ctc_loss_and_grad(acts.float(), ...)``, with its gradient rounded by ``.to(dtype)``.  Where K1 assigns row
elements to lanes by index (the warp-per-row kernel, V <= 256) the two must be bit-identical; the streaming and
CTA-per-row kernels read a reduced-precision row in other groupings, so their fp32 sums may differ in the last bit
and a gradient element may land one ulp of the dtype away."""
import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
import test_gpu_peaked as pk
from oracle import ctc_ref, peaked_ref
from pytorch_end2end_speech_recognition_b200 import ctc as ctc_mod

pytestmark = pytest.mark.gpu

DTYPES = [torch.bfloat16, torch.float16]
REL_ULP = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}   # one ulp, relative, of the dtype


def ordered_bits(x):
    """Integers in the order of the dtype's values (-0 and +0 both 0): adjacent values differ by one."""
    i = x.view(torch.int16).to(torch.int32)
    return torch.where(i < 0, -(i & 0x7FFF), i)


def assert_within_one_ulp(g, g_ref, what=""):
    assert g.dtype == g_ref.dtype and g.shape == g_ref.shape
    d = (ordered_bits(g) - ordered_bits(g_ref)).abs()
    assert int(d.max()) <= 1, "%s: %d elements more than one ulp away" % (what, int((d > 1).sum()))


def ragged_batch(V, seed, B=6, T=50, Lmax=12, infeasible=True):
    """Batch with padding frames, an empty label sequence and (optionally) an infeasible utterance."""
    rng = np.random.RandomState(seed)
    act_lens = rng.randint(T // 2, T + 1, size=B).astype(np.int32)
    act_lens[0] = T
    label_lens = rng.randint(1, Lmax + 1, size=B).astype(np.int32)
    label_lens[1] = 0                                          # L = 0
    if infeasible:
        act_lens[2], label_lens[2] = 5, Lmax                   # L > T_b: cost +inf, zero gradient
    labels = np.concatenate([rng.randint(1, V, size=L) for L in label_lens]).astype(np.int32)
    acts = rng.randn(T, B, V).astype(np.float32) * 2.0
    return acts, labels, act_lens, label_lens


def batch_major(acts, dtype):
    """[T, B, V] numpy -> the reference's batch-major [B, T, V] CUDA tensor of `dtype`, viewed as [T, B, V]."""
    logits = torch.from_numpy(acts).transpose(0, 1).contiguous().cuda().to(dtype)
    return logits, logits.transpose(0, 1)


def composition(acts, labels_d, act_lens_d, label_lens_d, need_grad=True):
    c, l, g = b200.ctc_loss_and_grad(acts.float(), labels_d, act_lens_d, label_lens_d, need_grad=need_grad)
    return c, l, (g.to(acts.dtype) if g is not None else None)


def run_both(acts, labels, act_lens, label_lens):
    dev = pk.device_args(labels, act_lens, label_lens)
    c, l, g = b200.ctc_loss_and_grad(acts, *dev)
    fb = ctc_mod.last_fallbacks(with_invalid=True)
    c_ref, l_ref, g_ref = composition(acts, *dev)
    fb_ref = ctc_mod.last_fallbacks(with_invalid=True)
    torch.cuda.synchronize()
    assert c.dtype == torch.float32 and l.dtype == torch.float32 and g.dtype == acts.dtype
    return (c, l, g, fb), (c_ref, l_ref, g_ref, fb_ref)


# ---- bit-identical: the warp-per-row softmax --------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", [30, 62, 129, 256])
def test_warp_kernel_results_are_bit_identical_to_the_composition(V, dtype):
    acts_np, labels, act_lens, label_lens = ragged_batch(V, seed=V)
    _, acts = batch_major(acts_np, dtype)
    (c, l, g, fb), (c_ref, l_ref, g_ref, fb_ref) = run_both(acts, labels, act_lens, label_lens)
    assert torch.equal(c, c_ref) and torch.equal(l, l_ref)
    assert torch.equal(g.view(torch.int16), g_ref.view(torch.int16))
    assert fb == fb_ref
    assert torch.isinf(c[2]) and not g[:, 2].view(torch.int16).any()           # infeasible: +inf, +0 gradient
    for b, Tb in enumerate(act_lens):
        assert not g[Tb:, b].view(torch.int16).any()                              # padding rows: exact +0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", [30, 62, 129, 256])
def test_call_site_is_bit_identical_to_the_composition(V, dtype):
    """ctc_loss_from_padded with temperature 1.3 and label smoothing 0.1, back-propagated into the logits."""
    acts_np, labels, act_lens, label_lens = ragged_batch(V, seed=100 + V, infeasible=False)
    ys = pk.padded_labels(labels - 1, label_lens, pad=0)
    logits, _ = batch_major(acts_np, dtype)
    lg = logits.clone().requires_grad_(True)
    loss = b200.ctc_loss_from_padded(lg, ys, act_lens, label_lens, logits_temperature=1.3, label_smoothing=0.1)
    loss.backward()
    lg32 = logits.float().requires_grad_(True)
    loss_ref = b200.ctc_loss_from_padded(lg32, ys, act_lens, label_lens, logits_temperature=1.3, label_smoothing=0.1)
    loss_ref.backward()
    assert loss.dtype == torch.float32 and torch.equal(loss, loss_ref)
    assert lg.grad.dtype == dtype
    assert torch.equal(lg.grad.view(torch.int16), lg32.grad.to(dtype).view(torch.int16))


# ---- one ulp: the streaming and CTA-per-row softmax ------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", [257, 3386, 14075])
def test_large_vocabulary_within_one_ulp_of_the_composition(V, dtype):
    B, T = (6, 50) if V < 10000 else (3, 24)
    acts_np, labels, act_lens, label_lens = ragged_batch(V, seed=V, B=B, T=T, Lmax=10)
    _, acts = batch_major(acts_np, dtype)
    (c, l, g, fb), (c_ref, l_ref, g_ref, fb_ref) = run_both(acts, labels, act_lens, label_lens)
    assert fb == fb_ref
    f = torch.isfinite(c_ref)
    assert torch.equal(torch.isinf(c), ~f)
    assert torch.allclose(c[f], c_ref[f], rtol=1e-5, atol=0)
    assert_within_one_ulp(g, g_ref, "V=%d" % V)
    for b, Tb in enumerate(act_lens):
        assert not g[Tb:, b].view(torch.int16).any()
    # the fp64 oracle on the widened logits: its tolerance plus the one rounding to the dtype
    wide = acts.float().cpu().numpy()
    c64, g64 = ctc_ref.ctc_cost_and_grad(wide, labels, act_lens, label_lens)
    cf = np.isfinite(c64)
    assert np.allclose(c.cpu().numpy()[cf], c64[cf], rtol=1e-5, atol=0)
    gg = g.float().cpu().numpy()
    assert np.all(np.abs(gg - g64) <= 1e-4 + REL_ULP[dtype] * np.abs(g64))


# ---- the fp64 safe lattice on reduced-precision logits ---------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", [30, 300])
def test_must_redo_case_on_reduced_logits(V, dtype):
    utts = pk.redo_utterances(V)
    acts_np, labels, act_lens, label_lens = pk.batch(utts)
    acts = torch.from_numpy(acts_np).cuda().to(dtype)
    (c, l, g, fb), (c_ref, l_ref, g_ref, fb_ref) = run_both(acts, labels, act_lens, label_lens)
    assert fb_ref[1] > 0, "the rounded case no longer loses range: %s" % (fb_ref,)
    assert fb == fb_ref
    if V <= 256:
        assert torch.equal(c, c_ref) and torch.equal(g.view(torch.int16), g_ref.view(torch.int16))
    else:
        assert torch.allclose(c, c_ref, rtol=1e-5, atol=0)
        assert_within_one_ulp(g, g_ref, "redo V=%d" % V)


@pytest.mark.parametrize("V", [30, 300])
def test_extreme_row_in_bfloat16(V):
    acts_np, labels, act_lens, label_lens = pk.edge_batch(V, -69.5, 1.0)
    acts = torch.from_numpy(acts_np).cuda().to(torch.bfloat16)
    wide = acts.float().cpu().numpy()
    assert peaked_ref.min_log_prob(wide[:act_lens[0], 0]) < -69.0        # still past K1's threshold once rounded
    (c, l, g, fb), (c_ref, l_ref, g_ref, fb_ref) = run_both(acts, labels, act_lens, label_lens)
    assert fb == fb_ref == (1, 0, 0)
    if V <= 256:
        assert torch.equal(c, c_ref) and torch.equal(g.view(torch.int16), g_ref.view(torch.int16))
    else:
        f = torch.isfinite(c_ref)
        assert torch.equal(torch.isinf(c), ~f) and torch.allclose(c[f], c_ref[f], rtol=1e-5, atol=0)
        assert_within_one_ulp(g, g_ref, "edge V=%d" % V)


# ---- range and padding -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [30, 300])
def test_float16_logits_near_the_range_limit_stay_finite(V):
    acts_np, labels, act_lens, label_lens = ragged_batch(V, seed=7 + V, infeasible=False)
    acts_np[3, 0, 1] = 6.0e4
    acts_np[4, 0, 2] = -6.0e4
    acts_np[10, 3, :] = -6.0e4
    acts_np[10, 3, 0] = 6.0e4
    acts_np[act_lens[4]:, 4] = 6.0e4                                   # padding frames: never read
    _, acts = batch_major(acts_np, torch.float16)
    assert torch.isfinite(acts).all()
    (c, l, g, fb), (c_ref, l_ref, g_ref, fb_ref) = run_both(acts, labels, act_lens, label_lens)
    assert torch.isfinite(c).all() and torch.isfinite(g).all()
    assert fb == fb_ref and fb[0] > 0
    if V <= 256:
        assert torch.equal(c, c_ref) and torch.equal(g.view(torch.int16), g_ref.view(torch.int16))
    else:
        assert torch.allclose(c, c_ref, rtol=1e-5, atol=0)
        assert_within_one_ulp(g, g_ref)
    for b, Tb in enumerate(act_lens):
        assert not g[Tb:, b].view(torch.int16).any()


def test_cost_only_call_matches():
    acts_np, labels, act_lens, label_lens = ragged_batch(300, seed=5)
    _, acts = batch_major(acts_np, torch.bfloat16)
    dev = pk.device_args(labels, act_lens, label_lens)
    c, l, g = b200.ctc_loss_and_grad(acts, *dev, need_grad=False)
    c_ref, l_ref, _ = composition(acts, *dev, need_grad=False)
    f = torch.isfinite(c_ref)
    assert g is None and torch.equal(torch.isinf(c), ~f) and torch.allclose(c[f], c_ref[f], rtol=1e-5, atol=0)


# ---- backward: grad_output multiplied in fp32, one rounding ----------------------------------------------------
def expected_scaled(g, scale):
    """grads * grad_output formed in fp32 and rounded once to the gradient's dtype."""
    s = scale.reshape(1, -1, 1) if scale.dim() else scale
    return (g.float() * s.float()).to(g.dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("reduction", ["sum", "mean", "none"])
@pytest.mark.parametrize("V", [30, 300])
def test_ctc_loss_backward_scales_in_fp32(V, reduction, dtype):
    acts_np, labels, act_lens, label_lens = ragged_batch(V, seed=40 + V, infeasible=False)
    _, acts = batch_major(acts_np, dtype)
    dev = pk.device_args(labels, act_lens, label_lens)
    _, _, g = b200.ctc_loss_and_grad(acts, *dev)
    x = acts.detach().requires_grad_(True)
    loss = b200.ctc_loss(x, *dev, reduction=reduction)
    go = torch.rand(loss.shape, device="cuda") * 3.0 + 0.1          # not representable in the dtype
    loss.backward(go)
    scale = go.reshape(-1) if reduction == "none" else go.reshape(-1)[0] / (acts.size(1) if reduction == "mean" else 1)
    assert x.grad.dtype == dtype
    assert torch.equal(x.grad.view(torch.int16), expected_scaled(g, scale).view(torch.int16))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("per_utterance", [False, True])
@pytest.mark.parametrize("aligned", [True, False])
def test_scale_kernel_layouts(dtype, per_utterance, aligned):
    """Vector body and scalar path; per-utterance scales whose rows straddle the eight-element groups (V = 30)."""
    T, B, V = 37, 5, 30
    n = T * B * V
    buf = (torch.randn(n + 1, device="cuda") * 0.5).to(dtype)
    g = (buf[:n] if aligned else buf[1:]).view(T, B, V)
    scale = torch.rand(B if per_utterance else 1, device="cuda") * 5.0 + 0.1
    out = ctc_mod._ext().scale_grads(g, scale)
    ref = expected_scaled(g, scale if per_utterance else scale.reshape(()))
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


def test_grad_scaler_factor_stays_finite_in_float16():
    """2^16 (a GradScaler's initial scale) is inf in float16: the gradient must be multiplied by it in fp32."""
    acts_np, labels, act_lens, label_lens = ragged_batch(30, seed=9, infeasible=False)
    _, acts = batch_major(acts_np, torch.float16)
    dev = pk.device_args(labels, act_lens, label_lens)
    x = acts.detach().requires_grad_(True)
    loss = b200.ctc_loss(x, *dev)
    loss.backward(torch.full_like(loss, 65536.0))
    _, _, g = b200.ctc_loss_and_grad(acts, *dev)
    small = g.float().abs() < 0.5                                 # 0.5 * 2^16 < 65504
    assert small.any() and torch.isfinite(x.grad[small]).all()
    assert torch.equal(x.grad.view(torch.int16), expected_scaled(g, torch.tensor(65536.0, device="cuda")).view(torch.int16))


# ---- CUDA graph, determinism -----------------------------------------------------------------------------------
def test_bfloat16_call_in_a_cuda_graph_equals_the_eager_call():
    acts_np, labels, act_lens, label_lens = ragged_batch(300, seed=11, B=8, T=60)
    _, acts = batch_major(acts_np, torch.bfloat16)
    dev = pk.device_args(labels, act_lens, label_lens)
    c0, l0, g0 = b200.ctc_loss_and_grad(acts, *dev)
    c1, l1, g1 = b200.ctc_loss_and_grad(acts, *dev)
    assert torch.equal(c0, c1) and torch.equal(l0, l1) and torch.equal(g0.view(torch.int16), g1.view(torch.int16))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        b200.ctc_loss_and_grad(acts, *dev)                         # warm-up: the stream's workspace
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        cg, lg, gg = b200.ctc_loss_and_grad(acts, *dev)
    for _ in range(2):
        cg.zero_(); gg.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(cg, c0) and torch.equal(lg, l0) and torch.equal(gg.view(torch.int16), g0.view(torch.int16))


# ---- end to end under autocast ---------------------------------------------------------------------------------
def _autocast_step(lin, x, ys, x_lens, y_lens, widen):
    lin.weight.grad = None
    lin.bias.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16):
        logits = lin(x)
    assert logits.dtype == torch.bfloat16
    if widen:                                                  # the workaround: an fp32 copy of the logits
        logits = logits.float()
    loss = b200.ctc_loss_from_padded(logits, ys, x_lens, y_lens)
    loss.backward()
    return loss.detach(), lin.weight.grad.clone(), lin.bias.grad.clone()


def _model(V, H, B, T, seed):
    torch.manual_seed(seed)
    lin = torch.nn.Linear(H, V).cuda()
    x = torch.randn(B, T, H, device="cuda")
    return lin, x


def test_autocast_linear_backward_equals_the_composition():
    wl_V, H, B, T = 62, 96, 8, 120
    lin, x = _model(wl_V, H, B, T, 0)
    rng = np.random.RandomState(1)
    x_lens = np.sort(rng.randint(T // 2, T + 1, size=B))[::-1].astype(np.int32)
    y_lens = rng.randint(5, 30, size=B).astype(np.int32)
    ys = rng.randint(0, wl_V - 1, size=(B, 30)).astype(np.int64)
    loss, gw, gb = _autocast_step(lin, x, ys, x_lens, y_lens, widen=False)
    loss_ref, gw_ref, gb_ref = _autocast_step(lin, x, ys, x_lens, y_lens, widen=True)
    assert torch.equal(loss, loss_ref)
    assert torch.equal(gw, gw_ref) and torch.equal(gb, gb_ref)


def test_autocast_step_at_c4_shape_uses_less_memory_than_the_composition():
    """CSJ-shaped (C4: B=64, T=1000, V=3386): the peak memory of one forward + backward step of a bfloat16 projection
    feeding the loss, with the logits passed as they are and with the fp32 workaround."""
    V, H, B, T = 3386, 256, 64, 1000
    lin, x = _model(V, H, B, T, 2)
    rng = np.random.RandomState(3)
    x_lens = np.sort(rng.randint(T // 2, T + 1, size=B))[::-1].astype(np.int32)
    y_lens = rng.randint(75, 151, size=B).astype(np.int32)
    ys = rng.randint(0, V - 1, size=(B, 150)).astype(np.int64)
    peaks, results = {}, {}
    for widen in (True, False, True, False):                     # the second round is measured: warm caches
        ctc_mod.release_workspaces()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        results[widen] = _autocast_step(lin, x, ys, x_lens, y_lens, widen)
        torch.cuda.synchronize()
        peaks[widen] = torch.cuda.max_memory_allocated() - base
    print("\nC4 autocast step peak memory: bf16 logits %.1f MB, fp32 workaround %.1f MB (one fp32 [B,T,V] = %.1f MB)"
          % (peaks[False] / 1e6, peaks[True] / 1e6, 4 * B * T * V / 1e6))
    assert peaks[False] < peaks[True]
    loss, gw, gb = results[False]
    loss_ref, gw_ref, gb_ref = results[True]
    assert torch.allclose(loss, loss_ref, rtol=1e-5, atol=0)
    assert torch.allclose(gw, gw_ref, rtol=2e-2, atol=1e-3 * float(gw_ref.abs().max()))
    assert torch.allclose(gb, gb_ref, rtol=2e-2, atol=1e-3 * float(gb_ref.abs().max()))


# ---- what stays fp32 only --------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
def test_reduced_logits_with_host_labels_raise(dtype):
    acts_np, labels, act_lens, label_lens = ragged_batch(30, seed=2, infeasible=False)
    acts = torch.from_numpy(acts_np).cuda().to(dtype)
    with pytest.raises(b200.B200CTCError):
        b200.ctc_loss_and_grad(acts, labels, act_lens, label_lens)
    grads = torch.zeros_like(acts)
    with pytest.raises(b200.B200CTCError):
        b200.gpu_ctc(acts, grads, torch.from_numpy(labels), torch.from_numpy(label_lens), torch.from_numpy(act_lens),
                     acts.size(1), torch.zeros(acts.size(1)))
    with pytest.raises(b200.B200CTCError):                     # float64 stays out on the device path too
        b200.ctc_loss_and_grad(acts.double(), *pk.device_args(labels, act_lens, label_lens))
