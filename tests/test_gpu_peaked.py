"""The CTC loss on peaked posteriors -- what a trained acoustic model produces: probability near one on the aligned
symbol, e^-20 .. e^-60 on the others, and stretches it misrecognises.  Covers the fast lattice's range check and the
fp64 redo it triggers (FLAG_PRECISION_LOST: gradient rows the fast reducers already rewrote are rebuilt), K1's
extreme-row threshold at its edge, the CTA-per-row softmax kernel, the plan kernel's large-batch branch and K1's
lane-geometry switches.

Every case is checked against the fp64 oracle, a bit-identical twin call, or an exact property (a zero row, a NaN
cost, a fallback count).  Which utterances must be redone and which must stay on the fast lattice is predicted on the
CPU by oracle/peaked_ref.py; the tests without the gpu mark verify those declarations."""
import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from oracle import ctc_ref, peaked_ref
from oracle.ctc_cpu import ctc_cpu
from pytorch_end2end_speech_recognition_b200 import ctc as ctc_mod

GRAD_ATOL = 1e-4
COST_RTOL = 1e-5
# Cost floor for near-certain alignments (c_ref < 1): fp32 softmax and lattice resolve a probability near one to
# about 2^-24 per frame (K1 alone rounds y of the aligned symbol that finely), so a cost of 1e-5 cannot be held to
# 1e-5 relative; it is held to T_b * 2^-23 absolute instead.
COST_FLOOR_PER_FRAME = 2.0 ** -23
CALL_SITE_SCALE = 1.0 / 1.3          # logits_temperature 1.3

# ---------------------------------------------------------------------------------------------------------------
# cases (declared classes are verified on the CPU by the unmarked tests at the end of this file)
# ---------------------------------------------------------------------------------------------------------------
# Confident model, must stay on the fast lattice: (T, L, margin, error rate) per vocabulary, noise 1, one-frame errors.
STAY_FAST = [(400, 80, 5, 0.0), (400, 80, 5, 0.05), (400, 80, 5, 0.2),
             (800, 120, 10, 0.0), (800, 120, 10, 0.05), (800, 120, 10, 0.2),
             (400, 80, 20, 0.0), (400, 80, 20, 0.05), (400, 80, 20, 0.2)]
# Must be redone by the safe lattice: margin 58, noise 0.5, 20 % of the frames in two-frame error runs; (T, L, seed).
REDO_MARGIN, REDO_NOISE, REDO_ERR, REDO_RUN = 58.0, 0.5, 0.2, 2
REDO = {30: [(300, 80, 2), (200, 60, 0)], 300: [(300, 80, 17), (200, 60, 3)], 1500: [(300, 80, 9)]}
EDGE_LEVELS = (-68.5, -69.5)         # min ln y of the edge rows: just inside / just outside K1's threshold (-69)


def utterance(V, T, L, margin, err_rate, seed, noise=1.0, err_run=1):
    """Peaked logits [T, V] (float32) and labels [L] (int32) of one utterance."""
    rng = np.random.RandomState(seed)
    lab = rng.randint(1, V, size=L)
    acts, _ = peaked_ref.peaked_case(rng, T, lab, V, margin, noise, err_rate, err_run)
    return acts, lab.astype(np.int32)


def stay_fast_utterances(V):
    return [utterance(V, T, L, m, e, 1000 * V + 10 * m + int(e * 100)) for T, L, m, e in STAY_FAST]


def redo_utterances(V):
    return [utterance(V, T, L, REDO_MARGIN, REDO_ERR, seed, REDO_NOISE, REDO_RUN) for T, L, seed in REDO[V]]


def benign_twin(V, T, L, seed):
    """Same lengths as REDO's utterance (T, L, seed), margin 10 and no errors: stays on the fast lattice."""
    return utterance(V, T, L, 10.0, 0.0, seed + 5000)


def ordinary_utterance(V, T, L, seed):
    rng = np.random.RandomState(seed)
    return rng.randn(T, V).astype(np.float32), rng.randint(1, V, size=L).astype(np.int32)


def edge_batch(V, level, scale):
    """K1's threshold: three utterances, T = 40.
      0: live rows whose smallest ln y (of the scaled logits) is exactly `level` -- on the blank, on a label, on a
         symbol outside the labels;
      1: a padding frame (t >= T_b) whose smallest ln y is -80;
      2: an infeasible utterance (L > T_b) with a -80 row.
    Only utterance 0 may ever be flagged, and only when level < -69."""
    rng = np.random.RandomState(V + int(-10 * level))
    T = 40
    z = rng.randn(T, 3, V)                                    # scaled logits, fp64

    def place(t, b, k, lvl):
        others = np.delete(z[t, b], k)
        z[t, b, k] = np.logaddexp.reduce(others) + lvl       # y_k = e^lvl / (1 + e^lvl): ln y_k = lvl to 1e-30

    lab0 = rng.randint(1, V, size=10)
    outside = next(k for k in range(1, V) if k not in set(lab0.tolist()))
    for t, k in ((3, 0), (17, int(lab0[4])), (30, outside)):
        place(t, 0, k, level)
    lab1 = rng.randint(1, V, size=8)
    place(35, 1, int(rng.randint(V)), -80.0)
    lab2 = rng.randint(1, V, size=25)
    place(5, 2, int(rng.randint(V)), -80.0)
    acts = (z / scale).astype(np.float32)
    labels = np.concatenate([lab0, lab1, lab2]).astype(np.int32)
    return acts, labels, np.array([40, 30, 20], np.int32), np.array([10, 8, 25], np.int32)


# ---------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------
def batch(utts, T=None, seed=0):
    """[T, B, V] acts (padding frames N(0,1): never read), flat labels, act_lens, label_lens."""
    T = max(a.shape[0] for a, _ in utts) if T is None else T
    V = utts[0][0].shape[1]
    acts = np.random.RandomState(seed).randn(T, len(utts), V).astype(np.float32)
    for b, (a, _) in enumerate(utts):
        acts[:a.shape[0], b] = a
    labels = np.concatenate([lab for _, lab in utts]).astype(np.int32)
    act_lens = np.array([a.shape[0] for a, _ in utts], np.int32)
    label_lens = np.array([len(lab) for _, lab in utts], np.int32)
    return acts, labels, act_lens, label_lens


def padded_labels(labels, label_lens, width=None, pad=-7):
    width = int(label_lens.max(initial=0)) if width is None else width
    ys = np.full((len(label_lens), max(width, 1)), pad, np.int32)
    off = 0
    for b, L in enumerate(label_lens):
        ys[b, :L] = labels[off:off + L]
        off += L
    return ys


def device_args(labels, act_lens, label_lens, width=None):
    return (torch.from_numpy(padded_labels(labels, label_lens, width)).cuda(),
            torch.from_numpy(act_lens.astype(np.int32)).cuda(), torch.from_numpy(label_lens.astype(np.int32)).cuda())


def check_costs(c, c_ref, act_lens, what=""):
    """Relative COST_RTOL for c_ref >= 1, T_b * 2^-23 absolute below; infeasible utterances: +inf on both sides."""
    c = np.asarray(c, np.float64)
    c_ref = np.asarray(c_ref, np.float64)
    inf = np.isinf(c_ref)
    assert np.array_equal(np.isinf(c) & (c > 0), inf), "%s: infeasible utterances differ: %s vs %s" % (what, c, c_ref)
    f = ~inf
    err = np.abs(c[f] - c_ref[f])
    lim = np.where(c_ref[f] >= 1.0, COST_RTOL * np.abs(c_ref[f]), act_lens[f] * COST_FLOOR_PER_FRAME)
    ratio = err / lim
    worst = int(np.argmax(ratio)) if ratio.size else 0
    assert np.all(err <= lim), ("%s: cost error %.3g at c_ref %.6g (limit %.3g); worst relative error %.3g" %
                                (what, err[worst], c_ref[f][worst], lim[worst],
                                 np.max(err / np.maximum(np.abs(c_ref[f]), 1e-30))))
    return float(np.max(ratio, initial=0.0))


def check_grads(g, g_ref, what="", atol=GRAD_ATOL):
    err = float(np.max(np.abs(np.asarray(g, np.float64) - g_ref), initial=0.0))
    assert err < atol, "%s: gradient error %.3g (limit %.3g)" % (what, err, atol)
    return err


def check_parity(c, g, acts, labels, act_lens, label_lens, what=""):
    c_ref, g_ref = ctc_cpu(acts, labels, act_lens, label_lens, 0, precision="f64", need_grad=g is not None)
    ratio = check_costs(c.cpu().numpy(), c_ref, act_lens, what)
    gerr = check_grads(g.cpu().numpy(), g_ref, what) if g is not None else 0.0
    print("%s: worst cost error / limit %.3g, worst gradient error %.3g, fallbacks %s"
          % (what, ratio, gerr, ctc_mod.last_fallbacks(with_invalid=True)))


def check_call_site(logits_np, ys, x_lens, y_lens, temp, ls, what=""):
    """ctc_loss_from_padded (temperature, / B, label smoothing fused) against the fp64 call-site restatement."""
    B = logits_np.shape[0]
    logits = torch.from_numpy(logits_np).cuda().requires_grad_(True)
    loss = b200.ctc_loss_from_padded(logits, ys, x_lens, y_lens, logits_temperature=temp, label_smoothing=ls)
    loss.backward()
    torch.cuda.synchronize()
    loss_ref, g_ref = ctc_ref.ctc_loss_call_site(logits_np, ys, x_lens, y_lens, temp, ls)
    got = float(loss.detach().cpu()[0])
    assert abs(got - loss_ref) <= COST_RTOL * abs(loss_ref), "%s: loss %.9g vs %.9g" % (what, got, loss_ref)
    g = logits.grad.cpu().numpy()
    check_grads(g, g_ref, what, GRAD_ATOL / B)                 # the gradient carries the 1/B of the loss
    for b in range(B):
        assert np.all(g[b, x_lens[b]:] == 0), "%s: padding frames of utterance %d not zero" % (what, b)


def streaming_softmax_max_V():
    """Largest V the streaming K1 kernel takes (softmax_rows.cu, launch_softmax_rows): at least two warps of two
    stages of (V + 6 + 3) & ~3 floats each within 220 KB of shared memory; past it, one CTA per row."""
    def fits(V):
        return (220 * 1024) // (2 * ((V + 6 + 3) & ~3) * 4) >= 2
    V = 257
    while fits(V + 1):
        V += 1
    return V


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cluster", ["0", "1"])
@pytest.mark.parametrize("V", [30, 300])
def test_confident_model_stays_on_the_fast_lattice(V, cluster, monkeypatch):
    """Margins 5-20, 0 / 5 / 20 % recognition errors, T up to 800: the range check must not send a confident model
    to the fp64 path, and the fast lattice must resolve near-certain costs to the floor."""
    monkeypatch.setenv("B200CTC_CLUSTER", cluster)
    acts, labels, act_lens, label_lens = batch(stay_fast_utterances(V), seed=V)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), labels, act_lens, label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, 0)
    check_parity(c, g, acts, labels, act_lens, label_lens, "stay-fast V=%d cluster=%s" % (V, cluster))


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", ["0", "1"])
@pytest.mark.parametrize("V", [30, 300, 1500])
def test_lost_range_is_redone_by_the_safe_lattice(V, cluster, monkeypatch):
    """Misrecognised stretches of a confident model: the range check must flag the utterance and the fp64 safe
    lattice must redo it -- at V=30 over gradient rows the fast reducers already rewrote in place, at V=300 / 1500 in
    gathered mode -- in training and cost-only calls, host-planned and device-resident (bit-identical), and through
    the fused call site (temperature 1.3, label smoothing 0.1)."""
    monkeypatch.setenv("B200CTC_CLUSTER", cluster)
    utts = redo_utterances(V)
    if len(utts) == 1:
        utts.append(benign_twin(V, 120, 30, 77))
    n_redo = len(REDO[V])
    acts, labels, act_lens, label_lens = batch(utts, seed=V + 1)
    what = "redo V=%d cluster=%s" % (V, cluster)
    acts_d = torch.from_numpy(acts).cuda()
    c, loss, g = b200.ctc_loss_and_grad(acts_d, labels, act_lens, label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, n_redo)
    check_parity(c, g, acts, labels, act_lens, label_lens, what)
    c_only, _, g_none = b200.ctc_loss_and_grad(acts_d, labels, act_lens, label_lens, need_grad=False)
    torch.cuda.synchronize()
    assert g_none is None and ctc_mod.last_fallbacks() == (0, n_redo)
    check_parity(c_only, None, acts, labels, act_lens, label_lens, what + " cost-only")
    c_d, loss_d, g_d = b200.ctc_loss_and_grad(acts_d, *device_args(labels, act_lens, label_lens))
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks(with_invalid=True) == (0, n_redo, 0)
    assert torch.equal(c, c_d) and torch.equal(loss, loss_d) and torch.equal(g, g_d)
    # the call site: batch-major logits, labels without the blank offset
    ys = padded_labels(labels, label_lens, pad=1).astype(np.int64) - 1
    check_call_site(np.ascontiguousarray(acts.transpose(1, 0, 2)), ys, act_lens, label_lens, 1.0 / CALL_SITE_SCALE, 0.1,
                    what + " call site")
    assert ctc_mod.last_fallbacks() == (0, n_redo)


@pytest.mark.gpu
@pytest.mark.parametrize("cluster", ["0", "1"])
@pytest.mark.parametrize("V", [30, 300])
def test_a_redone_utterance_leaves_its_neighbours_untouched(V, cluster, monkeypatch):
    """The redo rebuilds and rewrites one utterance's gradient rows: the other utterances of the batch must get
    bit-for-bit what they get next to a benign utterance of the same lengths, and the batch must be reproducible."""
    monkeypatch.setenv("B200CTC_CLUSTER", cluster)
    T, L, seed = REDO[V][0]
    redo = redo_utterances(V)[0]
    twin = benign_twin(V, T, L, seed)
    others = [ordinary_utterance(V, T - 17 * i, 20 + 9 * i, 300 + i) for i in range(4)]
    runs = []
    for mid, expect in ((redo, (0, 1)), (twin, (0, 0)), (redo, (0, 1))):
        acts, labels, act_lens, label_lens = batch(others[:2] + [mid] + others[2:], seed=V + 2)
        c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), labels, act_lens, label_lens)
        torch.cuda.synchronize()
        assert ctc_mod.last_fallbacks() == expect
        runs.append((c.clone(), loss.clone(), g.clone()))
    check_parity(runs[0][0], runs[0][2], acts, labels, act_lens, label_lens, "neighbours V=%d cluster=%s" % (V, cluster))
    keep = torch.tensor([0, 1, 3, 4], device="cuda")
    assert torch.equal(runs[0][0][keep], runs[1][0][keep])
    assert torch.equal(runs[0][2][:, keep], runs[1][2][:, keep])
    assert all(torch.equal(a, b) for a, b in zip(runs[0], runs[2]))


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, CALL_SITE_SCALE])
@pytest.mark.parametrize("level", EDGE_LEVELS)
@pytest.mark.parametrize("V,cta_per_row", [(30, False), (301, False), (301, True), ("past_streaming", False)])
def test_extreme_row_threshold_edge(V, cta_per_row, level, scale, monkeypatch):
    """K1 flags a row when some ln y < -69: -68.5 is the fast lattice at the bottom of its range (parity, no
    fallback); -69.5 sends the utterance to the safe lattice; a -80 row in a padding frame or in an infeasible
    utterance sends nothing anywhere.  Every K1 kernel: warp (V=30), streaming (V=301), CTA per row (forced, and past
    the streaming kernel's shared-memory limit); logits as given and scaled by 1/1.3 inside K1."""
    if V == "past_streaming":
        V = streaming_softmax_max_V() + 1
    if cta_per_row:
        monkeypatch.setenv("B200CTC_SOFTMAX_CTA_PER_ROW", "1")
    acts, labels, act_lens, label_lens = edge_batch(V, level, scale)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), *device_args(labels, act_lens, label_lens),
                                        logit_scale=scale)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks(with_invalid=True) == ((0, 0, 0) if level > -69.0 else (1, 0, 0))
    z = acts * np.float32(scale)                              # what K1 computes, in fp32
    check_parity(c, g, z, labels, act_lens, label_lens, "edge V=%d level=%g scale=%.3g" % (V, level, scale))
    g = g.cpu().numpy()
    assert np.all(g[30:, 1] == 0) and np.all(g[:, 2] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("V", ["streaming_limit", "past_streaming", 16400])
def test_cta_per_row_softmax_past_the_streaming_limit(V):
    """Vocabularies on both sides of the streaming kernel's shared-memory limit, and far past it: parity, zero
    padding rows, and the label-smoothing term (which the CTA-per-row kernel takes from its block sum)."""
    V = {"streaming_limit": streaming_softmax_max_V(), "past_streaming": streaming_softmax_max_V() + 1}.get(V, V)
    utts = [ordinary_utterance(V, T, L, V + i) for i, (T, L) in enumerate(((24, 8), (19, 5), (22, 10)))]
    acts, labels, act_lens, label_lens = batch(utts, seed=V)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), labels, act_lens, label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, 0)
    check_parity(c, g, acts, labels, act_lens, label_lens, "wide V=%d" % V)
    g = g.cpu().numpy()
    for b in range(len(utts)):
        assert np.all(g[act_lens[b]:, b] == 0)
    ys = padded_labels(labels, label_lens, pad=1).astype(np.int64) - 1
    check_call_site(np.ascontiguousarray(acts.transpose(1, 0, 2)), ys, act_lens, label_lens, 1.3, 0.1, "wide V=%d call site" % V)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [301, 3386])
@pytest.mark.parametrize("layout", ["contiguous", "batch_major_view", "offset_by_one_float", "offset_by_three_floats"])
def test_cta_per_row_softmax_forced_row_alignment(V, layout, monkeypatch):
    """B200CTC_SOFTMAX_CTA_PER_ROW forces the CTA-per-row kernel where the streaming kernel would run: rows at every
    16-byte phase, source and destination at different phases, a base that is not 16-byte aligned; with and without
    label smoothing."""
    monkeypatch.setenv("B200CTC_SOFTMAX_CTA_PER_ROW", "1")
    utts = [ordinary_utterance(V, T, L, V + 10 * i) for i, (T, L) in enumerate(((37, 9), (30, 7), (33, 4), (25, 9), (37, 6)))]
    ref, labels, act_lens, label_lens = batch(utts, seed=V + 3)
    T, B = ref.shape[:2]
    if layout == "contiguous":
        acts = torch.from_numpy(ref).cuda()
    elif layout == "batch_major_view":
        acts = torch.from_numpy(np.ascontiguousarray(ref.transpose(1, 0, 2))).cuda().transpose(0, 1)
        assert not acts.is_contiguous()
    else:
        k = 1 if layout == "offset_by_one_float" else 3
        buf = torch.empty(ref.size + 8, device="cuda")
        acts = buf[k:k + ref.size].view(T, B, V)
        acts.copy_(torch.from_numpy(ref))
        assert acts.data_ptr() % 16 == 4 * k
    what = "forced CTA V=%d %s" % (V, layout)
    c, loss, g = b200.ctc_loss_and_grad(acts, labels, act_lens, label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, 0)
    check_parity(c, g, ref, labels, act_lens, label_lens, what)
    gn = g.cpu().numpy()
    for b in range(B):
        assert np.all(gn[act_lens[b]:, b] == 0)
    # label smoothing: loss_sum = sum_b (1 - ls) cost_b + ls / V * XE_b, grads = d loss_sum / d logits
    c_s, loss_s, g_s = b200.ctc_loss_and_grad(acts, *device_args(labels, act_lens, label_lens), label_smoothing=0.1)
    torch.cuda.synchronize()
    ys = padded_labels(labels, label_lens, pad=1).astype(np.int64) - 1
    loss_ref, g_ref = ctc_ref.ctc_loss_call_site(ref.transpose(1, 0, 2), ys, act_lens, label_lens, 1.0, 0.1)
    got = float(loss_s.cpu()[0])
    assert abs(got - B * loss_ref) <= COST_RTOL * abs(B * loss_ref), "%s: loss_sum %.9g vs %.9g" % (what, got, B * loss_ref)
    check_grads(g_s.cpu().numpy(), B * g_ref.transpose(1, 0, 2), what + " label smoothing")


def _large_batch(B, seed, T=40, V=30, Lmax=12):
    rng = np.random.RandomState(seed)
    label_lens = rng.randint(1, Lmax + 1, size=B).astype(np.int32)
    act_lens = rng.randint(T - 10, T + 1, size=B).astype(np.int32)
    labels = rng.randint(1, V, size=int(label_lens.sum())).astype(np.int32)
    acts = rng.randn(T, B, V).astype(np.float32)
    return acts, labels, act_lens, label_lens


@pytest.mark.gpu
@pytest.mark.parametrize("B", [704, 705, 1500])
def test_large_batch_planning(B):
    """The plan kernel plans up to 704 utterances in shared memory and larger batches in place, one warp per
    utterance with worst-case offsets and the rank sort in global memory: bit-identical to the host-planned call,
    within tolerance of the oracle, loss_sum = sum of the costs; invalid utterances past index 704 are rejected."""
    acts, labels, act_lens, label_lens = _large_batch(B, B)
    acts_d = torch.from_numpy(acts).cuda()
    c_h, l_h, g_h = b200.ctc_loss_and_grad(acts_d, labels, act_lens, label_lens)
    ys, al, ll = device_args(labels, act_lens, label_lens, width=12)
    c_d, l_d, g_d = b200.ctc_loss_and_grad(acts_d, ys, al, ll)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks(with_invalid=True) == (0, 0, 0)
    assert torch.equal(c_h, c_d) and torch.equal(l_h, l_d) and torch.equal(g_h, g_d)
    check_parity(c_d, g_d, acts, labels, act_lens, label_lens, "plan B=%d" % B)
    c_ref, _ = ctc_cpu(acts, labels, act_lens, label_lens, 0, precision="f64", need_grad=False)
    total = c_ref.astype(np.float64).sum()
    assert abs(float(l_d.cpu()[0]) - total) <= COST_RTOL * total
    if B < 1500:
        return
    bad = [704, 1000, 1498, 1499]
    ys2, al2, ll2 = ys.clone(), al.clone(), ll.clone()
    ys2[bad[0], 0] = 30                  # label == V
    ys2[bad[1], int(ll[bad[1]]) - 1] = 0  # label == blank
    al2[bad[2]] = acts.shape[0] + 1      # act_len > T
    ll2[bad[3]] = ys.size(1) + 1         # label_len > padded width
    c2, _, g2 = b200.ctc_loss_and_grad(acts_d, ys2, al2, ll2)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks(with_invalid=True)[2] == len(bad)
    keep = torch.tensor(sorted(set(range(B)) - set(bad)), device="cuda")
    bad_t = torch.tensor(bad, device="cuda")
    assert bool(torch.isnan(c2[bad_t]).all()) and bool((g2[:, bad_t] == 0).all())
    assert torch.equal(c2[keep], c_d[keep]) and torch.equal(g2[:, keep], g_d[:, keep])


@pytest.mark.gpu
def test_back_to_back_large_batches_plan_in_place_after_the_previous_call():
    """Past 704 utterances the plan kernel writes the shared tables in place after griddepcontrol.wait: two calls with
    different lengths issued back to back must each give the result of an isolated call."""
    batches = [_large_batch(1500, s, T=40 + 8 * i) for i, s in enumerate((11, 12))]
    dev = [(torch.from_numpy(a).cuda(), device_args(lab, al, ll, width=12)) for a, lab, al, ll in batches]
    iso = []
    for a, args in dev:
        c, _, g = b200.ctc_loss_and_grad(a, *args)
        torch.cuda.synchronize()
        iso.append((c.clone(), g.clone()))
    for rep in range(3):
        outs = [b200.ctc_loss_and_grad(a, *args) for a, args in dev]      # no synchronisation in between
        torch.cuda.synchronize()
        for (c, _, g), (c0, g0) in zip(outs, iso):
            assert torch.equal(c, c0) and torch.equal(g, g0), rep


@pytest.mark.gpu
@pytest.mark.parametrize("V", [31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257])
def test_softmax_lane_geometry_switches(V):
    """K1's lane geometry changes at V = 32/33, 64/65, 128/129 (and the lattice goes to gathered mode at 129), the
    streaming kernel takes over at 257: parity on both sides, with and without the call-site options."""
    utts = [ordinary_utterance(V, T, L, 7 * V + i) for i, (T, L) in enumerate(((50, 15), (44, 9), (50, 1), (31, 12)))]
    acts, labels, act_lens, label_lens = batch(utts, seed=V)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), labels, act_lens, label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, 0)
    check_parity(c, g, acts, labels, act_lens, label_lens, "geometry V=%d" % V)
    ys = padded_labels(labels, label_lens, pad=1).astype(np.int64) - 1
    check_call_site(np.ascontiguousarray(acts.transpose(1, 0, 2)), ys, act_lens, label_lens, 1.3, 0.1, "geometry V=%d call site" % V)
    assert ctc_mod.last_fallbacks(with_invalid=True) == (0, 0, 0)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the declared class of every GPU case
# ---------------------------------------------------------------------------------------------------------------
def _assert_live_rows_unflagged(acts, what, scale=1.0):
    lp = peaked_ref.min_log_prob(acts, scale)
    assert lp >= -68.0, "%s: a live row has ln y = %.2f (K1 would flag it)" % (what, lp)


@pytest.mark.parametrize("V", [30, 300])
def test_stay_fast_cases_are_declared_correctly(V):
    for (T, L, m, e), (acts, lab) in zip(STAY_FAST, stay_fast_utterances(V)):
        what = "V=%d T=%d m=%g err=%g" % (V, T, m, e)
        assert L <= peaked_ref.WINDOW_MAX_L
        _assert_live_rows_unflagged(acts, what)
        bits = peaked_ref.predicted_range_bits(acts, lab)
        assert peaked_ref.range_class(bits) == "must-stay-fast", "%s: %.1f bits" % (what, bits)


@pytest.mark.parametrize("V", [30, 300, 1500])
def test_redo_cases_are_declared_correctly(V):
    """Must-redo on the logits as given and on the call site's scaled ones; the benign twin of the neighbours test
    and the filler of a single-utterance batch stay fast."""
    for (T, L, seed), (acts, lab) in zip(REDO[V], redo_utterances(V)):
        assert L <= peaked_ref.WINDOW_MAX_L
        for scale in (1.0, CALL_SITE_SCALE):
            what = "V=%d T=%d seed=%d scale=%.3g" % (V, T, seed, scale)
            _assert_live_rows_unflagged(acts, what, scale)
            bits = peaked_ref.predicted_range_bits(acts, lab, logit_scale=scale)
            assert peaked_ref.range_class(bits) == "must-redo", "%s: %.1f bits" % (what, bits)
    twins = [benign_twin(V, *REDO[V][0])] + ([benign_twin(V, 120, 30, 77)] if len(REDO[V]) == 1 else [])
    for acts, lab in twins:
        for scale in (1.0, CALL_SITE_SCALE):
            _assert_live_rows_unflagged(acts, "benign V=%d" % V, scale)
            assert peaked_ref.range_class(peaked_ref.predicted_range_bits(acts, lab, logit_scale=scale)) == "must-stay-fast"


@pytest.mark.parametrize("V", [30, 301, "past_streaming"])
@pytest.mark.parametrize("scale", [1.0, CALL_SITE_SCALE])
@pytest.mark.parametrize("level", EDGE_LEVELS)
def test_threshold_edge_cases_are_declared_correctly(V, scale, level):
    """Utterance 0's edge rows sit at `level` to 1e-3; below -69 it is K1's to flag, above it must stay fast.
    Utterance 1's -80 row is a padding frame, utterance 2 is infeasible."""
    V = streaming_softmax_max_V() + 1 if V == "past_streaming" else V
    acts, labels, act_lens, label_lens = edge_batch(V, level, scale)
    z0 = acts[:40, 0]
    lp = ctc_ref.log_softmax((z0 * np.float32(scale)).astype(np.float64), axis=1)
    assert abs(lp.min() - level) < 1e-3
    assert np.sum(lp.min(axis=1) < -20) == 3
    if level > -69.0:
        bits = peaked_ref.predicted_range_bits(z0, labels[:10], logit_scale=scale)
        assert peaked_ref.range_class(bits) == "must-stay-fast", "%.1f bits" % bits
    lp1 = ctc_ref.log_softmax((acts[:, 1] * np.float32(scale)).astype(np.float64), axis=1).min(axis=1)
    assert lp1[35] < -79.9 and lp1[:act_lens[1]].min() > -69.0
    assert label_lens[2] > act_lens[2]
    assert ctc_ref.log_softmax((acts[5, 2] * np.float32(scale)).astype(np.float64)).min() < -79.9

