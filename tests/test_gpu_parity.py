"""GPU parity tests proper: the CUDA path, called through the C ABI (the PyTorch extension for the loss,
ctypes for the decoders), against the CPU oracle on identical inputs.  Tolerances are the ones BASELINE.json's north_star states:
per-utterance loss within 1e-5 relative, gradients within 1e-4 absolute (fp32), decoded label
sequences bit-exact."""
import os

import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from oracle import ctc_ref
from oracle.ctc_cpu import ctc_cpu
from pytorch_end2end_speech_recognition_b200 import ctc as ctc_mod
from pytorch_end2end_speech_recognition_b200 import workloads

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-5
GRAD_ATOL = 1e-4


def run_gpu(acts_np, labels, act_lens, label_lens, blank=0, need_grad=True):
    acts = torch.from_numpy(np.ascontiguousarray(acts_np, dtype=np.float32)).cuda()
    costs, loss, grads = b200.ctc_loss_and_grad(acts, labels, act_lens, label_lens, blank=blank, need_grad=need_grad)
    torch.cuda.synchronize()
    return costs.cpu().numpy(), float(loss.cpu()[0]), (grads.cpu().numpy() if grads is not None else None)


def check(acts_np, labels, act_lens, label_lens, blank=0, oracle="numpy"):
    c, loss, g = run_gpu(acts_np, labels, act_lens, label_lens, blank)
    if oracle == "numpy":
        c_ref, g_ref = ctc_ref.ctc_cost_and_grad(acts_np, labels, act_lens, label_lens, blank)
    else:
        c_ref, g_ref = ctc_cpu(acts_np, labels, act_lens, label_lens, blank, precision="f64")
        c_ref = c_ref.astype(np.float64)
    fin = np.isfinite(c_ref)
    assert np.array_equal(np.isfinite(c), fin)
    assert np.all(np.isposinf(c[~fin]))
    rel = np.abs(c[fin] - c_ref[fin]) / np.maximum(np.abs(c_ref[fin]), 1e-3)
    assert rel.size == 0 or rel.max() < LOSS_RTOL, "cost rel err %g" % rel.max()
    err = np.max(np.abs(g - g_ref)) if g.size else 0.0
    assert err < GRAD_ATOL, "grad abs err %g" % err
    if fin.all():
        assert abs(loss - c_ref.sum()) <= LOSS_RTOL * max(abs(c_ref.sum()), 1e-3)
    return c, g


def test_golden_vectors(golden_dir):
    z = np.load(os.path.join(golden_dir, "ctc_golden.npz"))
    for i in range(int(z["n_cases"])):
        c, _, g = run_gpu(z["acts_%d" % i], z["labels_%d" % i], z["act_lens_%d" % i], z["label_lens_%d" % i])
        assert np.allclose(c, z["costs_%d" % i], rtol=LOSS_RTOL), i
        assert np.max(np.abs(g - z["grads_%d" % i])) < GRAD_ATOL, i


def test_reference_chainer_golden_vectors(golden_dir):
    """Costs/gradients produced by the reference's own in-tree CTC
    (models/chainer/ctc/ctc_loss_from_chainer.py, run by tests/golden/make_golden.py).  That code is a
    float32 log-space recursion with -1e10 padding, so the fixture itself carries rounding error against
    exact arithmetic.  The test MEASURES that error (fixture against the fp64 oracle) and asserts
      * our gradient is within GRAD_ATOL of the exact (fp64) gradient, always, and
      * our gradient is within GRAD_ATOL + the fixture's own measured error of the fixture
    instead of loosening the tolerance by a narrated amount."""
    z = np.load(os.path.join(golden_dir, "ctc_reference_golden.npz"))
    worst_fixture_err = 0.0
    for i in range(int(z["n_cases"])):
        acts = z["acts_%d" % i]
        lab, al, ll = z["labels_%d" % i], z["act_lens_%d" % i], z["label_lens_%d" % i]
        c, _, g = run_gpu(acts, lab, al, ll)
        assert np.allclose(c, z["costs_%d" % i], rtol=LOSS_RTOL), i
        c64, g64 = ctc_ref.ctc_cost_and_grad(acts, lab, al, ll)
        fixture_err = float(np.max(np.abs(z["grads_%d" % i] - g64)))
        worst_fixture_err = max(worst_fixture_err, fixture_err)
        assert np.max(np.abs(g - g64)) < GRAD_ATOL, i                       # against exact arithmetic
        assert np.max(np.abs(g - z["grads_%d" % i])) < GRAD_ATOL + fixture_err, i
        if acts.shape[0] <= 64:
            assert fixture_err < GRAD_ATOL, (i, fixture_err)               # short cases: the fixture itself is within tolerance
    assert worst_fixture_err < 5e-4       # the reference's fp32 log-space rounding stays below this on the fixture (T <= 96)


def test_kats():
    acts = np.array([[[0.3, -1.2, 2.0]]], np.float32)
    check(acts, [], [1], [0])                       # T=1, L=0
    check(acts, [2], [1], [1])                      # T=1, L=1
    rng = np.random.RandomState(0)
    check(rng.randn(2, 1, 4), [3], [2], [1])        # three paths
    for T in (1, 2, 3, 5, 8):                       # uniform logits: closed-form path count
        c, _ = check(np.zeros((T, 1, 2)), [1], [T], [1])
        assert np.isclose(c[0], -np.log(T * (T + 1) / 2 / 2.0 ** T), rtol=LOSS_RTOL)
    a3 = rng.randn(3, 1, 3)
    c, g = check(a3[:2], [1, 1], [2], [2])          # "aa", T=2: infeasible -> +inf, zero gradient
    assert np.isposinf(c[0]) and np.all(g == 0)
    check(a3, [1, 1], [3], [2])                     # "aa", T=3: exactly one path
    check(rng.randn(4, 1, 5), [1, 2, 3, 4], [4], [4])  # L == T


def test_padding_rows_are_zero_and_ignored():
    rng = np.random.RandomState(3)
    acts = rng.randn(10, 2, 6).astype(np.float32)
    labels = [1, 2, 3, 4, 5]
    c1, g1 = check(acts, labels, [10, 6], [3, 2])
    acts2 = acts.copy(); acts2[6:, 1] = rng.randn(4, 6) * 10
    c2, g2 = check(acts2, labels, [10, 6], [3, 2])
    assert np.all(g1[6:, 1] == 0) and np.all(g2[6:, 1] == 0)
    assert np.array_equal(c1, c2) and np.array_equal(g1[:, 1], g2[:, 1])


def test_extreme_logits_stability():
    rng = np.random.RandomState(4)
    acts = (rng.randn(30, 3, 8) * 50).astype(np.float32)
    c, g = check(acts, [1, 2, 2, 3, 7, 7, 1], [30, 20, 25], [3, 2, 2])
    assert np.all(np.isfinite(c)) and np.all(np.isfinite(g))
    assert sum(ctc_mod.last_fallbacks()) > 0        # +-50 logits: handled by the fp64 safe lattice
    acts = rng.randn(40, 2, 5).astype(np.float32)
    acts[::3, :, 1] += 50; acts[1::3, :, 2] -= 50
    check(acts, [1, 2, 1, 2, 3], [40, 33], [3, 2])


def test_empty_and_degenerate_inputs():
    rng = np.random.RandomState(5)
    acts = rng.randn(6, 3, 4).astype(np.float32)
    c, g = check(acts, [1, 2], [6, 0, 3], [2, 0, 0])     # T_b = 0 with L_b = 0 -> cost 0, zero grads
    assert c[1] == 0 and np.all(g[:, 1] == 0)
    c, g = check(acts, [1, 2, 3], [6, 0, 3], [2, 1, 0])  # T_b = 0 with L_b > 0 -> infeasible
    assert np.isposinf(c[1])
    check(acts[:, :1], [], [6], [0])                     # B = 1, empty target
    check(rng.randn(5, 2, 1).astype(np.float32), [], [5, 3], [0, 0])  # V = 1: only blank exists


def test_nonzero_blank_and_permutation_invariance():
    rng = np.random.RandomState(6)
    acts = rng.randn(12, 3, 5).astype(np.float32)
    labs = [[1, 2], [3], [0, 0, 1]]
    al, ll = [12, 9, 11], [2, 1, 3]
    c, g = check(acts, sum(labs, []), al, ll, blank=4)
    perm = [2, 0, 1]
    c2, g2 = check(acts[:, perm], sum([labs[i] for i in perm], []), [al[i] for i in perm], [ll[i] for i in perm], blank=4)
    assert np.allclose(c[perm], c2, rtol=1e-6) and np.allclose(g[:, perm], g2, atol=1e-6)


def test_random_small_cases_vs_numpy_oracle():
    rng = np.random.RandomState(7)
    for it in range(25):
        B, T, V = rng.randint(1, 7), rng.randint(1, 70), rng.randint(2, 40)
        act_lens = rng.randint(1, T + 1, size=B); act_lens[0] = T
        labels, label_lens = [], []
        for b in range(B):
            L = rng.randint(0, act_lens[b] + 1)
            lab = rng.randint(1, V, size=L)
            for j in range(1, L):
                if rng.uniform() < 0.15:
                    lab[j] = lab[j - 1]
            if it % 5 != 0:                      # every fifth case keeps infeasible utterances
                while L + ctc_ref.count_repeats(lab[:L]) > act_lens[b]:
                    L -= 1
            labels.append(lab[:L]); label_lens.append(L)
        flat = np.concatenate(labels).astype(np.int32)
        acts = (rng.randn(T, B, V) * rng.choice([0.3, 1.0, 4.0])).astype(np.float32)
        check(acts, flat, act_lens, label_lens)


def test_strided_batch_major_input_needs_no_copy():
    # the reference passes logits.transpose(0, 1) of a [B,T,V] tensor (ctc.py:319)
    wl = workloads.make_lengths_and_labels(None, B=5, T=50, V=11, Lmax=12, kind="var", seed=9)
    bt = torch.randn(wl.B, wl.T, wl.V, device="cuda")
    view = bt.transpose(0, 1)
    assert not view.is_contiguous()
    c1, l1, g1 = b200.ctc_loss_and_grad(view, wl.labels, wl.act_lens, wl.label_lens)
    c2, l2, g2 = b200.ctc_loss_and_grad(view.contiguous(), wl.labels, wl.act_lens, wl.label_lens)
    assert torch.equal(c1, c2) and torch.equal(g1, g2)
    c_ref, g_ref = ctc_ref.ctc_cost_and_grad(view.cpu().numpy(), wl.labels, wl.act_lens, wl.label_lens)
    assert np.allclose(c1.cpu().numpy(), c_ref, rtol=LOSS_RTOL)
    assert np.max(np.abs(g1.cpu().numpy() - g_ref)) < GRAD_ATOL


def test_cost_only_mode_matches():
    wl = workloads.make_lengths_and_labels(None, B=4, T=60, V=20, Lmax=15, kind="var", seed=10)
    acts = workloads.make_acts(wl).numpy()
    c1, _, _ = run_gpu(acts, wl.labels, wl.act_lens, wl.label_lens)
    c2, _, g2 = run_gpu(acts, wl.labels, wl.act_lens, wl.label_lens, need_grad=False)
    assert g2 is None and np.allclose(c1, c2, rtol=1e-6)


@pytest.mark.parametrize("key", ["C1", "C2", "C3", "C4", "C5"])
def test_full_size_configs(key):
    """BASELINE.json shapes at full size: parity against the fp64 C++ restatement (OpenMP, seconds)
    plus size-independent properties of the domain."""
    wl = workloads.make_lengths_and_labels(key)
    acts_t = workloads.make_acts(wl)
    acts = acts_t.numpy()
    c, g = check(acts, wl.labels, wl.act_lens, wl.label_lens, oracle="cpp")
    # the block-exponent fast lattice must be what ran: no utterance may have needed the fp64 safe path
    assert ctc_mod.last_fallbacks() == (0, 0)
    T_b = wl.act_lens
    t_idx = np.arange(wl.T)[:, None]
    valid = t_idx < T_b[None, :]
    rowsum = g.sum(axis=2)
    assert np.max(np.abs(rowsum[valid])) < 5e-5          # softmax minus a distribution
    assert np.all(g[~valid] == 0)                         # rows t >= T_b exactly zero
    assert np.all(c > 0)
    # log_softmax(acts) as input gives the same result (softmax is idempotent on log-probs)
    if key in ("C1", "C3"):
        lsm = torch.log_softmax(acts_t, dim=2).numpy()
        c2, _, g2 = run_gpu(lsm, wl.labels, wl.act_lens, wl.label_lens)
        assert np.allclose(c, c2, rtol=LOSS_RTOL) and np.max(np.abs(g - g2)) < GRAD_ATOL


def test_reentrancy_two_shapes_back_to_back():
    # hierarchical CTC issues two calls per step with different T and V (hierarchical_ctc.py:323-330)
    w1 = workloads.make_lengths_and_labels(None, B=6, T=80, V=30, Lmax=20, kind="var", seed=21)
    w2 = workloads.make_lengths_and_labels(None, B=6, T=40, V=300, Lmax=8, kind="var", seed=22)
    a1, a2 = workloads.make_acts(w1).cuda(), workloads.make_acts(w2).cuda()
    r1 = b200.ctc_loss_and_grad(a1, w1.labels, w1.act_lens, w1.label_lens)
    r2 = b200.ctc_loss_and_grad(a2, w2.labels, w2.act_lens, w2.label_lens)
    r1b = b200.ctc_loss_and_grad(a1, w1.labels, w1.act_lens, w1.label_lens)
    torch.cuda.synchronize()
    assert torch.equal(r1[0], r1b[0]) and torch.equal(r1[2], r1b[2])       # deterministic, no shared state
    for (w, a, r) in ((w1, a1, r1), (w2, a2, r2)):
        c_ref, g_ref = ctc_ref.ctc_cost_and_grad(a.cpu().numpy(), w.labels, w.act_lens, w.label_lens)
        assert np.allclose(r[0].cpu().numpy(), c_ref, rtol=LOSS_RTOL)
        assert np.max(np.abs(r[2].cpu().numpy() - g_ref)) < GRAD_ATOL


def _seq(rng, L, V):
    lab = rng.randint(1, V, size=L)
    for j in range(1, L):
        if rng.uniform() < 0.1:
            lab[j] = lab[j - 1]
    return lab.astype(np.int32)


def test_every_short_length_and_chunk_tail():
    """T = 1..26 crosses every chunk-tail / phase-split case of the lattice kernel (chunks of four
    frames, the two sweeps meet in the middle, helper warps fetch two chunks ahead)."""
    rng = np.random.RandomState(11)
    for T in range(1, 27):
        for L in sorted({0, 1, T // 3, T // 2}):
            lab = _seq(rng, L, 7)
            while len(lab) + ctc_ref.count_repeats(lab) > T:
                lab = lab[:-1]
            acts = rng.randn(T, 2, 7).astype(np.float32)
            check(acts, np.concatenate([lab, lab]), [T, T], [len(lab), len(lab)])


@pytest.mark.parametrize("L", [127, 128, 239, 240, 351, 352, 463, 464, 499])
def test_lattice_window_boundaries(L):
    """Label lengths at which the number of 256-state lattice windows per sweep changes (1..4 warps; windows
    overlap by 32 states, so a sweep of n windows holds 224 n + 32 states) and, from 464, the first lengths
    that no longer fit four windows and take the safe lattice."""
    rng = np.random.RandomState(L)
    V = 30
    lab = _seq(rng, L, V)
    T = L + ctc_ref.count_repeats(lab) + 40
    acts = rng.randn(T, 2, V).astype(np.float32)
    lab2 = _seq(rng, L // 2, V)
    check(acts, np.concatenate([lab, lab2]), [T, T - 17], [L, len(lab2)], oracle="cpp")
    assert ctc_mod.last_fallbacks() == (0, 0)


@pytest.mark.parametrize("V,L", [(30, 200), (62, 75), (100, 180), (128, 120)])
def test_symbol_group_reduce_paths(V, L):
    """The reducers hold one or two symbol groups per lane (up to 32 / 64 distinct symbols) and loop beyond
    that; V = 100 and 128 exercise the loop without the large-vocabulary gathered mode (V >= 129)."""
    rng = np.random.RandomState(V * 1000 + L)
    lab = rng.randint(1, V, size=L)
    T = L + ctc_ref.count_repeats(lab) + 30
    acts = rng.randn(T, 2, V).astype(np.float32)
    lab2 = rng.randint(1, V, size=L // 3)
    check(acts, np.concatenate([lab, lab2]), [T, T - 9], [L, len(lab2)], oracle="cpp")
    assert ctc_mod.last_fallbacks() == (0, 0)


def test_skewed_symbol_distribution():
    """Real transcripts are skewed (space, 'e', 't'): one symbol carries 60 % of the labels, so its group in
    the symbol-sorted posterior row is ~40 times the size of the others."""
    rng = np.random.RandomState(77)
    V, L = 30, 300
    lab = np.where(rng.rand(L) < 0.6, 5, rng.randint(1, V, size=L)).astype(np.int64)
    T = L + ctc_ref.count_repeats(lab) + 60
    acts = rng.randn(T, 2, V).astype(np.float32)
    lab2 = np.full(40, 7, dtype=np.int64)                     # a single symbol repeated: every label needs a blank
    check(acts, np.concatenate([lab, lab2]), [T, T - 5], [L, len(lab2)], oracle="cpp")
    assert ctc_mod.last_fallbacks() == (0, 0)


def test_label_sequence_beyond_the_fast_lattice_takes_the_safe_path():
    rng = np.random.RandomState(13)
    L, V = 520, 12
    lab = _seq(rng, L, V)
    T = L + ctc_ref.count_repeats(lab) + 25
    acts = rng.randn(T, 1, V).astype(np.float32)
    check(acts, lab, [T], [L], oracle="cpp")


def test_results_are_bit_reproducible():
    wl = workloads.make_lengths_and_labels(None, B=8, T=200, V=30, Lmax=80, kind="var", seed=15)
    acts = workloads.make_acts(wl).numpy()
    c1, l1, g1 = run_gpu(acts, wl.labels, wl.act_lens, wl.label_lens)
    c2, l2, g2 = run_gpu(acts, wl.labels, wl.act_lens, wl.label_lens)
    assert np.array_equal(c1, c2) and l1 == l2 and np.array_equal(g1, g2)
