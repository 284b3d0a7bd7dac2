"""GPU tests added in round 2: the device-resident call (plan kernel, CUDA-graph capture), the plan cache of
the host call, cost-only calls at full size, label sequences beyond the shared-memory budget of the
gathered mode, input clamping in the decoder, sharded evaluation of one batch."""
import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from oracle import ctc_ref
from oracle.ctc_cpu import ctc_cpu
from pytorch_end2end_speech_recognition_b200 import ctc as ctc_mod
from pytorch_end2end_speech_recognition_b200 import shard, workloads

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-5
GRAD_ATOL = 1e-4


def padded(wl, width=None):
    """[B, Lmax] int32 padded labels (pad value -7: must never be read) + CUDA length tensors."""
    width = int(wl.label_lens.max(initial=0)) if width is None else width
    ys = np.full((wl.B, max(width, 1)), -7, np.int32)
    off = 0
    for b, L in enumerate(wl.label_lens):
        ys[b, :L] = wl.labels[off:off + L]
        off += L
    return (torch.from_numpy(ys).cuda(), torch.from_numpy(wl.act_lens.astype(np.int32)).cuda(),
            torch.from_numpy(wl.label_lens.astype(np.int32)).cuda())


def assert_parity(c, g, acts, wl):
    c_ref, g_ref = ctc_cpu(acts, wl.labels, wl.act_lens, wl.label_lens, 0, precision="f64")
    c = c.cpu().numpy()
    assert np.max(np.abs(c - c_ref) / np.maximum(np.abs(c_ref), 1e-3)) < LOSS_RTOL
    if g is not None:
        assert np.max(np.abs(g.cpu().numpy() - g_ref)) < GRAD_ATOL


@pytest.mark.parametrize("key", [None, "C1", "C3", "C5"])
def test_device_resident_call_matches_host_call_and_oracle(key):
    """Labels and lengths on the GPU (plan kernel) give bit-identical results to the host-planned call."""
    wl = (workloads.make_lengths_and_labels(None, B=9, T=120, V=30, Lmax=40, kind="var", seed=31) if key is None
          else workloads.make_lengths_and_labels(key))
    acts_t = workloads.make_acts(wl)
    acts = acts_t.cuda()
    ys, al, ll = padded(wl, width=int(wl.label_lens.max()) + 3)
    c_h, l_h, g_h = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    c_d, l_d, g_d = b200.ctc_loss_and_grad(acts, ys, al, ll)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks(with_invalid=True) == (0, 0, 0)
    assert torch.equal(c_h, c_d) and torch.equal(g_h, g_d) and torch.equal(l_h, l_d)
    assert_parity(c_d, g_d, acts_t.numpy(), wl)


def test_device_resident_call_rejects_bad_utterances_on_the_device():
    wl = workloads.make_lengths_and_labels(None, B=5, T=40, V=12, Lmax=10, kind="var", seed=32)
    acts = workloads.make_acts(wl).cuda()
    ys, al, ll = padded(wl)
    good = b200.ctc_loss_and_grad(acts, ys, al, ll)
    ys2, al2, ll2 = ys.clone(), al.clone(), ll.clone()
    ys2[1, 0] = 12            # label == V
    ys2[2, 1] = 0             # label == blank
    al2[3] = 41               # act_len > T
    ll2[4] = ys.size(1) + 1   # label_len > padded width
    c, loss, g = b200.ctc_loss_and_grad(acts, ys2, al2, ll2)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks(with_invalid=True)[2] == 4
    c = c.cpu().numpy()
    assert np.isnan(c[1:]).all() and c[0] == good[0][0].item()
    g = g.cpu().numpy()
    assert np.all(g[:, 1:] == 0) and np.array_equal(g[:, 0], good[2][:, 0].cpu().numpy())


def test_device_resident_call_in_a_cuda_graph():
    """The device-resident call is kernel launches only: captured once, replayed with new inputs."""
    wl = workloads.make_lengths_and_labels(None, B=16, T=200, V=30, Lmax=60, kind="var", seed=33)
    wl2 = workloads.make_lengths_and_labels(None, B=16, T=200, V=30, Lmax=60, kind="var", seed=34)
    width = 60
    acts = workloads.make_acts(wl).cuda()
    ys, al, ll = padded(wl, width)
    grads = torch.empty_like(acts)
    costs = torch.empty(wl.B, device="cuda")
    loss = torch.empty(1, device="cuda")
    b200.ctc_loss_and_grad(acts, ys, al, ll, grads=grads, costs=costs, loss_sum=loss)    # warm-up (allocations)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        b200.ctc_loss_and_grad(acts, ys, al, ll, grads=grads, costs=costs, loss_sum=loss)
        torch.cuda.synchronize()
        with torch.cuda.graph(graph, stream=s):
            b200.ctc_loss_and_grad(acts, ys, al, ll, grads=grads, costs=costs, loss_sum=loss)
    torch.cuda.current_stream().wait_stream(s)
    for w in (wl, wl2, wl):
        a_new = workloads.make_acts(w, copy_index=3)
        y_new, al_new, ll_new = padded(w, width)
        acts.copy_(a_new.cuda()); ys.copy_(y_new); al.copy_(al_new); ll.copy_(ll_new)
        grads.fill_(7.0)
        graph.replay()
        torch.cuda.synchronize()
        assert_parity(costs, grads, a_new.numpy(), w)
        c_ref, _ = ctc_cpu(a_new.numpy(), w.labels, w.act_lens, w.label_lens, 0, precision="f64")
        assert abs(float(loss.cpu()[0]) - c_ref.sum()) < LOSS_RTOL * c_ref.sum()


def test_plan_cache_reuses_the_previous_plan():
    wl = workloads.make_lengths_and_labels(None, B=12, T=150, V=30, Lmax=50, kind="var", seed=35)
    acts = workloads.make_acts(wl).cuda()
    first = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    h0, m0 = ctc_mod.plan_cache_stats()
    again = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    h1, m1 = ctc_mod.plan_cache_stats()
    assert (h1, m1) == (h0 + 1, m0)
    labels2 = wl.labels.copy()
    labels2[5] = labels2[5] % (wl.V - 1) + 1                          # one label changed: must re-plan
    changed = b200.ctc_loss_and_grad(acts, labels2, wl.act_lens, wl.label_lens)
    h2, m2 = ctc_mod.plan_cache_stats()
    assert (h2, m2) == (h1, m1 + 1)
    torch.cuda.synchronize()
    assert torch.equal(first[0], again[0]) and torch.equal(first[2], again[2])
    c_ref, g_ref = ctc_ref.ctc_cost_and_grad(acts.cpu().numpy(), labels2, wl.act_lens, wl.label_lens)
    assert np.allclose(changed[0].cpu().numpy(), c_ref, rtol=LOSS_RTOL)
    assert np.max(np.abs(changed[2].cpu().numpy() - g_ref)) < GRAD_ATOL


@pytest.mark.parametrize("key", ["C3", "C1"])
def test_cost_only_call_at_full_size(key):
    """Validation loss (no gradient buffer) on the headline shape: same lattice, same shared-memory footprint
    as the training call (the softmax rows go to the workspace), no utterance on the safe path."""
    wl = workloads.make_lengths_and_labels(key)
    acts_t = workloads.make_acts(wl)
    c, loss, g = b200.ctc_loss_and_grad(acts_t.cuda(), wl.labels, wl.act_lens, wl.label_lens, need_grad=False)
    torch.cuda.synchronize()
    assert g is None and ctc_mod.last_fallbacks() == (0, 0)
    c_ref, _ = ctc_cpu(acts_t.numpy(), wl.labels, wl.act_lens, wl.label_lens, 0, precision="f64")
    assert np.max(np.abs(c.cpu().numpy() - c_ref) / c_ref) < LOSS_RTOL
    c2 = b200.ctc_loss_and_grad(acts_t.cuda(), wl.labels, wl.act_lens, wl.label_lens)[0]
    assert torch.equal(c, c2)


@pytest.mark.parametrize("V,L", [(300, 300), (1500, 260), (129, 400)])
def test_large_vocabulary_long_labels_beyond_the_shared_memory_budget(V, L):
    """Gathered mode (V >= 129): the emission-row ring grows with the label sequence, so the longest ones do
    not fit 227 KB and are evaluated by the safe lattice in the same launch -- the call must not fail."""
    rng = np.random.RandomState(V + L)
    labs = [rng.randint(1, V, size=n) for n in (L, L // 2, 30)]
    T = L + 40
    acts = rng.randn(T, 3, V).astype(np.float32)
    wl = workloads.Workload("x", T, 3, V, np.concatenate(labs).astype(np.int32), np.array([len(x) for x in labs], np.int32),
                            np.array([T, T - 3, T - 11], np.int32), 0)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), wl.labels, wl.act_lens, wl.label_lens)
    torch.cuda.synchronize()
    assert_parity(c, g, acts, wl)
    c2, _, g2 = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), wl.labels, wl.act_lens, wl.label_lens, need_grad=False)
    assert g2 is None and np.allclose(c2.cpu().numpy(), c.cpu().numpy(), rtol=1e-6)


def test_more_than_65535_frames():
    """The softmax-rows grid carries the frame index on (y, z): T is not limited to 65535."""
    rng = np.random.RandomState(41)
    T, V = 66000, 5
    acts = rng.randn(T, 1, V).astype(np.float32)
    wl = workloads.Workload("x", T, 1, V, np.array([1, 2, 2, 3], np.int32), np.array([4], np.int32), np.array([T], np.int32), 0)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), wl.labels, wl.act_lens, wl.label_lens)
    torch.cuda.synchronize()
    assert_parity(c, g, acts, wl)


def test_decoder_clamps_lengths_outside_the_tensor():
    rng = np.random.RandomState(42)
    logits = rng.randn(3, 20, 6).astype(np.float32)
    tokens, lens = b200.greedy_decode(torch.from_numpy(logits).cuda(), np.array([25, -3, 20]))
    ref = ctc_ref.greedy_decode(logits, np.array([20, 0, 20]))
    tokens, lens = tokens.cpu().numpy(), lens.cpu().numpy()
    for b in range(3):
        assert np.array_equal(tokens[b, :lens[b]], ref[b])
        assert np.all(tokens[b, lens[b]:] == -1)


def test_handle_rejects_a_call_on_another_device_or_threads_share_it():
    """Two host threads issuing calls on the same device share one handle (serialised by its mutex)."""
    import threading
    wl = workloads.make_lengths_and_labels(None, B=6, T=90, V=30, Lmax=25, kind="var", seed=43)
    acts = workloads.make_acts(wl).cuda()
    ref = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    torch.cuda.synchronize()
    out, err = [None] * 4, []

    def work(i):
        try:
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                for _ in range(20):
                    r = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
                s.synchronize()
            out[i] = r
        except Exception as exc:          # pragma: no cover
            err.append(exc)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not err
    for r in out:
        assert torch.equal(r[0], ref[0]) and torch.equal(r[2], ref[2])


def test_sharded_evaluation_of_one_batch_matches_the_whole_batch():
    """utils/parallel.py replacement, emulated on one device: the C5-shaped batch is split into two
    length-balanced shards (what ranks 0 and 1 of a 2-GPU job evaluate); shard losses add up to the loss of the
    whole batch and every utterance's cost and gradient is the one the unsharded call produces."""
    wl = workloads.make_lengths_and_labels(None, B=64, T=400, V=30, Lmax=100, kind="sweep", seed=44)
    acts = workloads.make_acts(wl).cuda()
    c_all, loss_all, g_all = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    total = 0.0
    seen = []
    for rank in range(2):
        loss, index, costs, grads = shard.sharded_ctc_loss(acts, wl.labels, wl.act_lens, wl.label_lens, rank=rank, world_size=2)
        total += float(loss.cpu()[0])
        seen.append(index)
        idx = torch.as_tensor(index, device="cuda")
        assert torch.equal(costs, c_all[idx])
        T_loc = int(wl.act_lens[index].max())
        assert tuple(grads.shape) == (T_loc, len(index), wl.V) and torch.equal(grads, g_all[:T_loc, idx])
    assert sorted(np.concatenate(seen).tolist()) == list(range(wl.B))
    assert abs(total - float(loss_all.cpu()[0])) < 1e-5 * float(loss_all.cpu()[0])
    c_ref, _ = ctc_cpu(acts.cpu().numpy(), wl.labels, wl.act_lens, wl.label_lens, 0, precision="f64")
    assert abs(total - c_ref.sum()) < LOSS_RTOL * c_ref.sum()


def _call_site_case(rng, B, T, V, Lmax, full_lens=False):
    logits = rng.randn(B, T, V).astype(np.float32)
    y_lens = rng.randint(max(1, Lmax // 2), Lmax + 1, size=B).astype(np.int32)
    ys = np.zeros((B, Lmax), dtype=np.int64)
    for b in range(B):
        ys[b, :y_lens[b]] = rng.randint(0, V - 1, size=y_lens[b])
    x_lens = np.full(B, T, np.int32) if full_lens else np.sort(rng.randint(T - T // 4, T + 1, size=B))[::-1].astype(np.int32)
    x_lens[0] = T
    return logits, ys, x_lens, y_lens


@pytest.mark.parametrize("B,T,V,Lmax", [(5, 60, 11, 9), (6, 500, 30, 220), (4, 200, 30, 6), (4, 160, 62, 70),
                                        (3, 260, 100, 120), (3, 200, 300, 80), (2, 120, 1500, 50)])
@pytest.mark.parametrize("temp,ls", [(1.0, 0.1), (2.0, 0.0), (1.3, 0.2)])
def test_fused_call_site_temperature_average_label_smoothing(B, T, V, Lmax, temp, ls):
    """ctc_loss_from_padded = ctc.py:299-337 in one device-resident call: logits / temperature, / len(xs) and the
    label-smoothing cross entropy are evaluated inside the kernels.  Loss and d loss / d logits against the fp64
    restatement of the reference's call site (every reducer path: one / two symbols per lane, the loop, the
    untouched vocabulary entries, gathered mode with both softmax kernels)."""
    rng = np.random.RandomState(B * 1000 + V + int(temp * 10) + int(ls * 100))
    logits_np, ys, x_lens, y_lens = _call_site_case(rng, B, T, V, Lmax)
    logits = torch.from_numpy(logits_np).cuda().requires_grad_(True)
    loss = b200.ctc_loss_from_padded(logits, ys, x_lens, y_lens, logits_temperature=temp, label_smoothing=ls)
    loss.backward()
    torch.cuda.synchronize()
    loss_ref, g_ref = ctc_ref.ctc_loss_call_site(logits_np, ys, x_lens, y_lens, temp, ls)
    assert abs(float(loss.detach().cpu()[0]) - loss_ref) < LOSS_RTOL * abs(loss_ref)
    g = logits.grad.cpu().numpy()
    assert np.max(np.abs(g - g_ref)) < GRAD_ATOL / B             # the gradient carries the 1/B of the loss
    for b in range(B):
        assert np.all(g[b, x_lens[b]:] == 0)                     # padded frames: exactly zero
    assert ctc_mod.last_fallbacks(with_invalid=True) == (0, 0, 0)


def test_fused_options_defaults_are_bit_identical_and_safe_path_honours_them():
    rng = np.random.RandomState(51)
    logits_np, ys, x_lens, y_lens = _call_site_case(rng, 4, 80, 12, 10)
    logits_np[1] *= 60.0                                          # utterance 1: extreme rows -> fp64 safe lattice
    acts = torch.from_numpy(logits_np).cuda().transpose(0, 1)
    ys_d = torch.from_numpy(ys + 1).to(torch.int32).cuda()
    xl, yl = torch.from_numpy(x_lens).cuda(), torch.from_numpy(y_lens).cuda()
    base = b200.ctc_loss_and_grad(acts, ys_d, xl, yl)
    same = b200.ctc_loss_and_grad(acts, ys_d, xl, yl, logit_scale=1.0, label_smoothing=0.0, loss_scale=1.0, grad_scale=1.0)
    assert torch.equal(base[0], same[0]) and torch.equal(base[2], same[2]) and torch.equal(base[1], same[1])
    assert ctc_mod.last_fallbacks()[0] >= 1
    logits = torch.from_numpy(logits_np).cuda().requires_grad_(True)
    loss = b200.ctc_loss_from_padded(logits, ys, x_lens, y_lens, logits_temperature=1.5, label_smoothing=0.1)
    loss.backward()
    loss_ref, g_ref = ctc_ref.ctc_loss_call_site(logits_np, ys, x_lens, y_lens, 1.5, 0.1)
    assert abs(float(loss.detach().cpu()[0]) - loss_ref) < LOSS_RTOL * abs(loss_ref)
    assert np.max(np.abs(logits.grad.cpu().numpy() - g_ref)) < GRAD_ATOL / 4


def test_fused_call_site_cost_only_and_upstream_gradient():
    rng = np.random.RandomState(52)
    logits_np, ys, x_lens, y_lens = _call_site_case(rng, 5, 90, 30, 25)
    with torch.no_grad():
        loss0 = b200.ctc_loss_from_padded(torch.from_numpy(logits_np).cuda(), ys, x_lens, y_lens,
                                          logits_temperature=2.0, label_smoothing=0.15)
    loss_ref, g_ref = ctc_ref.ctc_loss_call_site(logits_np, ys, x_lens, y_lens, 2.0, 0.15)
    assert abs(float(loss0.cpu()[0]) - loss_ref) < LOSS_RTOL * abs(loss_ref)
    logits = torch.from_numpy(logits_np).cuda().requires_grad_(True)
    (3.0 * b200.ctc_loss_from_padded(logits, ys, x_lens, y_lens, logits_temperature=2.0, label_smoothing=0.15)).sum().backward()
    assert np.max(np.abs(logits.grad.cpu().numpy() - 3.0 * g_ref)) < 3 * GRAD_ATOL / 5


def test_back_to_back_device_resident_calls_and_single_call_graph_replays_do_not_race():
    """The plan kernel of a call runs underneath the lattice kernel of the previous call (programmatic dependent
    launch) and writes the shared tables only after that kernel has completed: consecutive calls with DIFFERENT
    lengths on one stream, and back-to-back replays of a graph that holds a single call, must each give the
    result of an isolated call."""
    wls = [workloads.make_lengths_and_labels(None, B=48, T=300, V=30, Lmax=120, kind="var", seed=70 + i) for i in range(3)]
    acts = [workloads.make_acts(w, copy_index=i).cuda() for i, w in enumerate(wls)]
    pads = [padded(w, 120) for w in wls]
    ref = []
    for a, (ys, al, ll) in zip(acts, pads):
        r = b200.ctc_loss_and_grad(a, ys, al, ll)
        torch.cuda.synchronize()
        ref.append((r[0].clone(), r[2].clone()))
    for rep in range(5):
        outs = [b200.ctc_loss_and_grad(a, ys, al, ll) for a, (ys, al, ll) in zip(acts, pads)]   # no sync in between
        torch.cuda.synchronize()
        for (c, _, g), (c0, g0) in zip(outs, ref):
            assert torch.equal(c, c0) and torch.equal(g, g0)
    # one call per graph, replayed without synchronisation, inputs swapped by copies on the same stream
    a, (ys, al, ll) = acts[0].clone(), tuple(x.clone() for x in pads[0])
    grads, costs, loss = torch.empty_like(a), torch.empty(48, device="cuda"), torch.empty(1, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        b200.ctc_loss_and_grad(a, ys, al, ll, grads=grads, costs=costs, loss_sum=loss)
        torch.cuda.synchronize()
        with torch.cuda.graph(graph, stream=s):
            b200.ctc_loss_and_grad(a, ys, al, ll, grads=grads, costs=costs, loss_sum=loss)
        got = []
        for k in range(9):
            i = k % 3
            a.copy_(acts[i]); ys.copy_(pads[i][0]); al.copy_(pads[i][1]); ll.copy_(pads[i][2])
            graph.replay()
            got.append((costs.clone(), grads.clone()))
    torch.cuda.synchronize()
    for k, (c, g) in enumerate(got):
        assert torch.equal(c, ref[k % 3][0]) and torch.equal(g, ref[k % 3][1]), k


@pytest.mark.parametrize("B,T,V,Lmax", [(6, 300, 30, 140), (3, 500, 30, 400), (8, 120, 62, 40), (4, 200, 300, 60), (2, 64, 12, 0)])
def test_cluster_and_single_cta_lattice_agree(B, T, V, Lmax, monkeypatch):
    """Mini-batches that leave half of the SMs idle run the lattice as a two-CTA thread-block cluster per utterance
    (alpha sweep on one SM, beta sweep on another); B200CTC_CLUSTER=0/1 forces either variant.  Same arithmetic in
    the same order: bit-identical costs and gradients, and both within tolerance of the oracle."""
    wl = workloads.make_lengths_and_labels(None, B=B, T=T, V=V, Lmax=max(Lmax, 1), kind="var", seed=90 + B)
    if Lmax == 0:
        wl = workloads.Workload(wl.name, T, B, V, np.zeros(0, np.int32), np.zeros(B, np.int32), wl.act_lens, 0)
    acts_t = workloads.make_acts(wl)
    acts = acts_t.cuda()
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("B200CTC_CLUSTER", mode)
        c, l, g = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
        c2 = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens, need_grad=False)[0]
        torch.cuda.synchronize()
        assert ctc_mod.last_fallbacks() == (0, 0)
        out[mode] = (c.clone(), l.clone(), g.clone(), c2.clone())
    for a, b_ in zip(out["0"], out["1"]):
        assert torch.equal(a, b_)
    assert_parity(out["1"][0], out["1"][2], acts_t.numpy(), wl)


def test_cluster_variant_falls_back_to_the_safe_lattice(monkeypatch):
    monkeypatch.setenv("B200CTC_CLUSTER", "1")
    rng = np.random.RandomState(95)
    wl = workloads.make_lengths_and_labels(None, B=4, T=90, V=12, Lmax=20, kind="var", seed=95)
    acts = workloads.make_acts(wl).numpy()
    acts[:, 1] *= 60.0                                             # extreme rows: utterance 1 takes the fp64 safe lattice
    c, l, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), wl.labels, wl.act_lens, wl.label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks()[0] >= 1
    c_ref, g_ref = ctc_ref.ctc_cost_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    assert np.max(np.abs(c.cpu().numpy() - c_ref) / np.maximum(np.abs(c_ref), 1e-3)) < LOSS_RTOL
    assert np.max(np.abs(g.cpu().numpy() - g_ref)) < GRAD_ATOL


@pytest.mark.parametrize("key,repeats", [("C3", 150), ("C5", 60), ("C2", 60)])
def test_results_do_not_depend_on_what_the_workspace_held(key, repeats):
    """The call's scratch is uninitialised memory: whatever it holds on entry (here NaN bit patterns) must never
    reach a result.  Caught a missing proxy fence at the lattice's midpoint -- bulk copies of the records written
    just before the rendezvous could deliver the old contents for about one call in fifty (one utterance NaN or
    rescaled by 1e-6) -- which same-input repeats cannot see, because the stale records then are the right ones."""
    import ctypes
    from pytorch_end2end_speech_recognition_b200 import _lib
    lib = _lib.load()                     # signatures set by _lib.declare
    ip = ctypes.POINTER(ctypes.c_int)
    wl = workloads.make_lengths_and_labels(key)
    acts = workloads.make_acts(wl).cuda()
    h = ctypes.c_void_p()
    assert lib.b200ctc_create(ctypes.byref(h), torch.cuda.current_device()) == 0
    n = ctypes.c_size_t()
    ll, al, lab = wl.label_lens.ctypes.data_as(ip), wl.act_lens.ctypes.data_as(ip), wl.labels.ctypes.data_as(ip)
    assert lib.b200ctc_get_workspace_size(ll, al, wl.T, wl.V, wl.B, ctypes.byref(n)) == 0
    ws = torch.empty(n.value, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    first = None
    try:
        for it in range(repeats):
            ws.fill_(0xff)
            grads = torch.full_like(acts, float("nan"))
            costs, loss = torch.empty(wl.B, device="cuda"), torch.empty(1, device="cuda")
            st = lib.b200ctc_loss_and_grad(h, acts.data_ptr(), acts.stride(0), acts.stride(1), grads.data_ptr(), lab, ll, al,
                                           wl.T, wl.V, wl.B, 0, costs.data_ptr(), loss.data_ptr(), ws.data_ptr(), n.value, stream)
            assert st == 0
            torch.cuda.synchronize()
            if first is None:
                first = (grads, costs)
                assert bool(torch.isfinite(grads).all()) and bool(torch.isfinite(costs).all())
            else:
                assert torch.equal(costs, first[1]), "costs changed at repeat %d" % it
                assert torch.equal(grads, first[0]), "gradients changed at repeat %d" % it
    finally:
        lib.b200ctc_destroy(h)


@pytest.mark.parametrize("V", [301, 515, 1003])
@pytest.mark.parametrize("layout", ["contiguous", "batch_major_view", "offset_by_one_float", "offset_by_three_floats"])
def test_streaming_softmax_row_alignment(V, layout):
    """K1 for V > 256 moves the 16-byte-aligned window around every row with a TMA bulk copy: rows at every
    16-byte phase (odd V), source and destination rows at different phases (batch-major view), and a tensor whose
    first / last rows' windows would leave it (base not 16-byte aligned: those rows take plain loads)."""
    wl = workloads.make_lengths_and_labels(None, B=5, T=37, V=V, Lmax=9, kind="var", seed=V)
    ref_acts = workloads.make_acts(wl)                                  # [T, B, V] on the host
    if layout == "contiguous":
        acts = ref_acts.cuda()
    elif layout == "batch_major_view":
        acts = ref_acts.transpose(0, 1).contiguous().cuda().transpose(0, 1)
        assert not acts.is_contiguous()
    else:
        k = 1 if layout == "offset_by_one_float" else 3
        buf = torch.empty(ref_acts.numel() + 8, device="cuda")
        acts = buf[k:k + ref_acts.numel()].view(wl.T, wl.B, V)
        acts.copy_(ref_acts)
        assert acts.data_ptr() % 16 == 4 * k
    costs, loss, grads = b200.ctc_loss_and_grad(acts, wl.labels, wl.act_lens, wl.label_lens)
    torch.cuda.synchronize()
    c_ref, g_ref = ctc_ref.ctc_cost_and_grad(ref_acts.numpy(), wl.labels, wl.act_lens, wl.label_lens)
    c = costs.cpu().numpy()
    assert np.max(np.abs(c - c_ref) / np.maximum(np.abs(c_ref), 1e-3)) < LOSS_RTOL
    g = grads.cpu().numpy()
    assert np.max(np.abs(g - g_ref)) < GRAD_ATOL
    for b in range(wl.B):
        assert np.all(g[wl.act_lens[b]:, b] == 0)                       # padding rows: exactly zero
    assert ctc_mod.last_fallbacks() == (0, 0)


@pytest.mark.parametrize("V,L,expo", [(30, 400, 1.0), (30, 380, 1.5), (30, 250, 0.7), (62, 330, 1.2), (50, 120, 2.0),
                                      (64, 400, 1.0), (33, 64, 1.5)])
@pytest.mark.parametrize("cluster", ["0", "1"])
def test_split_symbol_groups_of_text_like_labels(V, L, expo, cluster, monkeypatch):
    """Text-like label statistics (p_k ~ 1 / k^s: a few symbols carry most of the labels): the reducers cut the slot
    range of a frequent symbol into pieces that several lanes sum and combine (one or two groups per lane, pieces
    wrapping from the first slot of lane 31 into the second slot of lane 0), in both lattice variants."""
    monkeypatch.setenv("B200CTC_CLUSTER", cluster)
    rng = np.random.RandomState(V * 100 + L)
    p = 1.0 / (np.arange(V - 1) + 1.0) ** expo
    p /= p.sum()
    lab = 1 + rng.choice(V - 1, size=L, p=p)
    lab2 = 1 + rng.choice(V - 1, size=L // 2, p=p[::-1])          # the rare symbols of the first utterance are the frequent ones here
    T = L + ctc_ref.count_repeats(lab) + 40
    T2 = len(lab2) + ctc_ref.count_repeats(lab2) + 11
    acts = rng.randn(T, 2, V).astype(np.float32)
    labels = np.concatenate([lab, lab2]).astype(np.int32)
    c, g = None, None
    costs, loss, grads = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), labels, np.array([T, T2], np.int32),
                                                np.array([L, len(lab2)], np.int32))
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, 0)
    c_ref, g_ref = ctc_cpu(acts, labels, np.array([T, T2], np.int32), np.array([L, len(lab2)], np.int32), 0, precision="f64")
    assert np.max(np.abs(costs.cpu().numpy() - c_ref) / np.maximum(np.abs(c_ref), 1e-3)) < LOSS_RTOL
    assert np.max(np.abs(grads.cpu().numpy() - g_ref)) < GRAD_ATOL
    # with the call-site options (every entry of a live row rewritten: the untouched-symbol list next to split groups)
    logits = torch.from_numpy(np.ascontiguousarray(acts.transpose(1, 0, 2))).cuda().requires_grad_(True)
    ys = np.zeros((2, L), np.int64)
    ys[0, :L] = lab - 1
    ys[1, :len(lab2)] = lab2 - 1
    x_lens, y_lens = np.array([T, T2], np.int32), np.array([L, len(lab2)], np.int32)
    out = b200.ctc_loss_from_padded(logits, ys, x_lens, y_lens, logits_temperature=1.3, label_smoothing=0.1)
    out.backward()
    loss_ref, gl_ref = ctc_ref.ctc_loss_call_site(acts.transpose(1, 0, 2), ys, x_lens, y_lens, 1.3, 0.1)
    assert abs(float(out.detach().cpu()[0]) - loss_ref) < LOSS_RTOL * abs(loss_ref)
    assert np.max(np.abs(logits.grad.cpu().numpy() - gl_ref)) < GRAD_ATOL / 2


@pytest.mark.parametrize("V,L", [(1500, 190), (1500, 205), (1500, 222), (1500, 240), (200, 236), (30, 463)])
def test_record_ring_depth_follows_the_label_sequence(V, L):
    """The lattice's record ring is four chunks deep when the shared memory allows and three or two when the longest
    label sequence needs the room (gathered mode: the emission-row ring grows with the labels): label sequences up
    to the capacity of the shallowest ring (195 / 210 / 226 labels for V >= 1000) still run on the block-exponent
    lattice, longer ones on the safe lattice in the same launch; every depth gives the oracle's result."""
    rng = np.random.RandomState(V + L)
    labs = [rng.randint(1, V, size=n) for n in (L, L // 3)]
    T = L + ctc_ref.count_repeats(labs[0]) + 24
    acts = rng.randn(T, 2, V).astype(np.float32)
    wl = workloads.Workload("x", T, 2, V, np.concatenate(labs).astype(np.int32), np.array([len(x) for x in labs], np.int32),
                            np.array([T, T - 7], np.int32), 0)
    c, loss, g = b200.ctc_loss_and_grad(torch.from_numpy(acts).cuda(), wl.labels, wl.act_lens, wl.label_lens)
    torch.cuda.synchronize()
    assert ctc_mod.last_fallbacks() == (0, 0)
    assert_parity(c, g, acts, wl)
