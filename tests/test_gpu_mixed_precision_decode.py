"""GPU tests of the decoders and the evaluation path on bfloat16 and float16 logits.

Every 16-bit call must give exactly what the same call gives on ``x.float()`` (widening is exact, so there is no
tolerance), and the greedy results must also equal the oracle's numpy arg-max.  The greedy cases cover each arg-max
kernel (group V <= 64, warp V <= 512, streaming) and both keys of the streaming kernel (32-bit on raw bits for
V <= 65536, 64-bit on widened values above)."""
import os

import numpy as np
import pytest
import torch

import pytorch_end2end_speech_recognition_b200 as b200
from pytorch_end2end_speech_recognition_b200 import B200CTCError
from oracle import ctc_ref

pytestmark = pytest.mark.gpu

DTYPES = [torch.bfloat16, torch.float16]
VOCABS = [5, 30, 33, 64, 65, 512, 513, 3386, 4100, 65537]
# NaN bit patterns (both signs, several payloads) as int16
NANS = {torch.bfloat16: [0x7fc0, 0xffc0, 0x7f81, 0xff81, 0x7fff, 0xffff],
        torch.float16: [0x7e00, 0xfe00, 0x7c01, 0xfc01, 0x7fff, 0xffff]}


def i16(bits):
    return bits - 0x10000 if bits >= 0x8000 else bits


def greedy_pair(x, lens, blank=0):
    """greedy_decode on x and on x.float(): both must agree exactly; returns the first."""
    t16, l16 = b200.greedy_decode(x, lens, blank)
    t32, l32 = b200.greedy_decode(x.float(), lens, blank)
    assert torch.equal(t16, t32) and torch.equal(l16, l32)
    return t16, l16


def check_oracle(x, lens, tokens, out_lens, blank=0):
    T = x.shape[1]
    clamped = np.clip(np.asarray(lens), 0, T)
    ref = ctc_ref.greedy_decode(x.float().cpu().numpy(), clamped, blank)
    tokens, out_lens = tokens.cpu().numpy(), out_lens.cpu().numpy()
    for b, h in enumerate(ref):
        assert out_lens[b] == len(h), b
        assert np.array_equal(tokens[b, :out_lens[b]], h), b
        assert np.all(tokens[b, out_lens[b]:] == -1), b


def shape_for(V):
    return (2, 9) if V > 10000 else (3, 40)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", VOCABS)
def test_greedy_random_logits_with_ties(V, dtype):
    B, T = shape_for(V)
    g = torch.Generator(device="cuda").manual_seed(V)
    # a coarse grid: 16-bit rounding of small integers and halves leaves many exact ties in every row
    x = (torch.randint(-6, 7, (B, T, V), device="cuda", generator=g).float() * 0.5).to(dtype)
    lens = [T, 0, T + 5][:B] if B == 3 else [T + 3, -2]
    blank = 0 if V < 10 else 3
    tokens, out_lens = greedy_pair(x, lens, blank)
    check_oracle(x, lens, tokens, out_lens, blank)
    y = torch.randn(B, T, V, device="cuda", generator=g).to(dtype)
    lens = [T, T - 7, 1][:B]
    tokens, out_lens = greedy_pair(y, lens, blank)
    check_oracle(y, lens, tokens, out_lens, blank)


def special_rows(B, T, V, dtype, seed):
    """Rows of random values with NaN (both signs, several payloads), +-inf and +-0 at positions in the head, the
    unrolled body, the single-vector body and the tail of the streaming kernel's row split."""
    rng = np.random.RandomState(seed)
    x = (rng.randn(B, T, V) - 3.0).astype(np.float32)
    bits = torch.from_numpy(x).to(dtype).view(torch.int16).numpy().copy()
    inf = 0x7f80 if dtype == torch.bfloat16 else 0x7c00
    nvec_unrolled = 32 * 8 * 8                              # elements one unrolled trip of a warp covers
    cands = sorted(set([0, 1, 2, 3, 5, 7, 8, 9, V // 2, min(nvec_unrolled + 3, V - 1), min(nvec_unrolled + 300, V - 1)]
                       + [V - k for k in range(1, 9) if V - k >= 0]))
    cands = [c for c in cands if 0 <= c < V]
    for b in range(B):
        for t in range(T):
            kind = (b * T + t) % 6
            row = bits[b, t]
            pos = rng.choice(cands, size=min(3, len(cands)), replace=False)
            if kind == 0:                                   # NaNs of mixed sign and payload
                for p in pos:
                    row[p] = i16(NANS[dtype][rng.randint(len(NANS[dtype]))])
            elif kind == 1:                                 # +inf twice and -inf: the first +inf wins
                row[pos[0]] = i16(inf); row[pos[-1]] = i16(inf); row[pos[1 % len(pos)]] = i16(inf | 0x8000)
            elif kind == 2:                                 # all negative but some zeros of either sign: first zero wins
                for p in pos:
                    row[p] = i16(0x8000) if rng.randint(2) else 0
            elif kind == 3:                                 # all -inf, one -0 somewhere
                row[:] = i16(inf | 0x8000)
                if rng.randint(2):
                    row[pos[0]] = i16(0x8000)
            elif kind == 4:                                 # -0 before +0 as the row's only maxima
                row[:] = i16(inf | 0x8000)
                p0, p1 = sorted(pos[:2]) if len(pos) > 1 else (pos[0], pos[0])
                row[p0] = i16(0x8000); row[p1] = 0
            # kind 5: random values only
    return torch.from_numpy(bits).view(dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", VOCABS)
def test_greedy_nan_inf_and_signed_zero_at_every_alignment(V, dtype):
    B, T = (2, 6) if V > 10000 else (3, 12)
    rows = special_rows(B, T, V, dtype, V + (dtype == torch.float16)).cuda()
    n = B * T * V
    flat = torch.empty(n + 8, dtype=dtype, device="cuda")
    lens = [T] * B
    for phase in range(8):                                  # base pointer at every 2-byte phase of a 16-byte line
        flat.view(torch.int16).fill_(0x1234)
        x = flat[phase:phase + n].view(B, T, V)
        x.copy_(rows)
        tokens, out_lens = greedy_pair(x, lens, blank=1)
        check_oracle(x, lens, tokens, out_lens, blank=1)
        # the frame arg-max itself, through one-frame utterances and a blank that is no symbol (nothing collapses)
        t1, _ = greedy_pair(x.reshape(B * T, 1, V), [1] * (B * T), blank=-1)
        ref = np.argmax(x.float().cpu().numpy().reshape(B * T, V), axis=1)
        assert np.array_equal(t1[:, 0].cpu().numpy(), ref)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", [30, 300, 3386])
def test_greedy_batch_major_view_of_time_major_logits(V, dtype):
    B, T = 5, 37
    g = torch.Generator(device="cuda").manual_seed(7)
    tm = torch.randn(T, B, V, device="cuda", generator=g).to(dtype)
    x = tm.transpose(0, 1)
    lens = [37, 0, 12, 40, -1]
    tokens, out_lens = greedy_pair(x, lens, blank=2)
    check_oracle(x, lens, tokens, out_lens, blank=2)


@pytest.mark.parametrize("dtype", DTYPES)
def test_greedy_full_c4_batch(dtype):
    B, T, V = 64, 1000, 3386                                # warps loop over several rows each
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(B, T, V, device="cuda", generator=g).to(dtype)
    lens = torch.randint(500, T + 1, (B,), device="cuda", generator=g)
    greedy_pair(x, lens)
    ref = torch.argmax(x.float(), dim=-1).int()
    tok, _ = greedy_pair(x.reshape(B * T, 1, V), torch.ones(B * T, dtype=torch.int32, device="cuda"), blank=-1)
    assert torch.equal(tok[:, 0], ref.reshape(-1))          # torch's arg-max: first index on ties, no NaN here


def beam_pair(lp, lens, W, blank=0):
    out16 = b200.beam_search_decode(lp, lens, W, blank=blank, return_scores=True)
    out32 = b200.beam_search_decode(lp.float(), lens, W, blank=blank, return_scores=True)
    for a, b in zip(out16, out32):
        assert torch.equal(a, b)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("W", [1, 2, 10, 64])
def test_beam_search_on_rounded_golden_log_probs(golden_dir, W, dtype):
    z = np.load(os.path.join(golden_dir, "beam_golden.npz"))
    for i in range(int(z["n_cases"])):
        lp = torch.from_numpy(z["log_probs_%d" % i]).cuda().to(dtype)
        beam_pair(lp, z["x_lens_%d" % i], W)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("W", [1, 2, 10, 64])
def test_beam_search_on_log_softmax_of_16bit_logits(W, dtype):
    g = torch.Generator(device="cuda").manual_seed(W)
    B, T, V = 3, 30, 40
    logits = (torch.randn(B, T, V, device="cuda", generator=g) * 2.0).to(dtype)
    lp = torch.log_softmax(logits, dim=-1)                  # 16-bit, as autocast's log_softmax of 16-bit logits
    assert lp.dtype == dtype
    beam_pair(lp, [30, 17, 0], W, blank=0)
    beam_pair(lp.transpose(0, 1).contiguous().transpose(0, 1), [30, 31, 5], W, blank=4)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("V", [30, 3386])
@pytest.mark.parametrize("temperature", [1.0, 1.3])
def test_posteriors(V, temperature, dtype):
    g = torch.Generator(device="cuda").manual_seed(V)
    B, T = 4, 50
    x = (torch.randn(B, T, V, device="cuda", generator=g) * 3.0).to(dtype)
    x[1, 3, 5] = float("nan")                               # a NaN row stays NaN in both
    for view in (x, x.transpose(0, 1).contiguous().transpose(0, 1), x[:, ::2]):
        p16 = b200.posteriors(view, temperature)
        p32 = b200.posteriors(view.float(), temperature)
        assert p16.dtype == torch.float32
        torch.testing.assert_close(p16, p32, rtol=0, atol=0, equal_nan=True)


@pytest.mark.parametrize("W", [1, 2, 10])
def test_evaluate_batch_on_bfloat16_logits(W):
    g = torch.Generator(device="cuda").manual_seed(W)
    B, T, V = 6, 60, 31
    logits = (torch.randn(B, T, V, device="cuda", generator=g) * 2.0).to(torch.bfloat16)
    x_lens = torch.tensor([60, 55, 0, 40, 60, 13], device="cuda")
    ys = torch.randint(0, V - 1, (B, 20), device="cuda", generator=g)
    y_lens = torch.tensor([20, 15, 3, 10, 0, 7], device="cuda")
    a = b200.evaluate_batch(logits, x_lens, ys, y_lens, beam_width=W)
    b = b200.evaluate_batch(logits.float(), x_lens, ys, y_lens, beam_width=W)
    for u, v in zip(a, b):
        assert torch.equal(u, v)


def test_decoder_classes_take_bfloat16_tensors():
    g = torch.Generator(device="cuda").manual_seed(0)
    logits = torch.randn(3, 25, 30, device="cuda", generator=g).to(torch.bfloat16)
    x_lens = [25, 20, 3]
    for got, want in ((b200.GreedyDecoder(0)(logits, x_lens), b200.GreedyDecoder(0)(logits.float(), x_lens)),
                      (b200.BeamSearchDecoder(0)(torch.log_softmax(logits, -1), x_lens, beam_width=4),
                       b200.BeamSearchDecoder(0)(torch.log_softmax(logits, -1).float(), x_lens, beam_width=4))):
        assert len(got) == len(want)
        for h, w in zip(got, want):
            assert np.array_equal(h, w)


def test_float64_logits_are_rejected():
    x = torch.randn(2, 5, 30, device="cuda", dtype=torch.float64)
    with pytest.raises(B200CTCError):
        b200.greedy_decode(x, [5, 5])
    with pytest.raises(B200CTCError):
        b200.beam_search_decode(x, [5, 5], 2)
    with pytest.raises(B200CTCError):
        b200.posteriors(x)
