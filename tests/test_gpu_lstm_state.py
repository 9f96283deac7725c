"""GPU: the LSTM recurrence checked state by state.  Every case runs
  (a) the training forward and the teacher-forced float64 check of its tape (oracle/lstm_step.py: every valid
      (layer, b, t) step recomputed from the h_{t-1}, c_{t-1} the kernel used -- gates, c_t, h_t, and h_t == 0 exactly
      past the length), with guards that the weights keep the gates informative;
  (b) the inference forward with an identity head (y_dim = H, W = I, b = 0): the bf16 head GEMM then returns the top
      layer's h exactly, which must be bit-identical to the training forward's tape (zeros past the length included),
      and last_logits must be h[b, max(len_b - 1, 0)];
  (c) a y_dim = 1 head on the same weights (head1_kernel) against the float64 head over the tape's h, with
      post = sigmoid(logits) and dec = post > 0.5.
Shapes cover every recurrence path the driver picks (csrc/lstm.cu): the CTA-pair kernel with chunk-interleaved layers
(H = 1024, and H = 832 / 960 with an odd number of K blocks), one and two chunks, one and two 128-row batch slices,
two batch groups, padded input widths, the one-CTA-per-block persist kernel at H = 64 .. 768 across batch groups,
1 and 3 layers (the loop without chunks), and the per-step GEMM fallback at H = 1088.  Lengths always include 0, 1, T
and the steps around every chunk boundary."""
import math

import pytest
import torch

from avvad import engine as E
from avvad import lib as L
from oracle import lstm_step as S
from util import lstm_test_weights

pytestmark = pytest.mark.gpu

# Bounds at about twice the maxima measured on a B200 (1000 W) over every case below
HEAD_REL = 2e-7    # y_dim = 1 head: |logit - ref| / (|b| + sum_k |h_k w_k|), fp32 dot product; measured 8.9e-8
POST_ABS = 2e-7    # |post - sigmoid(logit)|: one fp32 expf and division; measured 8.5e-8


def _n_chunks(T):
    """Chunks of the two-layer forward at this T (csrc/lstm.cu: up to 8, each at least 16 steps)."""
    n = 8
    while n > 1 and T // n < 16:
        n -= 1
    return n


def _lengths(B, T, seed):
    n = _n_chunks(T)
    special = [T, 0, 1]
    for c in range(1, n):
        t1 = T * c // n
        special += [t1 - 1, t1, t1 + 1]
    special = [min(max(v, 0), T) for v in special]
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(0, T + 1, (B,), generator=g).tolist()
    for i, v in enumerate(special[:B]):
        lens[i] = v
    if B >= 2 * len(special):   # and at the end: the last batch slice / group
        for i, v in enumerate(special):
            lens[B - 1 - i] = v
    return lens


def _handle(layers, I, H, ws, head_w, head_b):
    lstm = E.Lstm(layers, I, H, head_w.shape[0])
    sd = {"head.weight": head_w, "head.bias": head_b}
    for l, w in enumerate(ws):
        for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), w):
            sd[f"lstm.{name}_l{l}"] = t
    lstm.load(sd, "cuda", "lstm", "head")
    return lstm


def _inputs(lstm, B, T, I, seed):
    g = torch.Generator().manual_seed(seed)
    xs = (0.5 * torch.randn(B, T, I, generator=g)).to(torch.bfloat16).cuda()
    x = lstm.new_input(B, T, "cuda")   # columns >= I stay zero (the API contract)
    x[..., :I] = xs
    return xs, x


def _run_case(H, I, layers, B, T, seed=0):
    tag = f"[H={H} I={I} layers={layers} B={B} T={T}]"
    ws = lstm_test_weights(layers, I, H, seed)
    lens = _lengths(B, T, seed + 2)
    ident = _handle(layers, I, H, ws, torch.eye(H), torch.zeros(H))
    xs, x = _inputs(ident, B, T, I, seed + 1)

    # (a) training forward: the tape against the float64 step reference
    lg_train, pack = E.lstm_train_forward(ident, x, lens)
    views = E.lstm_tape_views(ident, pack, B, T)
    rep = S.check_tape(views, xs, lens, ws)
    print(f"{tag} tape vs float64 step reference\n{rep.summary()}")
    assert rep.ok, f"{tag} {rep.message()}"
    if T >= 16:   # over one or two steps an upper layer only sees the first, small h of the layer below
        assert all(0.3 <= s <= 3.0 for s in rep.pre_std), (tag, rep.pre_std)
    assert all(s < 0.05 for s in rep.saturated), (tag, rep.saturated)
    h_top = views[-1][2]
    lens_t = torch.tensor(lens, device="cuda")
    assert torch.equal(lg_train, h_top.float()), f"{tag} training forward's identity head != its tape's top h"

    # (b) inference forward, identity head: bit-identical to the tape
    logits, _, _, last = ident.forward(x, lens, want_last=True)
    same = logits == h_top.float()
    assert bool(same.all()), f"{tag} inference h != training tape h at {int((~same).sum())} entries, first (b, t, u) " \
                             f"{tuple(int(v) for v in (~same).nonzero()[0])}"
    at = (lens_t - 1).clamp(min=0)
    h_last = h_top[torch.arange(B, device="cuda"), at].float()
    assert torch.equal(last, h_last), f"{tag} last_logits != h[b, max(len_b - 1, 0)]"
    del ident, logits, lg_train

    # (c) y_dim = 1 head on the same weights
    g = torch.Generator().manual_seed(seed + 3)
    w1 = torch.randn(1, H, generator=g) * (3.0 / math.sqrt(H))
    b1 = torch.tensor([0.25])
    one = _handle(layers, I, H, ws, w1, b1)
    lg1, post, dec, last1 = one.forward(x, lens, want_post=True, want_dec=True, want_last=True)
    hd = h_top.double()
    wd = w1.double().cuda()
    ref = hd @ wd.t() + float(b1)
    scale = hd.abs() @ wd.abs().t() + abs(float(b1))
    head_err = float(((lg1.double() - ref).abs() / scale).max())
    ref_last = hd[torch.arange(B, device="cuda"), at] @ wd.t() + float(b1)
    last_err = float(((last1.double() - ref_last).abs() / (hd[torch.arange(B, device="cuda"), at].abs() @ wd.abs().t()
                                                           + abs(float(b1)))).max())
    post_err = float((post.double() - torch.sigmoid(lg1.double())).abs().max())
    print(f"{tag} y_dim=1 head: logits {head_err:.2e}, last {last_err:.2e} (bound {HEAD_REL:.0e} relative), "
          f"post {post_err:.2e} (bound {POST_ABS:.0e}), logit std {float(lg1.std(correction=0)):.3f}")
    assert head_err <= HEAD_REL and last_err <= HEAD_REL, tag
    assert post_err <= POST_ABS, tag
    assert torch.equal(dec, (post > 0.5).int()), tag
    del one, pack, views
    torch.cuda.empty_cache()


# (B, T): pair kernel with chunk-interleaved layers, I = H = 1024
H1024_SHAPES = [
    (1, 1), (3, 2),
    (7, 31),      # one chunk
    (64, 32),     # two chunks; the second CTA of every pair has no rows
    (128, 48), (129, 40),
    (200, 130),
    (256, 317),   # the benchmarked shape
    (257, 33), (300, 64),   # two batch groups
]


@pytest.mark.parametrize("B,T", H1024_SHAPES, ids=[f"B{b}_T{t}" for b, t in H1024_SHAPES])
def test_h1024_two_layers(B, T):
    _run_case(1024, 1024, 2, B, T)


@pytest.mark.parametrize("I", [513, 1025])   # padded operand widths 576 and 1088
def test_input_width(I):
    _run_case(1024, I, 2, 130, 50)


# (H, B) at T = 40: the persist kernel (H <= 768: 128-row x 64-column CTAs, Bg = min(16, 148 / (H / 16)) * 128 rows per
# cooperative launch, B spans two groups) and the pair kernel with an odd number of 64-unit K blocks (832: 13, 960: 15)
OTHER_H = [(64, 2100), (128, 2100), (256, 1200), (512, 600), (768, 400), (832, 300), (960, 300)]


@pytest.mark.parametrize("H,B", OTHER_H, ids=[f"H{h}_B{b}" for h, b in OTHER_H])
def test_other_hidden_sizes(H, B):
    _run_case(H, 513, 2, B, 40)


@pytest.mark.parametrize("layers", [1, 3])   # the layer loop without chunks
def test_layer_counts(layers):
    _run_case(1024, 1024, layers, 150, 70)


GEMM_FALLBACK_H_ABS = 4e-3   # free-running h (see below); measured 1.95e-3 at T = 40 on a B200


def test_per_step_gemm_fallback_h1088():
    """H > 1024 has no persistent recurrence: every step is one tcgen05 GEMM with the cell update in its epilogue
    (EPI_LSTM).  The training forward needs the persistent kernel and must refuse with a message.  The inference forward
    (identity head) is compared free-running with the float64 emulator: the kernel's bf16 h feeds back into its next
    step, so unlike the teacher-forced bounds this one can grow with T; at T = 40 the measured difference is still the
    bf16 rounding of h (1.95e-3)."""
    H, I, B, T = 1088, 513, 130, 40
    ws = lstm_test_weights(1, I, H, 7)
    lens = _lengths(B, T, 9)
    ident = _handle(1, I, H, ws, torch.eye(H), torch.zeros(H))
    xs, x = _inputs(ident, B, T, I, 8)
    with pytest.raises(L.AvvadError, match="persistent recurrence"):
        E.lstm_train_forward(ident, x, lens)
    logits, _, _, last = ident.forward(x, lens, want_last=True)
    h_emu = S.emulate_tape(xs, lens, ws)[0][2]
    valid = torch.arange(T, device="cuda").view(1, T) < torch.tensor(lens, device="cuda").view(B, 1)
    err = (logits - h_emu.float()).abs().amax(-1)
    max_err = float(err[valid].max())
    print(f"[H={H} I={I} layers=1 B={B} T={T}] per-step GEMM, free-running h vs emulator: max {max_err:.3e} "
          f"(bound {GEMM_FALLBACK_H_ABS:.0e}), first step {float(err[:, 0][valid[:, 0]].max()):.3e}")
    assert max_err <= GEMM_FALLBACK_H_ABS
    assert bool((logits[~valid] == 0).all()), "h past the length must be exactly 0"
    at = (torch.tensor(lens, device="cuda") - 1).clamp(min=0)
    assert torch.equal(last, logits[torch.arange(B, device="cuda"), at])
