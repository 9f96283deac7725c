"""CPU: the teacher-forced LSTM tape checker (oracle/lstm_step.py) accepts an ideal kernel's tape, restates
oracle.models.lstm_packed, and fails -- at the right (layer, t, b, 64-unit block) -- on each defect a recurrence kernel
can plausibly have.  Also the tape layout the library reports (avvad_lstm_tape_layout) against avvad_lstm_tape_bytes."""
import ctypes as C
import types

import pytest
import torch

from avvad import engine as E
from avvad import lib as L
from oracle import lstm_step as S
from oracle import models as om
from util import lstm_test_weights

B, T, I, H, LAYERS = 130, 40, 80, 128, 2   # B crosses a 128-row batch slice; H = two 64-unit blocks
T1 = 20                                    # the chunk boundary the two-layer forward uses at T = 40 (two chunks)


def _lengths():
    g = torch.Generator().manual_seed(5)
    lens = torch.randint(1, T + 1, (B,), generator=g).tolist()
    lens[:8] = [T, 0, 1, T1, T1 - 1, T1 + 1, T, 2]
    lens[127:130] = [T, T, T]
    return lens


def _weights(seed=3):
    return lstm_test_weights(LAYERS, I, H, seed)


@pytest.fixture(scope="module")
def case():
    g = torch.Generator().manual_seed(11)
    x = (0.5 * torch.randn(B, T, I, generator=g)).to(torch.bfloat16)
    return x, _lengths(), _weights()


def test_emulated_tape_passes(case):
    x, lens, ws = case
    rep = S.check_tape(S.emulate_tape(x, lens, ws), x, lens, ws)
    print(rep.message())
    assert rep.ok, rep.message()
    # an ideal kernel is off by its bf16 storage only: half an ulp of a value below 1 (2^-9), plus 2^-25 because the
    # float64 -> bf16 conversion rounds through fp32 as the kernel's own stores do
    assert rep.stats["gate"].max <= 2 ** -9 + 2 ** -24 and rep.stats["h"].max <= 2 ** -9 + 2 ** -24
    assert rep.stats["c"].max < 1e-6
    assert 0.3 <= min(rep.pre_std) and max(rep.pre_std) <= 3 and max(rep.saturated) < 0.05


def test_step_reference_chained_is_lstm_packed(case):
    """In exact arithmetic (bf16-representable weights, no storage rounding) the step reference chained over t is
    nn.LSTM over packed sequences on the valid frames.  Past the length they differ on purpose: the oracle freezes h
    and c there, the kernel stores h = 0 and keeps updating c."""
    x, lens, ws = case
    sd = {}
    for l, w in enumerate(ws):
        for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), w):
            sd[f"lstm.{name}_l{l}"] = S.bf16_round(t) if name.startswith("weight") else t.double()
    ref = om.lstm_packed(x.double(), lens, sd, "lstm", layers=LAYERS)
    inp = x.double()
    for l, (w_ih, w_hh, b_ih, b_hh) in enumerate(ws):
        h = torch.zeros(B, H, dtype=torch.float64)
        c = torch.zeros(B, H, dtype=torch.float64)
        outs = []
        for t in range(T):
            st = S.step_reference(inp[:, t], h, c, w_ih, w_hh, b_ih, b_hh)
            h, c = st.h, st.c
            outs.append(h)
        out = torch.stack(outs, 1)
        inp = out
    for b, n in enumerate(lens):
        torch.testing.assert_close(out[b, :n], ref[b, :n], rtol=0, atol=1e-12)


def _stale(rows, block, t_at, layer):
    """h_{t-1} of `rows` (units of `block`, or all) replaced by h_{t-2} at one step: a stale flag / missing fence."""
    def hook(l, t, hp, ctx):
        if l != layer or t != t_at:
            return hp
        hp = hp.clone()
        cols = slice(None) if block is None else slice(64 * block, 64 * block + 64)
        hp[rows, cols] = ctx["h"][rows, t - 2, cols].double()
        return hp
    return {"h_prev": hook}


def _x_from_previous_step(t_at):
    def hook(l, t, xt, ctx):
        return ctx["inp"][:, t - 1].double() if (l == 0 and t == t_at) else xt
    return {"x": hook}


def _c_reset(layer, t_at):
    def hook(l, t, c, ctx):
        return torch.zeros_like(c) if (l == layer and t == t_at) else c
    return {"c_prev": hook}


def _swap_if(layer, unit):
    def hook(l, t, pre, ctx):
        if l != layer:
            return pre
        pre = pre.clone()
        pre[:, unit, [0, 1]] = pre[:, unit, [1, 0]]
        return pre
    return {"pre": hook}


def _swap_rows(b0):
    def hook(l, t, xt, ctx):
        if l != 0:
            return xt
        xt = xt.clone()
        xt[[b0, b0 + 1]] = xt[[b0 + 1, b0]]
        return xt
    return {"x": hook}


def _drop_bias(layer, colblock):
    def hook(l, t, pre, ctx):
        if l != layer:
            return pre
        pre = pre.clone().view(pre.shape[0], -1)
        cols = slice(64 * colblock, 64 * colblock + 64)
        pre[:, cols] -= ctx["bias"][cols]
        return pre.view(pre.shape[0], -1, 4)
    return {"pre": hook}


# (name, hooks, layer, t, b, 64-unit block or None, quantity that must report it or None).  The block is asserted only
# where the defect lives in one block of OUTPUT units (the i/f swap, the dropped bias block).  A stale block of the
# INPUT h_{t-1} feeds every gate column through W_hh, so all output blocks of that (layer, t, b) fail and the location
# it can be pinned to is (layer, t, b).  Likewise a whole stale batch slice or an input offset.
MUTATIONS = [
    ("stale_h_block", _stale([5], 1, 7, 0), 0, 7, 5, None, "gate"),
    ("stale_h_batch_slice", _stale(slice(128, 130), None, 12, 1), 1, 12, 128, None, "gate"),
    ("xT_time_offset", _x_from_previous_step(9), 0, 9, 0, None, "gate"),
    ("c_reset_at_chunk_boundary", _c_reset(1, T1), 1, T1, 0, None, "c"),
    ("i_f_swapped_one_unit", _swap_if(0, 70), 0, 0, None, 1, "gate"),
    ("xT_rows_swapped", _swap_rows(40), 0, 0, 40, None, "gate"),
    ("bias_dropped_one_column_block", _drop_bias(1, 5), 1, 0, None, 1, "gate"),   # columns 320..383 = units 80..95
    ("h_nonzero_at_len", None, 1, T1, 3, None, "h_pad"),
]


@pytest.mark.parametrize("name,hooks,layer,t,b,block,quantity", MUTATIONS, ids=[m[0] for m in MUTATIONS])
def test_mutation_is_caught(case, name, hooks, layer, t, b, block, quantity):
    x, lens, ws = case
    tape = S.emulate_tape(x, lens, ws, hooks)
    if name == "h_nonzero_at_len":
        # the row's live h_t = o tanh(c_t) stored at t = len_b instead of 0
        assert lens[b] == t
        G, Cs, Hs = tape[layer]
        o = G[b, t].view(H, 4)[:, 3].double()
        Hs[b, t] = (o * torch.tanh(Cs[b, t].double())).to(torch.bfloat16)
    rep = S.check_tape(tape, x, lens, ws)
    print(name, rep.failing(), rep.first_failure())
    assert not rep.ok, f"{name} was not caught:\n{rep.summary()}"
    q, where = rep.first_failure()
    assert (where.layer, where.t) == (layer, t), (name, str(where))
    if b is not None:
        assert where.b == b, (name, str(where))
    if block is not None:
        assert where.block == block and rep.stats[q].worst.block == block, (name, str(where))
    assert q == quantity, (name, q)


@pytest.mark.parametrize("layers,hidden,Bt,Tt", [(1, 64, 1, 1), (2, 1024, 256, 317), (3, 128, 130, 7),
                                                 (2, 1088, 3, 5), (8, 64, 257, 33)])
def test_tape_layout_matches_tape_bytes(layers, hidden, Bt, Tt):
    n = (C.c_int64 * (3 * layers))()
    L.check(L.lib().avvad_lstm_tape_layout(layers, hidden, Bt, Tt, n, 3 * layers))
    off = list(n)
    sizes = [Bt * Tt * 4 * hidden * 2, Bt * Tt * hidden * 4, Bt * Tt * hidden * 2] * layers
    total = L.lib().avvad_lstm_tape_bytes(layers, hidden, Bt, Tt)
    assert off[0] == 0
    for k in range(3 * layers):
        assert off[k] % 256 == 0
        end = off[k] + sizes[k]
        assert end <= (off[k + 1] if k + 1 < 3 * layers else total)
        if k + 1 < 3 * layers:
            assert off[k + 1] - end < 256   # regions are packed, only the 256-byte alignment in between
    assert total - (off[-1] + sizes[-1]) < 512
    # the views the tests read the tape through
    lstm = types.SimpleNamespace(hidden=hidden, layers=layers)
    if Bt * Tt * hidden * layers <= 1 << 22:
        tape = torch.zeros(total, dtype=torch.uint8)
        views = E.lstm_tape_views(lstm, tape, Bt, Tt)
        assert len(views) == layers
        for l, (g, c, h) in enumerate(views):
            assert g.shape == (Bt, Tt, 4 * hidden) and g.dtype == torch.bfloat16
            assert c.shape == (Bt, Tt, hidden) and c.dtype == torch.float32
            assert h.shape == (Bt, Tt, hidden) and h.dtype == torch.bfloat16
            g.fill_(1.0), c.fill_(2.0), h.fill_(3.0)
        for l, (g, c, h) in enumerate(views):   # no view overlaps another
            assert bool((g == 1.0).all() and (c == 2.0).all() and (h == 3.0).all())


def test_tape_layout_rejects_bad_arguments():
    n = (C.c_int64 * 6)()
    assert L.lib().avvad_lstm_tape_layout(2, 1024, 4, 4, n, 5) != 0
    assert b"3 entries per layer" in L.lib().avvad_last_error()
    assert L.lib().avvad_lstm_tape_layout(0, 1024, 4, 4, n, 0) != 0
