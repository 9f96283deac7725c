"""CPU: the float64 stateful LSTM reference the stateful training tests use (tests/lstm_state_ref.py).
  * at zero state it is oracle.models.lstm_packed;
  * with a state it is nn.LSTM(x, hx) on packed sequences (outputs, h_n, c_n and every gradient, h0 and c0 included);
  * two blocks with the state carried equal one call;
  * emulate_tape_state passes check_tape_state, which rejects it when given another state."""
import torch
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

from lstm_state_ref import check_tape_state, emulate_tape_state, lstm_packed_hx
from oracle import lstm_step as S
from oracle import models as om
from util import lstm_test_weights

B, T, I, H, LAYERS = 5, 9, 12, 64, 2
LENS = [9, 0, 1, 5, 9]


def _setup(seed=0):
    g = torch.Generator().manual_seed(seed)
    ws = [tuple(w.double() for w in lw) for lw in lstm_test_weights(LAYERS, I, H, seed)]
    x = 0.5 * torch.randn(B, T, I, generator=g, dtype=torch.float64)
    h0 = 0.5 * torch.randn(LAYERS, B, H, generator=g, dtype=torch.float64)
    c0 = torch.randn(LAYERS, B, H, generator=g, dtype=torch.float64)
    return ws, x, h0, c0


def _sd(ws):
    sd = {}
    for l, w in enumerate(ws):
        for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), w):
            sd[f"lstm.{name}_l{l}"] = t
    return sd


def test_zero_state_is_the_stateless_oracle():
    ws, x, _, _ = _setup()
    out, (h_n, _) = lstm_packed_hx(x, LENS, ws)
    ref, last = om.lstm_packed(x, LENS, _sd(ws), "lstm", LAYERS, return_state=True)
    assert torch.equal(out, ref)
    assert torch.equal(h_n[-1], last)


def test_matches_nn_lstm_with_hx_and_its_gradients():
    ws, x, h0, c0 = _setup(1)
    g = torch.Generator().manual_seed(5)
    G = torch.randn(B, T, H, generator=g, dtype=torch.float64)
    Gh = torch.randn(LAYERS, B, H, generator=g, dtype=torch.float64)
    Gc = torch.randn(LAYERS, B, H, generator=g, dtype=torch.float64)

    def leaves():
        return [t.clone().requires_grad_(True) for t in (x, h0, c0)]
    x1, h1, c1 = leaves()
    ws1 = [tuple(w.clone().requires_grad_(True) for w in lw) for lw in ws]
    out, (hn, cn) = lstm_packed_hx(x1, LENS, ws1, (h1, c1))
    ((out * G).sum() + (hn * Gh).sum() + (cn * Gc).sum()).backward()

    # nn.LSTM takes rows of length >= 1 only: rows of length 0 pass their state (and its gradient) through
    keep = [b for b, n in enumerate(LENS) if n > 0]
    lstm = torch.nn.LSTM(I, H, LAYERS, batch_first=True).double()
    with torch.no_grad():
        for l, w in enumerate(ws):
            for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), w):
                getattr(lstm, f"{name}_l{l}").copy_(t)
    x2, h2, c2 = leaves()
    packed = pack_padded_sequence(x2[keep], [LENS[b] for b in keep], batch_first=True, enforce_sorted=False)
    po, (hn2, cn2) = lstm(packed, (h2[:, keep], c2[:, keep]))
    out2, _ = pad_packed_sequence(po, batch_first=True, total_length=T)
    ((out2 * G[keep]).sum() + (hn2 * Gh[:, keep]).sum() + (cn2 * Gc[:, keep]).sum()).backward()

    tol = dict(rtol=1e-10, atol=1e-12)
    assert torch.allclose(out[keep], out2, **tol)
    assert torch.allclose(hn[:, keep], hn2, **tol) and torch.allclose(cn[:, keep], cn2, **tol)
    drop = [b for b in range(B) if b not in keep]
    assert torch.equal(hn[:, drop], h0[:, drop]) and torch.equal(cn[:, drop], c0[:, drop])
    assert torch.equal(out[drop], torch.zeros_like(out[drop]))
    assert torch.allclose(x1.grad[keep], x2.grad[keep], **tol)
    assert torch.allclose(h1.grad[:, keep], h2.grad[:, keep], **tol)
    assert torch.allclose(c1.grad[:, keep], c2.grad[:, keep], **tol)
    assert torch.equal(h1.grad[:, drop], Gh[:, drop]) and torch.equal(c1.grad[:, drop], Gc[:, drop])
    for l, lw in enumerate(ws1):
        for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), lw):
            assert torch.allclose(t.grad, getattr(lstm, f"{name}_l{l}").grad, **tol), (l, name)


def test_two_blocks_with_the_state_carried_equal_one_call():
    ws, x, h0, c0 = _setup(2)
    out, (hn, cn) = lstm_packed_hx(x, LENS, ws, (h0, c0))
    t1 = 4
    la = [min(n, t1) for n in LENS]
    lb = [max(n - t1, 0) for n in LENS]
    oa, sa = lstm_packed_hx(x[:, :t1], la, ws, (h0, c0))
    ob, sb = lstm_packed_hx(x[:, t1:], lb, ws, sa)
    tol = dict(rtol=1e-12, atol=1e-14)
    assert torch.allclose(torch.cat([oa, ob], 1), out, **tol)
    assert torch.allclose(sb[0], hn, **tol) and torch.allclose(sb[1], cn, **tol)


def test_emulated_stateful_tape_passes_the_check_and_a_wrong_state_fails_it():
    ws, x, h0, c0 = _setup(3)
    xb = x.float().to(torch.bfloat16)
    state = (h0.float().to(torch.bfloat16), c0.float())
    ws32 = [tuple(w.float() for w in lw) for lw in ws]
    tape = emulate_tape_state(xb, LENS, ws32, state)
    assert tape[0][0].shape == (B, T + 1, 4 * H)
    rep = check_tape_state(tape, xb, LENS, ws32, state)
    print("emulated stateful tape:", rep)
    assert rep["ok"], rep
    # the same tape checked against a state it was not computed from
    wrong_c = (state[0], state[1] + 0.25)
    rep = check_tape_state(tape, xb, LENS, ws32, wrong_c)
    assert not rep["ok"] and rep["state"] > 0 and rep["c"] > S.Bounds().c, rep
    wrong_h = ((h0 * 0.5).float().to(torch.bfloat16), state[1])
    rep = check_tape_state(tape, xb, LENS, ws32, wrong_h)
    assert not rep["ok"] and rep["state"] > 0 and rep["gate"] > S.Bounds().gate, rep
    # and a tape emulated from a zero state fails against the nonzero one
    zero = (torch.zeros_like(state[0]), torch.zeros_like(state[1]))
    tape0 = emulate_tape_state(xb, LENS, ws32, zero)
    assert check_tape_state(tape0, xb, LENS, ws32, zero)["ok"]
    rep = check_tape_state(tape0, xb, LENS, ws32, state)
    assert not rep["ok"], rep

