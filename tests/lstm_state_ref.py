"""Float64 references of the LSTM with a carried state (nn.LSTM's ``hx``), for the stateful training tests.

Built on the stateless oracles, which stay as they are:
  * lstm_packed_hx   -- oracle.models.lstm_packed with an initial state, also returning (h_n, c_n) at each row's last
                        valid step (the initial state for rows of length 0), as nn.LSTM does for packed input;
  * emulate_tape_state -- oracle.lstm_step.emulate_tape started from a state (through its h_prev / c_prev hooks), laid
                        out as the stateful training tape: T + 1 positions, position 0 = the state with zero gates;
  * check_tape_state -- the teacher-forced step check of oracle.lstm_step.check_tape (same step reference, same Bounds)
                        over positions 1..T of a stateful tape, position 1 continuing from the GIVEN state, plus the
                        exact check that position 0 holds that state.
"""
from typing import Optional, Sequence

import torch

from oracle import lstm_step as S


def lstm_packed_hx(x: torch.Tensor, lengths: Sequence[int], weights, hx=None):
    """x [B][T][I]; weights per layer (w_ih, w_hh, b_ih, b_hh) in PyTorch layout; hx = (h0, c0) each [L][B][H] or None
    (zero).  Returns (out [B][T][H], exactly zero for t >= len_b, (h_n, c_n) each [L][B][H]).  Differentiable."""
    B, T, _ = x.shape
    m_all = torch.tensor([int(v) for v in lengths], device=x.device)
    inp = x
    hs, cs = [], []
    for l, (w_ih, w_hh, b_ih, b_hh) in enumerate(weights):
        H = w_hh.shape[1]
        h = hx[0][l] if hx is not None else x.new_zeros(B, H)
        c = hx[1][l] if hx is not None else x.new_zeros(B, H)
        outs = []
        for t in range(T):
            g = inp[:, t] @ w_ih.t() + h @ w_hh.t() + (b_ih + b_hh)
            i, f, gg, o = g.chunk(4, dim=1)
            c_new = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h_new = torch.sigmoid(o) * torch.tanh(c_new)
            m = (m_all > t).to(x.dtype).unsqueeze(1)
            c = m * c_new + (1 - m) * c
            h = m * h_new + (1 - m) * h
            outs.append(m * h_new)
        inp = torch.stack(outs, dim=1)
        hs.append(h)
        cs.append(c)
    return inp, (torch.stack(hs), torch.stack(cs))


def emulate_tape_state(x: torch.Tensor, lengths: Sequence[int], weights, state):
    """An ideal kernel's stateful tape: per layer (gates bf16 [B][T+1][4H], c f32 [B][T+1][H], h bf16 [B][T+1][H]) with
    position 0 = (zero gates, c0, h0).  state = (h0 bf16 values, c0 f32), each [L][B][H]."""
    h0, c0 = state
    dev = x.device
    hooks = {"h_prev": lambda l, t, v, ctx: h0[l].to(dev).double() if t == 0 else v,
             "c_prev": lambda l, t, v, ctx: c0[l].to(dev).double() if t == 0 else v}
    out = []
    for l, (G, Cs, Hs) in enumerate(S.emulate_tape(x, lengths, weights, hooks)):
        B, _, H = Hs.shape
        out.append((torch.cat([G.new_zeros(B, 1, 4 * H), G], 1),
                    torch.cat([c0[l].to(dev, torch.float32).view(B, 1, H), Cs], 1),
                    torch.cat([h0[l].to(dev, torch.bfloat16).view(B, 1, H), Hs], 1)))
    return out


def check_tape_state(tape, x: torch.Tensor, lengths: Sequence[int], weights, state,
                     bounds: Optional[S.Bounds] = None, rows_per_block: int = 8192) -> dict:
    """Maximum errors of a stateful tape (per layer (gates, c, h), T + 1 positions, as ``engine.lstm_tape_views(lstm,
    tape, B, T + 1)`` returns them): "gate", "c" (relative to 1 + |c_{t-1}|), "h" on valid steps, "h_pad" past the
    length (must be 0), "state" (position 0 against the given state and zero gates, must be 0), and "ok"."""
    bounds = bounds or S.Bounds()
    h0, c0 = state
    B, T, _ = x.shape
    dev = tape[0][0].device
    lens = torch.as_tensor([int(v) for v in lengths], device=dev)
    err = {"gate": 0.0, "c": 0.0, "h": 0.0, "h_pad": 0.0, "state": 0.0}
    inp = x.to(dev)
    bb = max(1, rows_per_block // T)
    for l, (w_ih, w_hh, b_ih, b_hh) in enumerate(weights):
        G, Cs, Hs = tape[l]
        H = Hs.shape[-1]
        Wt, b = S.pack_layer(w_ih, w_hh, b_ih, b_hh, dev)
        hl, cl = h0[l].to(dev), c0[l].to(dev)
        err["state"] = max(err["state"], float((Hs[:, 0].double() - hl.double()).abs().max()),
                           float((Cs[:, 0].double() - cl.double()).abs().max()), float(G[:, 0].double().abs().max()))
        for b0 in range(0, B, bb):
            b1 = min(B, b0 + bb)
            n = b1 - b0
            hp = Hs[b0:b1, :-1].double().clone()
            cp = Cs[b0:b1, :-1].double().clone()
            hp[:, 0] = hl[b0:b1].double()
            cp[:, 0] = cl[b0:b1].double()
            xin = (inp if l == 0 else tape[l - 1][2][:, 1:])[b0:b1].reshape(n * T, -1)
            st = S._step_packed(xin, hp.reshape(-1, H), cp.reshape(-1, H), Wt, b,
                                c_kernel=Cs[b0:b1, 1:].reshape(-1, H))
            valid = (torch.arange(T, device=dev).view(1, T) < lens[b0:b1].view(n, 1)).reshape(-1, 1)
            g = G[b0:b1, 1:].reshape(-1, H, 4).double()
            e = {"gate": (g - st.gates).abs().amax(-1),
                 "c": (Cs[b0:b1, 1:].reshape(-1, H).double() - st.c).abs() / (1.0 + cp.reshape(-1, H).abs()),
                 "h": (Hs[b0:b1, 1:].reshape(-1, H).double() - st.h).abs()}
            for q, v in e.items():
                v = torch.nan_to_num(v, nan=float("inf")).masked_fill(~valid, 0.0)
                err[q] = max(err[q], float(v.max()))
            pad = Hs[b0:b1, 1:].reshape(-1, H).double().abs().masked_fill(valid, 0.0)
            err["h_pad"] = max(err["h_pad"], float(pad.max()))
    err["ok"] = (err["gate"] <= bounds.gate and err["c"] <= bounds.c and err["h"] <= bounds.h and err["h_pad"] == 0.0
                 and err["state"] == 0.0)
    return err
