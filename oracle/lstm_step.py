"""Teacher-forced float64 reference of the LSTM recurrence, an ideal-kernel emulator and a checker for the training tape.

The training forward keeps, per layer and step (b, t), the post-activation gates (bf16, gate-interleaved 4u+g), the cell
state c_t (f32) and the output h_t (bf16, exactly 0 for t >= len_b) -- ``avvad.engine.lstm_tape_views``.  Given the
h_{t-1} and c_{t-1} the kernel actually used (the tape's own step t-1), one step can be recomputed in float64 and compared
with what the kernel wrote.  Every step is then checked on its own: the error does not build up over T, so the bounds
are element-wise and tight, and a failure names the layer, step, batch row and 64-unit block where it starts.

Kernel semantics this restates (csrc/lstm_persist.cuh, csrc/lstm_pair.cuh):
  * operands: X (bf16) and h_{t-1} as stored (bf16), weights rounded to bf16 (round to nearest even, as
    pack_lstm_w_kernel does), bias b_ih + b_hh; gates i, f, g, o; c_t = f c_{t-1} + i g; h_t = o tanh(c_t);
  * past the length (t >= len_b) h_t is stored as 0 and the recurrence goes on from that stored 0, with c still
    updated; the gates and c of those steps are not part of the contract (BPTT never reads them) and are not checked;
  * layer l+1 reads layer l's stored h sequence.

Error bounds (absolute unless stated; every term is a property of the kernel's arithmetic):
  * bf16 storage of a gate or of h (|value| < 1): half an ulp, 2^-9;
  * tanh.approx.f32: relative error about 2^-11, so at most 2^-11 on tanh (g, and tanh(c) in h); the sigmoid is
    0.5 tanh(x / 2) + 0.5, which halves it to 2^-12;
  * the pre-activation is an fp32 tensor-core sum over K = I + H <= ~2100 bf16 products (input projection + recurrent
    product, both biases folded in): worst case K 2^-24 sum|x_k w_k| (~1e-3 at these weight scales), in practice a
    random-walk sum orders of magnitude below that; its effect on a gate is scaled by sigma' <= 1/4 or tanh' <= 1.
  Which gives, in the worst case,  gates <= 2^-9 + 2^-11 + e_acc ~ 2.5e-3,  h <= 2^-9 + 2^-11 + 2^-12 + e_acc ~ 2.7e-3
  and |c_t - c_ref| <= (2^-12 + e_acc)|c_{t-1}| + 2^-12 + 2^-11 + e_acc  ~ 1e-3 (1 + |c_{t-1}|).
  The signed mean error of a gate type over N entries: bf16 rounding to nearest even is unbiased, so it is noise of
  order (max error) / sqrt(N) plus whatever systematic bias the hardware tanh carries.

Measured (NVIDIA B200 at its 1000 W limit, the 22 cases of tests/test_gpu_lstm_state.py, H = 64..1024, up to B = 2100
and T = 317): gates 1.960e-3 and h 1.960e-3 (the bf16 half ulp 1.953e-3 dominates both), c 9.8e-6 relative (the
hardware tanh and the fp32 sums are far better than their worst case on these arguments), signed gate means at most
2.6e-6 once N >= 1e6 (sigmoid gates consistently about -1.5e-6: a small bias of tanh.approx).  The defaults of
:class:`Bounds` are about twice these maxima; tests/test_lstm_step_oracle.py shows that every modelled kernel defect
fails under them.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch

GATES = ("i", "f", "g", "o")
QUANTITIES = ("gate", "c", "h", "h_pad")
Weights = Sequence[Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]]  # per layer (w_ih, w_hh, b_ih, b_hh)


def bf16_round(w: torch.Tensor) -> torch.Tensor:
    """float64 copy of `w` rounded to bf16 (round to nearest even, like __float2bfloat16_rn)."""
    return w.detach().to(torch.float32).to(torch.bfloat16).to(torch.float64)


def pack_layer(w_ih, w_hh, b_ih, b_hh, device=None):
    """(Wt [I+H][4H], bias [4H]) in float64, output column 4u+g (the tape's gate interleave), bf16-rounded weights."""
    H = w_hh.shape[1]
    W = torch.cat([bf16_round(w_ih), bf16_round(w_hh)], 1).to(device)   # [4H][I+H], PyTorch row g*H+u
    W = W.view(4, H, -1).transpose(0, 1).reshape(4 * H, -1)             # row 4u+g
    b = (b_ih.detach().double() + b_hh.detach().double()).view(4, H).t().reshape(4 * H).to(device)
    return W.t().contiguous(), b


@dataclass
class Step:
    pre: torch.Tensor    # [N][H][4] pre-activations (i, f, g, o)
    gates: torch.Tensor  # [N][H][4] sigmoid(i), sigmoid(f), tanh(g), sigmoid(o)
    c: torch.Tensor      # [N][H]
    h: torch.Tensor      # [N][H] o * tanh(c_kernel if given, else c)


def _activate(pre: torch.Tensor) -> torch.Tensor:
    return torch.stack([torch.sigmoid(pre[..., 0]), torch.sigmoid(pre[..., 1]), torch.tanh(pre[..., 2]),
                        torch.sigmoid(pre[..., 3])], -1)


def _step_packed(x, h_prev, c_prev, Wt, b, c_kernel=None) -> Step:
    N, H = h_prev.shape
    pre = torch.addmm(b, torch.cat([x.double(), h_prev.double()], 1), Wt).view(N, H, 4)
    gates = _activate(pre)
    c = gates[..., 1] * c_prev.double() + gates[..., 0] * gates[..., 2]
    h = gates[..., 3] * torch.tanh(c if c_kernel is None else c_kernel.double())
    return Step(pre, gates, c, h)


def step_reference(x_bf16, h_prev_bf16, c_prev_f32, W_ih, W_hh, b_ih, b_hh, c_kernel=None) -> Step:
    """One LSTM step in float64 for N independent rows: x [N][I], h_prev [N][H], c_prev [N][H] (any dtype, taken as
    they are), PyTorch-layout weights (rounded to bf16 here).  Runs on the device of `x`.  With `c_kernel` (the c_t
    the kernel computed) h is o * tanh(c_kernel), so an error of c is reported once, by c, and not again by h."""
    Wt, b = pack_layer(W_ih, W_hh, b_ih, b_hh, x_bf16.device)
    return _step_packed(x_bf16, h_prev_bf16, c_prev_f32, Wt, b, c_kernel)


Hook = Callable[[int, int, torch.Tensor, dict], torch.Tensor]


def emulate_tape(x: torch.Tensor, lengths: Sequence[int], weights: Weights,
                 hooks: Optional[Dict[str, Hook]] = None) -> List[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]:
    """An ideal kernel: the recurrence in float64 with the kernel's storage (gates and h bf16, c f32) and semantics
    (h_t = 0 stored for t >= len_b, the next step reads that stored 0, c keeps updating).  x [B][T][I] (bf16 values),
    on any device.  Returns per layer (gates bf16 [B][T][4H], c f32 [B][T][H], h bf16 [B][T][H]), the layout of
    ``avvad.engine.lstm_tape_views``.

    `hooks` inject defects the way a faulty kernel would make them (tests of the checker): each is called as
    hook(layer, t, value, ctx) and returns the value to use instead -- "x" (the step's layer input [B][I]), "h_prev"
    ([B][H], the stored h_{t-1}), "c_prev" ([B][H] float64) and "pre" ([B][H][4] pre-activations).  ctx holds the
    layer's input "inp", its tape so far ("h", "c", "gates") and its packed "bias" [4H] (column 4u+g)."""
    hooks = hooks or {}
    B, T, _ = x.shape
    dev = x.device
    lens = torch.as_tensor([int(v) for v in lengths], device=dev).view(B, 1)
    inp = x
    tape = []
    for l, (w_ih, w_hh, b_ih, b_hh) in enumerate(weights):
        H = w_hh.shape[1]
        Wt, b = pack_layer(w_ih, w_hh, b_ih, b_hh, dev)
        G = torch.zeros(B, T, 4 * H, dtype=torch.bfloat16, device=dev)
        Cs = torch.zeros(B, T, H, dtype=torch.float32, device=dev)
        Hs = torch.zeros(B, T, H, dtype=torch.bfloat16, device=dev)
        ctx = {"inp": inp, "h": Hs, "c": Cs, "gates": G, "bias": b}
        c = torch.zeros(B, H, dtype=torch.float64, device=dev)
        for t in range(T):
            xt = inp[:, t].double()
            hp = Hs[:, t - 1].double() if t > 0 else torch.zeros(B, H, dtype=torch.float64, device=dev)
            if "x" in hooks:
                xt = hooks["x"](l, t, xt, ctx)
            if "h_prev" in hooks:
                hp = hooks["h_prev"](l, t, hp, ctx)
            if "c_prev" in hooks:
                c = hooks["c_prev"](l, t, c, ctx)
            pre = torch.addmm(b, torch.cat([xt, hp], 1), Wt).view(B, H, 4)
            if "pre" in hooks:
                pre = hooks["pre"](l, t, pre, ctx)
            gt = _activate(pre)
            c = gt[..., 1] * c + gt[..., 0] * gt[..., 2]
            h = gt[..., 3] * torch.tanh(c)
            G[:, t] = gt.reshape(B, 4 * H).to(torch.bfloat16)
            Cs[:, t] = c.to(torch.float32)
            Hs[:, t] = torch.where(lens > t, h, torch.zeros_like(h)).to(torch.bfloat16)
        tape.append((G, Cs, Hs))
        inp = Hs
    return tape


@dataclass
class Bounds:
    gate: float = 4e-3         # |gate - ref|, every valid (layer, b, t, unit, gate); measured 1.960e-3
    c: float = 2e-5            # |c_t - ref| / (1 + |c_{t-1}|); measured 9.8e-6
    h: float = 4e-3            # |h_t - o_ref tanh(c_t)|, valid steps; measured 1.960e-3.  h_t == 0 exactly past the length
    gate_mean: float = 5e-6    # |signed mean error| of one gate type over a layer's valid entries, plus noise below;
                               # measured 2.6e-6

    def mean_bound(self, n: int) -> float:
        """The mean of n rounding errors is noise of order (max error) / sqrt(n): 2 gate / sqrt(n) on top."""
        return self.gate_mean + 2.0 * self.gate / math.sqrt(max(n, 1))


@dataclass
class Where:
    layer: int
    t: int
    b: int
    block: int   # 64-unit block of the hidden units (units 64 block .. 64 block + 63)

    def __str__(self):
        return f"(layer {self.layer}, t {self.t}, b {self.b}, units {64 * self.block}..{64 * self.block + 63})"


@dataclass
class QuantityStats:
    bound: float
    max: float = 0.0
    worst: Optional[Where] = None
    first: Optional[Where] = None   # first failing entry in (layer, t, b, block) order
    n_fail: int = 0                 # failing (layer, b, t) rows


@dataclass
class TapeReport:
    bounds: Bounds
    stats: Dict[str, QuantityStats] = field(default_factory=dict)
    mean: List[Dict[str, float]] = field(default_factory=list)       # per layer, per gate type: signed mean error
    mean_bound: List[float] = field(default_factory=list)
    pre_std: List[float] = field(default_factory=list)               # per layer, over valid steps
    saturated: List[float] = field(default_factory=list)             # fraction of gates within 1e-3 of 0 or 1

    @property
    def mean_failures(self) -> List[Tuple[int, str, float]]:
        return [(l, g, m[g]) for l, m in enumerate(self.mean) for g in GATES if not abs(m[g]) <= self.mean_bound[l]]

    @property
    def ok(self) -> bool:
        return all(s.n_fail == 0 for s in self.stats.values()) and not self.mean_failures

    def failing(self) -> List[str]:
        """Names of the checks that fail: quantities of QUANTITIES and "gate_mean"."""
        out = [q for q in QUANTITIES if self.stats[q].n_fail]
        return out + (["gate_mean"] if self.mean_failures else [])

    def first_failure(self) -> Optional[Tuple[str, Where]]:
        """The earliest failing entry over all quantities, in (layer, t, b, block) order."""
        cands = [(q, s.first) for q, s in self.stats.items() if s.first is not None]
        if not cands:
            return None
        return min(cands, key=lambda c: (c[1].layer, c[1].t, c[1].b, c[1].block, QUANTITIES.index(c[0])))

    def summary(self) -> str:
        lines = []
        for q in QUANTITIES:
            s = self.stats[q]
            lines.append(f"  {q:6s} max {s.max:.3e} (bound {s.bound:.1e})  worst {s.worst}"
                         + (f"  FAIL x{s.n_fail}, first {s.first}" if s.n_fail else ""))
        for l, m in enumerate(self.mean):
            lines.append(f"  layer {l}: signed mean " + " ".join(f"{g} {m[g]:+.2e}" for g in GATES)
                         + f" (bound {self.mean_bound[l]:.1e});  pre-activation std {self.pre_std[l]:.3f}, "
                         f"saturated gates {100 * self.saturated[l]:.2f} %")
        return "\n".join(lines)

    def message(self) -> str:
        if self.ok:
            return "tape matches the float64 step reference\n" + self.summary()
        ff = self.first_failure()
        head = f"first failure: {ff[0]} at {ff[1]}" if ff else "gate means out of bounds"
        return head + "\n" + self.summary()


def check_tape(tape, x: torch.Tensor, lengths: Sequence[int], weights: Weights, bounds: Optional[Bounds] = None,
               rows_per_block: int = 8192) -> TapeReport:
    """Teacher-forced check of a tape (per layer (gates, c, h) as from ``avvad.engine.lstm_tape_views``) against the
    float64 step reference, on the tape's device, in blocks of `rows_per_block` (b, t) rows.  x: the layer-0 input
    [B][T][I] (bf16 values, without the padding columns).  Layer l > 0 takes layer l-1's tape h as its input."""
    bounds = bounds or Bounds()
    B, T, _ = x.shape
    dev = tape[0][0].device
    lens = torch.as_tensor([int(v) for v in lengths], device=dev)
    limits = {"gate": bounds.gate, "c": bounds.c, "h": bounds.h, "h_pad": 0.0}
    rep = TapeReport(bounds, {q: QuantityStats(limits[q]) for q in QUANTITIES})
    rows = B * T
    ridx = torch.arange(rows, device=dev)
    tpos, bpos = ridx % T, ridx // T
    valid = tpos < lens[bpos]
    n_valid = int(valid.sum())
    inp = x.to(dev)
    # per (layer, row): max error over units and gates, first failing and worst 64-unit block
    for l, (w_ih, w_hh, b_ih, b_hh) in enumerate(weights):
        G, Cs, Hs = tape[l]
        H = Hs.shape[-1]
        nb = H // 64
        Wt, b = pack_layer(w_ih, w_hh, b_ih, b_hh, dev)
        Xf = (inp if l == 0 else tape[l - 1][2]).reshape(rows, -1)
        Gf, Cf, Hf = G.reshape(rows, H, 4), Cs.reshape(rows, H), Hs.reshape(rows, H)
        row_err = {q: torch.zeros(rows, dtype=torch.float64, device=dev) for q in QUANTITIES}
        row_first = {q: torch.full((rows,), -1, dtype=torch.int64, device=dev) for q in QUANTITIES}
        row_worst = {q: torch.zeros(rows, dtype=torch.int64, device=dev) for q in QUANTITIES}
        gsum = torch.zeros(4, dtype=torch.float64, device=dev)
        pre_s = torch.zeros(2, dtype=torch.float64, device=dev)
        n_sat = torch.zeros((), dtype=torch.float64, device=dev)
        for r0 in range(0, rows, rows_per_block):
            r1 = min(rows, r0 + rows_per_block)
            first = (tpos[r0:r1] == 0).view(-1, 1)
            prev = (ridx[r0:r1] - 1).clamp(min=0)
            hp = Hf[prev].double().masked_fill(first, 0.0)
            cp = Cf[prev].double().masked_fill(first, 0.0)
            st = _step_packed(Xf[r0:r1], hp, cp, Wt, b, c_kernel=Cf[r0:r1])
            v = valid[r0:r1]
            vf = v.view(-1, 1)
            dg = Gf[r0:r1].double() - st.gates                                   # [n][H][4]
            gsum += (dg * vf.view(-1, 1, 1)).sum((0, 1))
            pre_v = st.pre[v]
            pre_s += torch.stack([pre_v.sum(), (pre_v * pre_v).sum()])
            gv = Gf[r0:r1][v].double()
            n_sat += ((gv.abs() < 1e-3) | ((gv - 1).abs() < 1e-3) | ((gv + 1).abs() < 1e-3)).sum()
            errs = {
                "gate": dg.abs().amax(-1),
                "c": (Cf[r0:r1].double() - st.c).abs() / (1.0 + cp.abs()),
                "h": (Hf[r0:r1].double() - st.h).abs(),
                "h_pad": Hf[r0:r1].double().abs(),
            }
            masks = {"gate": vf, "c": vf, "h": vf, "h_pad": ~vf}
            for q, e in errs.items():
                e = torch.nan_to_num(e, nan=math.inf).masked_fill(~masks[q], 0.0)
                eb = e.view(-1, nb, 64).amax(-1)                                 # [n][blocks]
                bad = eb > rep.stats[q].bound
                row_err[q][r0:r1] = eb.amax(-1)
                row_worst[q][r0:r1] = eb.argmax(-1)
                none = torch.full((r1 - r0,), -1, dtype=torch.int64, device=dev)
                row_first[q][r0:r1] = torch.where(bad.any(-1), bad.int().argmax(-1), none)
        # per-layer summaries
        nv = n_valid * H
        rep.mean.append({g: float(gsum[k]) / max(nv, 1) for k, g in enumerate(GATES)})
        rep.mean_bound.append(bounds.mean_bound(nv))
        cnt = max(4 * nv, 1)
        mu = float(pre_s[0]) / cnt
        rep.pre_std.append(math.sqrt(max(float(pre_s[1]) / cnt - mu * mu, 0.0)))
        rep.saturated.append(float(n_sat) / cnt)
        for q in QUANTITIES:
            s = rep.stats[q]
            e = row_err[q]
            k = int(e.argmax())
            if s.worst is None or float(e[k]) > s.max:
                s.max = float(e[k])
                s.worst = Where(l, int(tpos[k]), int(bpos[k]), int(row_worst[q][k]))
            failing = row_first[q] >= 0
            nf = int(failing.sum())
            if nf and s.first is None:   # layers are visited in order: the first failing layer holds the first entry
                key = torch.where(failing, tpos * B + bpos, torch.full_like(tpos, rows))
                k = int(key.argmin())
                s.first = Where(l, int(tpos[k]), int(bpos[k]), int(row_first[q][k]))
            s.n_fail += nf
    return rep
