"""GPU: LSTM training with a carried state (avvad_lstm_forward_train_state / avvad_lstm_backward_state, engine
lstm_train_forward(state=) / lstm_train_backward(d_state=), the models' forward(hx=)).

  1. Against float64: nonzero h0 / c0 and dh_out / dc_out, ragged lengths with 0, 1 and T.  Every weight, bias and head
     gradient, dx, dh_in, dc_in, h_out and c_out against float64 autograd of the stateful reference
     (tests/lstm_state_ref.py, pinned to nn.LSTM(x, hx) on packed sequences by tests/test_lstm_train_state_oracle.py)
     on bf16-rounded weights and inputs, 3e-2 relative Frobenius per tensor and per layer (tests/test_gpu_train.py's
     bound).  Rows of length 0 pass h, c and their gradients through exactly.  Each case also checks the stateful tape
     step by step (check_tape_state: the teacher-forced float64 step check of oracle/lstm_step.py with its bounds).
     The cases hit every backward schedule: the two-layer wavefront (2B <= 128), the chunked two-stream chains (two
     layers, larger B; two 128-row batch slices in the forward), the per-layer loop (1 and 3 layers, and the graph-less
     loop of AVVAD_BPTT_GRAPH=0 in a subprocess), the CTA-pair (H = 1024) and one-CTA-per-block (H <= 768) forward
     kernels, y_dim = 1 and 513.
  2. Zero state equals stateless: logits, the tape (positions 1..T against 0..T-1) and dx bit-identical; weight and
     bias gradients within fp32 reordering of their K = B (T + 1) reductions.
  3. A sequence run as three chained blocks equals the whole sequence: logits bit-identical, gradients (summed over
     the blocks, state gradients handed back from block to block) within the float64 bound.
  4. Modules: eval-mode forward(hx=) is bit-identical to Lstm.forward(state=); train-mode backward through hx matches
     float64 autograd for the audio net and the AV net with MCB; a truncated-BPTT loop lowers the loss."""
import os
import subprocess
import sys

import pytest
import torch

from avvad import engine as E
from avvad import synth
from lstm_state_ref import check_tape_state, lstm_packed_hx
from oracle import lstm_step as S
from oracle import models as om
from util import lstm_test_weights

pytestmark = pytest.mark.gpu

GRAD_REL = 3e-2        # relative Frobenius error per tensor (tests/test_gpu_train.py)
REORDER_REL = 1e-5     # zero state vs stateless weight / bias gradients, fp32 reordering only; measured 1.1e-6


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _handle(layers, I, H, ws, head_w, head_b):
    lstm = E.Lstm(layers, I, H, head_w.shape[0])
    sd = {"head.weight": head_w, "head.bias": head_b}
    for l, w in enumerate(ws):
        for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), w):
            sd[f"lstm.{name}_l{l}"] = t
    lstm.load(sd, "cuda", "lstm", "head")
    return lstm


def _lengths(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(0, T + 1, (B,), generator=g).tolist()
    for i, v in enumerate([T, 0, 1, T - 1, 0, T][:B]):
        lens[i] = v
    return lens


class Case:
    def __init__(self, H, I, layers, B, T, y_dim, seed=0):
        self.H, self.I, self.layers, self.B, self.T, self.y = H, I, layers, B, T, y_dim
        self.tag = f"[H={H} I={I} layers={layers} B={B} T={T} y={y_dim}]"
        self.ws = lstm_test_weights(layers, I, H, seed)
        g = torch.Generator().manual_seed(seed + 10)
        self.head_w = (torch.rand(y_dim, H, generator=g) * 2 - 1) / H ** 0.5
        self.head_b = 0.1 * torch.randn(y_dim, generator=g)
        self.lstm = _handle(layers, I, H, self.ws, self.head_w, self.head_b)
        self.lens = _lengths(B, T, seed + 2)
        self.xs = (0.5 * torch.randn(B, T, I, generator=g)).to(torch.bfloat16).cuda()
        self.x = self.lstm.new_input(B, T, "cuda")
        self.x[..., :I] = self.xs
        self.h0 = (0.5 * torch.randn(layers, B, H, generator=g)).to(torch.bfloat16).cuda()
        self.c0 = torch.randn(layers, B, H, generator=g).cuda()
        self.G = torch.randn(B, T, y_dim, generator=g).cuda()
        self.Gh = torch.randn(layers, B, H, generator=g).cuda()
        self.Gc = torch.randn(layers, B, H, generator=g).cuda()

    def reference(self, lens=None, x=None, G=None):
        """float64 autograd of the stateful reference: (logits, h_n, c_n, grads dict)."""
        lens = self.lens if lens is None else lens
        wd = [tuple(S.bf16_round(w).cuda().requires_grad_(True) for w in lw[:2]) +
              tuple(b.double().cuda().requires_grad_(True) for b in lw[2:]) for lw in self.ws]
        hw = self.head_w.double().cuda().requires_grad_(True)
        hb = self.head_b.double().cuda().requires_grad_(True)
        xd = (self.xs if x is None else x).double().requires_grad_(True)
        h0 = self.h0.double().requires_grad_(True)
        c0 = self.c0.double().requires_grad_(True)
        out, (hn, cn) = lstm_packed_hx(xd, lens, wd, (h0, c0))
        logits = out @ hw.t() + hb
        G = self.G if G is None else G
        ((logits * G.double()).sum() + (hn * self.Gh.double()).sum() + (cn * self.Gc.double()).sum()).backward()
        grads = {"weight_ih": [w[0].grad for w in wd], "weight_hh": [w[1].grad for w in wd],
                 "bias": [w[2].grad for w in wd], "head_w": hw.grad, "head_b": hb.grad, "dx": xd.grad,
                 "dh_in": h0.grad, "dc_in": c0.grad}
        return logits.detach(), hn.detach(), cn.detach(), grads


def _compare_grads(tag, got, ref, layers, dx_cols=None):
    report = {}
    for k in ("weight_ih", "weight_hh", "bias"):
        for l in range(layers):
            report[f"{k}[{l}]"] = _rel(got[k][l], ref[k][l])
    for k in ("head_w", "head_b"):
        report[k] = _rel(got[k].view(-1), ref[k].view(-1))
    report["dx"] = _rel(got["dx"], ref["dx"] if dx_cols is None else ref["dx"][..., :dx_cols])
    for k in ("dh_in", "dc_in"):
        for l in range(layers):
            report[f"{k}[{l}]"] = _rel(got[k][l], ref[k][l])
    print(f"{tag} gradient rel_fro: " + "  ".join(f"{k} {v:.2e}" for k, v in report.items()))
    print(f"{tag} worst {max(report, key=report.get)} {max(report.values()):.3e}")
    bad = {k: v for k, v in report.items() if not v < GRAD_REL}
    assert not bad, f"{tag} {bad}"
    return report


CASES = {
    "pair-wavefront": (1024, 513, 2, 32, 64, 1),
    "pair-chunked": (1024, 513, 2, 200, 64, 1),
    "persist-wavefront-ibm": (768, 256, 2, 48, 40, 513),
    "one-layer": (256, 100, 1, 20, 30, 1),
    "three-layers-ibm": (256, 100, 3, 20, 30, 513),
}


@pytest.mark.parametrize("name", list(CASES))
def test_against_float64(name):
    c = Case(*CASES[name])
    B, T, L = c.B, c.T, c.layers
    logits, pack, (h_out, c_out) = E.lstm_train_forward(c.lstm, c.x, c.lens, state=(c.h0, c.c0))
    views = E.lstm_tape_views(c.lstm, pack, B, T + 1)
    rep = check_tape_state(views, c.xs, c.lens, c.ws, (c.h0, c.c0))
    print(f"{c.tag} stateful tape vs float64 steps: {rep}")
    assert rep["ok"], (c.tag, rep)
    g = E.lstm_train_backward(c.lstm, pack, c.G, want_dx=True, d_state=(c.Gh, c.Gc), want_state_grad=True)
    torch.cuda.synchronize()
    ref_lg, hn, cn, ref = c.reference()
    valid = torch.zeros(B, T, dtype=torch.bool, device="cuda")
    for b, n in enumerate(c.lens):
        valid[b, :n] = True
    fw = {"logits": _rel(logits[valid], ref_lg[valid])}
    for l in range(L):
        fw[f"h_out[{l}]"] = _rel(h_out[l].float(), hn[l])
        fw[f"c_out[{l}]"] = _rel(c_out[l], cn[l])
    print(f"{c.tag} forward rel_fro: " + "  ".join(f"{k} {v:.2e}" for k, v in fw.items()))
    assert all(v < GRAD_REL for v in fw.values()), (c.tag, fw)
    _compare_grads(c.tag, g, ref, L)
    zero = [b for b, n in enumerate(c.lens) if n == 0]
    assert zero
    assert torch.equal(h_out[:, zero], c.h0[:, zero]) and torch.equal(c_out[:, zero], c.c0[:, zero])
    assert torch.equal(g["dh_in"][:, zero], c.Gh[:, zero]) and torch.equal(g["dc_in"][:, zero], c.Gc[:, zero])
    assert torch.equal(g["dx"][zero], torch.zeros_like(g["dx"][zero]))


def test_against_float64_without_graphs():
    """The backward without CUDA graphs (AVVAD_BPTT_GRAPH=0 is read once per process): the wavefront and the per-layer
    loop once more in a fresh interpreter."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, AVVAD_BPTT_GRAPH="0")
    me = os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-s",
                        me + "::test_against_float64[pair-wavefront]", me + "::test_against_float64[one-layer]"],
                       cwd=os.path.dirname(here), env=env, capture_output=True, text=True, timeout=1800)
    print(r.stdout[-6000:])
    print(r.stderr[-3000:])
    assert r.returncode == 0
    assert "2 passed" in r.stdout


ZERO_CASES = {"pair-wavefront": CASES["pair-wavefront"], "pair-chunked": CASES["pair-chunked"],
              "persist-wavefront-ibm": CASES["persist-wavefront-ibm"], "three-layers-ibm": CASES["three-layers-ibm"]}


@pytest.mark.parametrize("name", list(ZERO_CASES))
def test_zero_state_equals_stateless(name):
    c = Case(*ZERO_CASES[name])
    B, T = c.B, c.T
    lg0, pack0 = E.lstm_train_forward(c.lstm, c.x, c.lens)
    lgs, packs, _ = E.lstm_train_forward(c.lstm, c.x, c.lens, state=(None, None))
    assert torch.equal(lg0, lgs), c.tag
    v0 = E.lstm_tape_views(c.lstm, pack0, B, T)
    vs = E.lstm_tape_views(c.lstm, packs, B, T + 1)
    valid = torch.zeros(B, T, dtype=torch.bool, device="cuda")
    for b, n in enumerate(c.lens):
        valid[b, :n] = True
    for l in range(c.layers):
        assert torch.equal(v0[l][2], vs[l][2][:, 1:]), (c.tag, l, "h")
        assert torch.equal(v0[l][0][valid], vs[l][0][:, 1:][valid]), (c.tag, l, "gates")
        assert torch.equal(v0[l][1][valid], vs[l][1][:, 1:][valid]), (c.tag, l, "c")
        assert torch.equal(vs[l][2][:, 0], torch.zeros_like(vs[l][2][:, 0]))
        assert torch.equal(vs[l][1][:, 0], torch.zeros_like(vs[l][1][:, 0]))
    g0 = E.lstm_train_backward(c.lstm, pack0, c.G, want_dx=True)
    gs = E.lstm_train_backward(c.lstm, packs, c.G, want_dx=True)
    assert torch.equal(g0["dx"], gs["dx"]), c.tag
    diff = {}
    for k in ("weight_ih", "weight_hh", "bias"):
        for l in range(c.layers):
            diff[f"{k}[{l}]"] = _rel(gs[k][l], g0[k][l])
    for k in ("head_w", "head_b"):
        diff[k] = _rel(gs[k], g0[k])
    print(f"{c.tag} zero state vs stateless, gradient rel_fro: " +
          "  ".join(f"{k} {v:.1e}" for k, v in diff.items()) + f"  max {max(diff.values()):.2e}")
    assert max(diff.values()) < REORDER_REL, (c.tag, diff)


def test_block_chain_equals_whole_sequence():
    c = Case(1024, 513, 2, 32, 317, 1, seed=3)
    B, T = c.B, c.T
    bounds = [0, 90, 220, 317]   # three unequal blocks
    lens = list(c.lens)
    lens[6:12] = [45, 89, 90, 91, 150, 219]   # rows that end inside the first block, and at / around the boundaries
    c.lens = lens
    lg_w, pack_w, (hw, cw) = E.lstm_train_forward(c.lstm, c.x, lens, state=(c.h0, c.c0))
    g_w = E.lstm_train_backward(c.lstm, pack_w, c.G, want_dx=True, d_state=(c.Gh, c.Gc), want_state_grad=True)
    state = (c.h0, c.c0)
    blocks = []
    for s, e in zip(bounds[:-1], bounds[1:]):
        lk = [min(max(n - s, 0), e - s) for n in lens]
        lg, pack, state = E.lstm_train_forward(c.lstm, c.x[:, s:e].contiguous(), lk, state=state)
        blocks.append((s, e, lg, pack))
    assert torch.equal(torch.cat([b[2] for b in blocks], 1), lg_w), "chained logits != whole-sequence logits"
    assert torch.equal(state[0], hw) and torch.equal(state[1], cw)
    d = (c.Gh, c.Gc)
    total = None
    dx = [None] * len(blocks)
    for k in reversed(range(len(blocks))):
        s, e, _, pack = blocks[k]
        g = E.lstm_train_backward(c.lstm, pack, c.G[:, s:e].contiguous(), want_dx=True, d_state=d,
                                  want_state_grad=True)
        d = (g["dh_in"], g["dc_in"])
        dx[k] = g["dx"]
        if total is None:
            total = {k2: ([t.clone() for t in v] if isinstance(v, list) else v.clone())
                     for k2, v in g.items() if k2 not in ("dx", "dh_in", "dc_in")}
        else:
            for k2 in total:
                if isinstance(total[k2], list):
                    for l in range(len(total[k2])):
                        total[k2][l] += g[k2][l]
                else:
                    total[k2] += g[k2]
    total.update(dx=torch.cat(dx, 1), dh_in=d[0], dc_in=d[1])
    torch.cuda.synchronize()
    _, _, _, ref = c.reference()
    rep = _compare_grads("[chain 90+130+97 vs float64]", total, ref, c.layers)
    rep_w = _compare_grads("[whole T=317 vs float64]", g_w, ref, c.layers)
    dist = {}
    for k in ("weight_ih", "weight_hh", "bias"):
        for l in range(c.layers):
            dist[f"{k}[{l}]"] = _rel(total[k][l], g_w[k][l])
    for k in ("head_w", "head_b", "dx", "dh_in", "dc_in"):
        dist[k] = _rel(total[k], g_w[k])
    print("[chain vs whole-sequence GPU gradients] rel_fro: " + "  ".join(f"{k} {v:.1e}" for k, v in dist.items()) +
          f"  max {max(dist.values()):.2e}")
    assert max(rep.values()) < GRAD_REL and max(rep_w.values()) < GRAD_REL


# ---- modules ---------------------------------------------------------------------------------------------------------
def _audio_model(sd, hidden):
    from packages.models.Audio_Net import DeepVAD_audio
    m = DeepVAD_audio(2, hidden, 1)
    m.load_state_dict(sd)
    return m.cuda()


def test_audio_eval_hx_is_lstm_forward_state():
    B, T, H = 4, 37, 1024
    sd = synth.seeded_state_dict(synth.model_spec("audio", hidden=H), seed=77)
    m = _audio_model(sd, H).eval()
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, T, 513, generator=g).cuda()
    lens = [37, 0, 20, 1]
    h0 = 0.5 * torch.randn(2, B, H, generator=g).cuda()
    c0 = torch.randn(2, B, H, generator=g).cuda()
    with torch.no_grad():
        logits, (hn, cn) = m(x, lens, hx=(h0, c0))
        eng = E.Lstm(2, 513, H, 1)
        eng.load({k: v.cuda() for k, v in sd.items()}, "cuda", "lstm_audio", "vad_audio")
        xb = eng.new_input(B, T, "cuda")
        E.pack_rows_bf16(x.reshape(B * T, 513).contiguous(), xb.view(B * T, -1), 0, False)
        st = E.LstmState(eng, B)
        st.h.copy_(h0)
        st.c.copy_(c0)
        ref, _, _, _ = eng.forward(xb, lens, state=st)
    assert torch.equal(logits, ref)
    assert torch.equal(hn, st.h.float()) and torch.equal(cn, st.c)
    with pytest.raises(ValueError):
        m(x, lens, return_posteriors=True, hx=(h0, c0))


def _lstm_weights(p, prefix, layers=2):
    return [tuple(p[f"{prefix}.{n}_l{l}"] for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))
            for l in range(layers)]


def test_audio_train_hx_gradients_match_float64():
    B, T, H = 5, 24, 1024
    sd = synth.seeded_state_dict(synth.model_spec("audio", hidden=H), seed=78)
    m = _audio_model(sd, H).train()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, T, 513, generator=g)
    lens = [24, 17, 0, 9, 1]
    h0 = (0.5 * torch.randn(2, B, H, generator=g)).cuda().requires_grad_(True)
    c0 = torch.randn(2, B, H, generator=g).cuda().requires_grad_(True)
    G = torch.randn(B, T, 1, generator=g).cuda()
    Gh = torch.randn(2, B, H, generator=g).cuda()
    Gc = torch.randn(2, B, H, generator=g).cuda()
    logits, (hn, cn) = m(x.cuda(), lens, hx=(h0, c0))
    assert logits.requires_grad and hn.requires_grad and cn.requires_grad
    ((logits * G).sum() + (hn * Gh).sum() + (cn * Gc).sum()).backward()

    p = {k: (S.bf16_round(v) if "weight_" in k and k.startswith("lstm") else v.double()).cuda().requires_grad_(True)
         for k, v in sd.items()}
    xd = x.to(torch.bfloat16).double().cuda()
    h0d = h0.detach().to(torch.bfloat16).double().requires_grad_(True)
    c0d = c0.detach().double().requires_grad_(True)
    out, (hnd, cnd) = lstm_packed_hx(xd, lens, _lstm_weights(p, "lstm_audio"), (h0d, c0d))
    lg = om.head(out, p, "vad_audio")
    ((lg * G.double()).sum() + (hnd * Gh.double()).sum() + (cnd * Gc.double()).sum()).backward()
    report = {k: _rel(q.grad, p[k].grad) for k, q in m.named_parameters()}
    report["h0"] = _rel(h0.grad, h0d.grad)
    report["c0"] = _rel(c0.grad, c0d.grad)
    print("audio net through hx, gradient rel_fro:", {k: f"{v:.2e}" for k, v in report.items()})
    assert max(report.values()) < GRAD_REL, report


def test_av_mcb_train_hx_gradients_match_autograd():
    from packages.models.AV_Net import DeepVAD_AV
    B, T, H = 3, 10, 1024
    lens = [10, 7, 4]
    g = torch.Generator().manual_seed(8)
    a = torch.randn(B, T, 513, generator=g)
    v = torch.randn(B, T, 67, 67, generator=g)
    h0 = 0.5 * torch.randn(2, B, H, generator=g)
    c0 = torch.randn(2, B, H, generator=g)
    G = torch.randn(B, T, 1, generator=g)
    Gh = torch.randn(2, B, H, generator=g)
    Gc = torch.randn(2, B, H, generator=g)
    sd = synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), seed=55)
    # reference: train-mode forward of oracle/models.py (batch-statistics BN), trainable = everything but the trunk
    p = {k: (t.clone().requires_grad_(True) if (t.is_floating_point() and not k.startswith("features.")
                                                  and "running" not in k and not k.startswith("mcb.sketch")) else t.clone())
         for k, t in sd.items()}
    feat = om.resnet18_trunk(v.reshape(B * T, 67, 67), p, training=True).view(B, T, -1)
    y = om.mcb_fusion(a, feat, p, 1e-8, True)
    h0r = h0.to(torch.bfloat16).float().requires_grad_(True)
    c0r = c0.clone().requires_grad_(True)
    out, (hnr, cnr) = lstm_packed_hx(y, lens, _lstm_weights(p, "lstm_merged"), (h0r, c0r))
    lg_ref = om.head(out, p, "vad_merged")
    ((lg_ref * G).sum() + (hnr * Gh).sum() + (cnr * Gc).sum()).backward()

    m = DeepVAD_AV(2, H, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(sd)
    for q in m.features.parameters():
        q.requires_grad = False
    m = m.cuda().train()
    h0c = h0.cuda().requires_grad_(True)
    c0c = c0.cuda().requires_grad_(True)
    logits, (hn, cn) = m(a.cuda(), v.cuda(), torch.tensor(lens).cuda(), hx=(h0c, c0c))
    ((logits * G.cuda()).sum() + (hn * Gh.cuda()).sum() + (cn * Gc.cuda()).sum()).backward()
    names = ["lstm_merged.weight_ih_l0", "lstm_merged.weight_hh_l0", "lstm_merged.bias_ih_l0",
             "lstm_merged.weight_ih_l1", "lstm_merged.weight_hh_l1", "vad_merged.weight", "mcb_bn.weight",
             "mcb_bn.bias"]
    params = dict(m.named_parameters())
    report = {k: _rel(params[k].grad, p[k].grad) for k in names}
    report["h0"] = _rel(h0c.grad, h0r.grad)
    report["c0"] = _rel(c0c.grad, c0r.grad)
    print("AV (MCB) through hx, gradient rel_fro:", {k: f"{v:.2e}" for k, v in report.items()})
    assert max(report.values()) < 6e-2, report   # tests/test_gpu_train.py's AV bound (fp32 reference, MCB + BN)


def test_audio_tbptt_loop_lowers_the_loss():
    """Long synthetic utterances trained in blocks of 100 frames with the state carried (detached) between blocks."""
    B, T, H, blk = 4, 400, 256, 100
    torch.manual_seed(0)
    sd = synth.seeded_state_dict(synth.model_spec("audio", hidden=H), seed=79)
    m = _audio_model(sd, H).train()
    g = torch.Generator().manual_seed(6)
    x = torch.randn(B, T, 513, generator=g).cuda()
    y = (torch.cumsum(x[..., :4].mean(-1), 1) > 0).float().unsqueeze(-1)   # depends on the past: the state matters
    opt = torch.optim.Adam(m.parameters(), lr=2e-3)
    losses = []
    for epoch in range(8):
        hx = (torch.zeros(2, B, H, device="cuda"), torch.zeros(2, B, H, device="cuda"))
        tot = 0.0
        for s in range(0, T, blk):
            logits, hx = m(x[:, s:s + blk].contiguous(), [blk] * B, hx=hx)
            loss, _, dl = E.batch_bce(logits, y[:, s:s + blk].contiguous(), [blk] * B, 1e-8, want_grad=True)
            opt.zero_grad()
            logits.backward(dl)
            opt.step()
            hx = (hx[0].detach(), hx[1].detach())
            tot += float(loss)
        losses.append(tot)
    print("TBPTT loss per epoch:", [round(v, 3) for v in losses])
    assert losses[-1] < 0.8 * losses[0], losses
