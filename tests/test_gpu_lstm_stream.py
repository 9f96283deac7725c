"""GPU: the LSTM recurrence run in blocks with its state carried (avvad_lstm_forward_state, engine.LstmState).

Every case runs ragged sequences through one stateless call on the whole sequence, then through a series of stateful
calls on blocks of it, and checks
  * the identity head's logits (y_dim = H: the top layer's h) of every block against the whole-sequence call, bit for
    bit, rows past their length included;
  * after every call, h_out / c_out of every layer against the training forward's tape at step len - 1 of the whole
    sequence, bit for bit (the per-step GEMM fallback has no training forward: there the reference is one stateful call
    on the whole prefix);
  * that separate output buffers give the same state as the in-place update the engine does.
Blocks include a single step, blocks shorter and longer than one chunk of the two-layer overlap (csrc/lstm.cu: 16 steps
per chunk), rows with no step in a block, and one row reset in the middle of the run to start a new sequence.  Shapes
cover every recurrence path: the CTA-pair kernel at H = 1024 (one and two batch slices), H = 832 (an odd number of K
blocks), the one-CTA-per-block persist kernel at H = 256 and 768 over two batch groups, 1, 2 and 3 layers, padded input
widths, and the per-step GEMM fallback at H = 1088."""
import pytest
import torch

from avvad import engine as E
from avvad import lib as L
from util import lstm_test_weights

pytestmark = pytest.mark.gpu

BLOCK_SIZES = [1, 7, 40, 2, 16, 33, 1, 64, 5]


def _handle(layers, I, H, ws):
    lstm = E.Lstm(layers, I, H, H)
    sd = {"head.weight": torch.eye(H), "head.bias": torch.zeros(H)}
    for l, w in enumerate(ws):
        for name, t in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), w):
            sd[f"lstm.{name}_l{l}"] = t
    lstm.load(sd, "cuda", "lstm", "head")
    return lstm


def _inputs(lstm, B, T, I, g):
    x = lstm.new_input(B, T, "cuda")   # columns >= I stay zero (the API contract)
    x[..., :I] = (0.5 * torch.randn(B, T, I, generator=g)).to(torch.bfloat16).cuda()
    return x


def _blocks(T):
    out, a, i = [], 0, 0
    while a < T:
        n = min(BLOCK_SIZES[i % len(BLOCK_SIZES)], T - a)
        out.append((a, a + n))
        a += n
        i += 1
    return out


class _Reference:
    """Whole-sequence results of one batch: identity-head logits and each layer's (h, c) after n steps of each row."""

    def __init__(self, lstm, x, lens, tape_ok):
        self.lstm, self.x, self.lens = lstm, x, lens
        self.logits = lstm.forward(x, lens)[0]
        self.views = None
        if tape_ok:
            B, T, _ = x.shape
            _, pack = E.lstm_train_forward(lstm, x, lens)
            self.views = [(c.clone(), h.clone()) for _, c, h in E.lstm_tape_views(lstm, pack, B, T)]
            del pack
            lstm._tape = None
            lstm._tape_busy = False

    def state(self, steps):
        """(h, c) per layer after steps[b] steps of row b: the tape at step steps[b] - 1, zero for 0 steps."""
        B = self.x.shape[0]
        n = torch.tensor(steps, device="cuda")
        at = (n - 1).clamp(min=0)
        live = (n > 0).view(B, 1)
        rows = torch.arange(B, device="cuda")
        if self.views is not None:
            hs = torch.stack([torch.where(live, h[rows, at], torch.zeros_like(h[:, 0])) for _, h in self.views])
            cs = torch.stack([torch.where(live, c[rows, at], torch.zeros_like(c[:, 0])) for c, _ in self.views])
            return hs, cs
        # fallback: one stateful call over the prefix of max(steps) steps
        Tp = max(max(steps), 1)
        st = E.LstmState(self.lstm, B)
        self.lstm.forward(self.x[:, :Tp].contiguous(), steps, state=st)
        return st.h, st.c


def _run_case(H, I, layers, B, T, tape_ok=True, seed=0):
    tag = f"[H={H} I={I} layers={layers} B={B} T={T}]"
    ws = lstm_test_weights(layers, I, H, seed)
    lstm = _handle(layers, I, H, ws)
    g = torch.Generator().manual_seed(seed + 1)
    lens = torch.randint(0, T + 1, (B,), generator=g).tolist()
    lens[0] = T
    if B > 2:
        lens[1], lens[2] = 0, 1
    blocks = _blocks(T)
    # row r0 is reset after the second block and then streams a new sequence of length len_new
    r0 = B // 2
    lens[r0] = T
    a_m = blocks[1][1]
    len_new = max(T - a_m - 3, 0)
    x = _inputs(lstm, B, T, I, g)
    x_new = _inputs(lstm, B, T, I, g)
    x_new[:, T - a_m:] = 0
    lens_new = list(lens)
    lens_new[r0] = len_new
    ref1 = _Reference(lstm, x, lens, tape_ok)
    ref2 = _Reference(lstm, x_new, lens_new, tape_ok)

    state = E.LstmState(lstm, B)
    for i, (a, b) in enumerate(blocks):
        if a == a_m:
            state.reset([r0])
        n = b - a
        xb = x[:, a:b].clone()
        lb = [min(max(v - a, 0), n) for v in lens]
        if a >= a_m:
            xb[r0] = x_new[r0, a - a_m:b - a_m]
            lb[r0] = min(max(len_new - (a - a_m), 0), n)
        xb = xb.contiguous()
        if i % 2 == 0:   # engine: in place
            logits = lstm.forward(xb, lb, state=state)[0]
        else:            # C ABI with separate output buffers
            h_out, c_out = torch.empty_like(state.h), torch.empty_like(state.c)
            wsb = torch.empty(L.lib().avvad_lstm_state_workspace_bytes(lstm.h, B, n), dtype=torch.uint8, device="cuda")
            logits = torch.empty(B, n, H, dtype=torch.float32, device="cuda")
            lt = torch.tensor(lb, dtype=torch.int32, device="cuda")
            L.check(L.lib().avvad_lstm_forward_state(lstm.h, L.ptr(xb), L.ptr(lt), B, n, L.ptr(state.h), L.ptr(state.c),
                                                     L.ptr(h_out), L.ptr(c_out), L.ptr(wsb), wsb.numel(),
                                                     L.ptr(logits), None, None, None, L.stream_ptr()))
            state.h, state.c = h_out, c_out
        want = ref1.logits[:, a:b].clone()
        if a >= a_m:
            want[r0] = ref2.logits[r0, a - a_m:b - a_m]
        same = logits == want
        assert bool(same.all()), f"{tag} block [{a}, {b}): logits differ at {int((~same).sum())} entries, first " \
                                 f"(b, t, u) {tuple(int(v) for v in (~same).nonzero()[0])}"
        hs, cs = ref1.state([min(v, b) for v in lens])
        if a >= a_m:
            h2, c2 = ref2.state([min(v, b - a_m) for v in lens_new])
            hs[:, r0], cs[:, r0] = h2[:, r0], c2[:, r0]
        for l in range(layers):
            assert torch.equal(state.h[l], hs[l]), f"{tag} block [{a}, {b}) layer {l}: h_out != reference"
            assert torch.equal(state.c[l], cs[l]), f"{tag} block [{a}, {b}) layer {l}: c_out != reference"
    print(f"{tag} {len(blocks)} blocks: logits and state bit-identical")
    del lstm, ref1, ref2
    torch.cuda.empty_cache()


@pytest.mark.parametrize("B,T", [(1, 40), (100, 70), (200, 130)], ids=["B1_T40", "B100_T70", "B200_T130"])
def test_pair_h1024(B, T):
    _run_case(1024, 1024, 2, B, T)


def test_pair_h832_odd_k_blocks():
    _run_case(832, 513, 2, 100, 50)


@pytest.mark.parametrize("H,B", [(256, 1200), (768, 400)], ids=["H256_B1200", "H768_B400"])
def test_persist_two_groups(H, B):
    _run_case(H, 513, 2, B, 40)


@pytest.mark.parametrize("layers", [1, 3])
def test_layer_counts(layers):
    _run_case(1024, 1024, layers, 150, 70)


@pytest.mark.parametrize("I", [513, 1025])
def test_input_width(I):
    _run_case(1024, I, 2, 130, 50)


def test_per_step_gemm_fallback_h1088():
    _run_case(1088, 513, 2, 130, 40, tape_ok=False)


def test_zero_state_is_the_stateless_call():
    """h_in = c_in = NULL is the zero state, and the logit outputs may be omitted when only the state is wanted."""
    H, I, B, T = 1024, 1024, 130, 50
    lstm = _handle(2, I, H, lstm_test_weights(2, I, H, 3))
    g = torch.Generator().manual_seed(4)
    x = _inputs(lstm, B, T, I, g)
    lens = torch.randint(0, T + 1, (B,), generator=g).tolist()
    st = E.LstmState(lstm, B)
    want = lstm.forward(x, lens, state=st)[0]
    assert torch.equal(want, lstm.forward(x, lens)[0])
    h_out, c_out = torch.empty_like(st.h), torch.empty_like(st.c)
    wsb = torch.empty(L.lib().avvad_lstm_state_workspace_bytes(lstm.h, B, T), dtype=torch.uint8, device="cuda")
    lt = torch.tensor(lens, dtype=torch.int32, device="cuda")
    L.check(L.lib().avvad_lstm_forward_state(lstm.h, L.ptr(x), L.ptr(lt), B, T, None, None, L.ptr(h_out), L.ptr(c_out),
                                             L.ptr(wsb), wsb.numel(), None, None, None, None, L.stream_ptr()))
    assert torch.equal(h_out, st.h) and torch.equal(c_out, st.c)
