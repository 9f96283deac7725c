"""GPU: training the WaveNet encoder (csrc/wavenet_bwd.cuh).  The grad-enabled forward must be the inference forward
bit for bit, and every Conv1d weight / bias gradient and dx must match float64 autograd of the reference's `_encode`
(oracle.models.wavenet_encode).

The forward rounds its GEMM operands (x, relu(S_i), act_i, S_n and the weights) to bf16, and the gradient of a ReLU
network is discontinuous: where that rounding moves a pre-activation across zero, the exact gradient of the device's
function differs from the fp32 model's.  With these weights that alone is up to 9 % in dx and the causal weight (4 % in
the first dilated layer), whatever the backward does.  So the bound the LSTM backward uses (3e-2, relative Frobenius)
applies against float64 autograd of `bf16_encode` -- the oracle with the same operands rounded, the rounding passed
straight through by the backward -- and the plain oracle gets a sanity bound that catches a wrong gradient (sign,
layout, missing term) but not the rounding."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from avvad import synth
from oracle import models as om

pytestmark = pytest.mark.gpu

REL = 3e-2          # vs bf16_encode
REL_FP32 = 0.15     # vs the plain oracle (the fp32 model)
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_CFG = dict(k=2, q=16, dil=[1, 2, 4, 8, 1, 2, 4, 8], R=32, D=32, bott=16, pool=10, bias=True)

# (a) golden config, several time tiles + ragged last tile; (b) k = 3; (c) shift sum 127; (d) k = 1;
# (e) per-layer path (R = 128 > 64); (f1) L_final = 1 < pool; (f2) L_final % pool != 0
CONFIGS = {
    "a_golden": (GOLDEN_CFG, 3, 1000),
    "b_k3": (dict(k=3, q=16, dil=[1, 2, 4, 8, 16], R=32, D=48, bott=16, pool=9, bias=True), 2, 1500),
    "c_shift127": (dict(k=2, q=16, dil=[1, 2, 4, 8, 16, 32, 64], R=32, D=48, bott=16, pool=9, bias=True), 2, 900),
    "d_k1": (dict(k=1, q=16, dil=[1, 1], R=32, D=48, bott=16, pool=9, bias=True), 2, 300),
    "e_per_layer": (dict(k=3, q=64, dil=[1, 2, 4], R=128, D=64, bott=48, pool=7, bias=False), 2, 700),
    "f_L1_P3": (dict(k=2, q=16, dil=[1, 2], R=32, D=32, bott=16, pool=3, bias=True), 3, 5),
    "f_ragged_bins": (dict(k=2, q=16, dil=[1, 2, 4], R=32, D=32, bott=16, pool=7, bias=True), 2, 108),
}


def make(cfg, seed=16):
    from packages.models.wavenet_autoencoder import wavenet_autoencoder
    wn = wavenet_autoencoder(cfg["k"], cfg["q"], cfg["dil"], cfg["R"], cfg["D"], cfg["bott"], cfg["pool"],
                             use_bias=cfg["bias"])
    return synth.fill_module_(wn, seed=seed)


def inputs(cfg, B, N, seed=3):
    return torch.randn(B, cfg["q"], N, generator=torch.Generator().manual_seed(seed))


class _RoundBf16(torch.autograd.Function):
    """bf16 rounding in the forward, identity in the backward."""

    @staticmethod
    def forward(ctx, t):
        return t.to(torch.bfloat16).to(t.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


def bf16_encode(x, sd, dilations, pool):
    """oracle.models.wavenet_encode with every GEMM operand rounded to bf16 where the device rounds it."""
    F = torch.nn.functional
    r = _RoundBf16.apply

    def b(name):
        return sd.get(name + ".bias")

    def w(name):
        return r(sd[name + ".weight"])

    s = F.conv1d(r(x), w("en_causal_layer"), b("en_causal_layer"))
    for i, d in enumerate(dilations):
        cur = s
        a = r(F.relu(F.conv1d(r(F.relu(s)), w(f"en_dilation_layer_stack.{i}"), b(f"en_dilation_layer_stack.{i}"),
                              dilation=d)))
        s = F.conv1d(a, w(f"en_dense_layer_stack.{i}"), b(f"en_dense_layer_stack.{i}")) + cur[:, :, -a.shape[-1]:]
    s = F.relu(F.conv1d(r(s), w("bottleneck_layer"), b("bottleneck_layer")))
    return F.adaptive_avg_pool1d(s, pool)


def ref64(wn, cfg, x, dout, encode=bf16_encode):
    """(out, {param name: grad}, dx) of float64 autograd of `encode` on float64 copies."""
    sd = {k: v.detach().cpu().double().clone().requires_grad_(True) for k, v in wn.state_dict().items()}
    xd = x.detach().cpu().double().clone().requires_grad_(True)
    out = encode(xd, sd, cfg["dil"], cfg["pool"])
    out.backward(dout.cpu().double())
    return out, {k: v.grad for k, v in sd.items()}, xd.grad


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / (b.norm() + 1e-300))


def device_grads(wn, x, dout, want_dx=True):
    xg = x.cuda().requires_grad_(want_dx)
    out = wn(xg)
    out.backward(dout.cuda())
    return out, {k: p.grad for k, p in wn.named_parameters()}, xg.grad


def check_against_ref(name, got, dx, ref, ref_dx, bound=REL, what="bf16_encode"):
    errs = {k: rel(g, ref[k]) for k, g in got.items()}
    if ref_dx is not None:
        errs["dx"] = rel(dx, ref_dx)
    worst = max(errs, key=errs.get)
    print(f"[wavenet-train] {name} vs float64 {what}: worst relative Frobenius error {errs[worst]:.3e} ({worst})")
    assert errs[worst] <= bound, (name, worst, errs[worst])


def check_both(name, wn, cfg, x, dout, got, dx):
    _, ref, ref_dx = ref64(wn, cfg, x, dout)
    check_against_ref(name, got, dx, ref, ref_dx)
    _, ref, ref_dx = ref64(wn, cfg, x, dout, om.wavenet_encode)
    check_against_ref(name, got, dx, ref, ref_dx, REL_FP32, "oracle")


@pytest.mark.parametrize("name", list(CONFIGS))
def test_grad_forward_bit_identical(name):
    cfg, B, N = CONFIGS[name]
    wn = make(cfg).cuda()
    x = inputs(cfg, B, N).cuda()
    with torch.no_grad():
        ref = wn(x)
    out = wn(x)
    assert out.requires_grad
    assert torch.equal(out.detach(), ref)


@pytest.mark.parametrize("name", list(CONFIGS))
def test_gradients_vs_float64(name):
    cfg, B, N = CONFIGS[name]
    wn = make(cfg).cuda()
    x = inputs(cfg, B, N)
    with torch.no_grad():
        dout = torch.randn(wn(x.cuda()).shape, generator=torch.Generator().manual_seed(9))
    out, got, dx = device_grads(wn, x, dout)
    sd = {k: v.cpu() for k, v in wn.state_dict().items()}
    assert rel(out, om.wavenet_encode(x, sd, cfg["dil"], cfg["pool"])) < 2e-2
    assert set(got) == {k for k, _ in wn.named_parameters()}
    if not cfg["bias"]:
        assert not any(k.endswith(".bias") for k in got)
    check_both(name, wn, cfg, x, dout, got, dx)


def test_per_layer_path_gradients_vs_float64(tmp_path):
    """(g) the golden config with AVVAD_WAVENET_FUSED=0 (read once per process, hence the subprocess): within the bound
    of the float64 references, and bit-identical to the fused path's gradients (both paths write the same tape)."""
    cfg, B, N = CONFIGS["a_golden"]
    code = (
        "import sys; sys.path[:0] = [%r, %r, %r]\n"
        "import torch, numpy as np\n"
        "from test_gpu_wavenet_train import CONFIGS, make, inputs\n"
        "cfg, B, N = CONFIGS['a_golden']\n"
        "wn = make(cfg).cuda()\n"
        "x = inputs(cfg, B, N).cuda().requires_grad_(True)\n"
        "dout = torch.load(sys.argv[2])\n"
        "wn(x).backward(dout.cuda())\n"
        "g = {k: p.grad.cpu().numpy() for k, p in wn.named_parameters()}\n"
        "g['dx'] = x.grad.cpu().numpy()\n"
        "np.savez(sys.argv[1], **g)\n"
    ) % (os.path.join(REPO, "audio-visual-vad_b200"), REPO, os.path.join(REPO, "tests"))
    wn = make(cfg)
    x = inputs(cfg, B, N)
    dout = torch.randn(B, cfg["bott"], cfg["pool"], generator=torch.Generator().manual_seed(9))
    dpath, gpath = str(tmp_path / "dout.pt"), str(tmp_path / "grads.npz")
    torch.save(dout, dpath)
    subprocess.run([sys.executable, "-c", code, gpath, dpath], check=True,
                   env=dict(os.environ, AVVAD_WAVENET_FUSED="0"))
    g = dict(np.load(gpath))
    dx = torch.from_numpy(g.pop("dx"))
    check_both("g_per_layer_golden", wn, cfg, x, dout, {k: torch.from_numpy(v) for k, v in g.items()}, dx)
    _, fused, fused_dx = device_grads(make(cfg).cuda(), x, dout)
    assert set(fused) == set(g)
    for k, v in g.items():
        assert np.array_equal(fused[k].cpu().numpy(), v), k
    assert torch.equal(fused_dx.cpu(), dx)


def test_single_bin_loss_and_expanded_dout():
    cfg, B, N = CONFIGS["a_golden"]
    wn = make(cfg).cuda()
    x = inputs(cfg, B, N)
    # a loss on one pool bin of one channel
    xg = x.cuda()
    wn(xg)[1, 5, 3].backward()
    got = {k: p.grad.clone() for k, p in wn.named_parameters()}
    dout = torch.zeros(B, cfg["bott"], cfg["pool"])
    dout[1, 5, 3] = 1.0
    _, ref, _ = ref64(wn, cfg, x, dout)
    check_against_ref("single_bin", got, None, ref, None)
    # out.sum(): autograd hands over an expanded (stride-0) dout
    wn.zero_grad(set_to_none=True)
    xg = x.cuda().requires_grad_(True)
    wn(xg).sum().backward()
    check_both("sum", wn, cfg, x, torch.ones(B, cfg["bott"], cfg["pool"]),
               {k: p.grad for k, p in wn.named_parameters()}, xg.grad)


def test_dx_only_with_frozen_parameters():
    cfg, B, N = CONFIGS["b_k3"]
    wn = make(cfg).cuda()
    for p in wn.parameters():
        p.requires_grad_(False)
    x = inputs(cfg, B, N)
    xg = x.cuda().requires_grad_(True)
    out = wn(xg)
    assert out.requires_grad
    dout = torch.randn(out.shape, generator=torch.Generator().manual_seed(4))
    out.backward(dout.cuda())
    assert all(p.grad is None for p in wn.parameters())
    _, _, ref_dx = ref64(wn, cfg, x, dout)
    e = rel(xg.grad, ref_dx)
    assert e <= REL, e


def test_parameters_without_x():
    cfg, B, N = CONFIGS["a_golden"]
    wn = make(cfg).cuda()
    xg = inputs(cfg, B, N).cuda()
    wn(xg).square().mean().backward()
    assert xg.grad is None
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in wn.parameters())


def test_when_the_output_is_differentiable():
    """train() (the default): differentiable when a parameter or x requires grad.  eval(): differentiable when x
    requires grad -- gradients to x and the parameters equal train()'s bit for bit; parameters alone keep the
    inference output, with a warning.  torch.no_grad() and frozen parameters with a plain x: no graph.  The values
    are the no_grad values in every case."""
    cfg, B, N = CONFIGS["a_golden"]
    wn = make(cfg).cuda()
    x = inputs(cfg, B, N).cuda()
    with torch.no_grad():
        ref = wn(x)
    out = wn(x)
    assert wn.training and out.requires_grad and torch.equal(out.detach(), ref)

    def grads():
        wn.zero_grad(set_to_none=True)
        xg = x.clone().requires_grad_(True)
        out = wn(xg)
        assert out.requires_grad and torch.equal(out.detach(), ref)
        out.square().sum().backward()
        return [p.grad for p in wn.parameters()] + [xg.grad]

    train_grads = grads()
    wn.eval()
    for g, t in zip(grads(), train_grads):
        assert torch.equal(g, t)
    with pytest.warns(UserWarning, match="eval"):
        out = wn(x)
    assert not out.requires_grad and torch.equal(out, ref)
    with torch.no_grad():
        assert not wn(x).requires_grad
    wn.train().requires_grad_(False)
    assert not wn(x).requires_grad


def test_inplace_input_change_and_retain_graph():
    cfg, B, N = CONFIGS["a_golden"]
    wn = make(cfg).cuda()
    x = inputs(cfg, B, N).cuda()
    out = wn(x)
    x.mul_(2.0)   # the tape's copy of x would be stale: autograd's version check must refuse the backward
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        out.sum().backward()
    wn.zero_grad(set_to_none=True)
    out = wn(x)
    out.sum().backward(retain_graph=True)
    once = [p.grad.clone() for p in wn.parameters()]
    out.sum().backward()
    for p, g in zip(wn.parameters(), once):
        assert torch.equal(p.grad, g + g)
    with pytest.raises(RuntimeError, match="second time"):
        out.sum().backward()


def test_backward_deterministic_and_accumulates():
    cfg, B, N = CONFIGS["a_golden"]
    wn = make(cfg).cuda()
    x1 = inputs(cfg, B, N, seed=1).cuda().requires_grad_(True)
    x2 = inputs(cfg, B, N, seed=2).cuda().requires_grad_(True)

    def grads(x):
        wn.zero_grad(set_to_none=True)
        x.grad = None
        wn(x).square().sum().backward()
        return [p.grad.clone() for p in wn.parameters()] + [x.grad.clone()]

    a, b = grads(x1), grads(x1)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    c = grads(x2)
    # two forwards (two tapes) before one backward of the summed loss
    wn.zero_grad(set_to_none=True)
    x1.grad = x2.grad = None
    (wn(x1).square().sum() + wn(x2).square().sum()).backward()
    for p, u, v in zip(wn.parameters(), a, c):
        assert torch.equal(p.grad, u + v)
    assert torch.equal(x1.grad, a[-1]) and torch.equal(x2.grad, c[-1])


@pytest.mark.parametrize("name", ["a_golden", "e_per_layer"])
def test_adam_steps_lower_the_loss_and_repack(name):
    cfg, B, N = CONFIGS[name]
    wn = make(cfg).cuda()
    x = inputs(cfg, B, N).cuda()
    target = torch.randn(B, cfg["bott"], cfg["pool"], generator=torch.Generator().manual_seed(11)).cuda() * 0.1
    opt = torch.optim.Adam(wn.parameters(), lr=1e-3)
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = torch.nn.functional.mse_loss(wn(x), target)
        loss.backward()
        opt.step()
        losses.append(loss.item())
        # the packed device weights must follow the optimiser's in-place updates
        fresh = make(cfg).cuda()
        fresh.load_state_dict(wn.state_dict())
        with torch.no_grad():
            assert torch.equal(wn(x), fresh(x))
    assert losses[-1] < 0.8 * losses[0], losses


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_matches_single_gpu():
    cfg, B, N = CONFIGS["a_golden"]
    B = 4
    x = inputs(cfg, B, N).cuda()
    wn = make(cfg).cuda()
    wn(x).square().sum().backward()
    single = [p.grad.clone() for p in wn.parameters()]
    wn.zero_grad(set_to_none=True)
    dp = torch.nn.DataParallel(wn, device_ids=[0, 1])
    dp(x).square().sum().backward()
    for p, g in zip(wn.parameters(), single):
        assert rel(p.grad, g) < 1e-5, rel(p.grad, g)
