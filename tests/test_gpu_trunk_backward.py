"""GPU parity: back-propagation through the ResNet-18 trunk (csrc/resnet_bwd.cuh) -- scripts/train_video_net.py:145-173
leaves the trunk trainable and hands every parameter to Adam.

  * vs fp32 autograd of the CPU oracle on a 40-frame ragged batch: loss, logits and the gradient of EVERY parameter
    (20 conv weights, 40 BatchNorm affine parameters, LSTM, head), relative Frobenius error per tensor.  The yard-stick
    for the trunk is the oracle with `quant=bf16_ste` (fp32 autograd of the forward the device actually computes, bf16
    storage): the gradient of the PURE fp32 forward is 18-36 % away from that for every bf16 implementation (see
    oracle.models.bf16_ste), so against it only direction (cosine similarity) is asserted;
  * vs the UNMODIFIED reference module's own training step (tests/golden/ref_strong.npz: loss, gradient digests,
    running statistics of all 20 BatchNorm2d layers);
  * the concat-fusion AV model with a trainable trunk;  a full optimiser step lowers the loss."""
import numpy as np
import pytest
import torch

from oracle import models as om
from avvad import engine as E
from avvad import synth
from util import golden, ref_models, err_stats, grad_digest_of

pytestmark = pytest.mark.gpu
CONV_TOL = 3e-2       # conv / BatchNorm gradients, relative Frobenius error (bf16 operands, fp32 accumulation)


def _oracle_step(forward, sd, lens, y, trainable=lambda k: True):
    p = {k: (t.clone().requires_grad_(True) if t.is_floating_point() and "running" not in k and trainable(k) else t.clone())
         for k, t in sd.items()}
    logits = forward(p)
    loss = om.batch_loss(logits, y, lens, 1e-8)
    loss.backward()
    return logits.detach(), loss.item(), p


def _report(named_params, ref):
    rep = {}
    for k, q in named_params:
        if ref[k].grad is None:
            continue
        assert q.grad is not None, k
        rep[k] = err_stats(q.grad.cpu().numpy(), ref[k].grad.numpy())["rel_fro"]
    return rep


def test_trunk_backward_matches_the_from_tape_oracle():
    """The backward kernels in isolation: forward with a tape on the device, then the device backward against the
    textbook formulas evaluated in fp32 on THE SAME saved activations (oracle/trunk_backward.py, itself pinned against
    autograd by tests/test_oracle_trunk_backward.py).  Only the bf16 storage of the gradient activations separates them."""
    from oracle.trunk_backward import trunk_backward_from_tape
    n = 44
    g = torch.Generator().manual_seed(5)
    frames = torch.randn(n, 67, 67, generator=g)
    dfeat = torch.randn(n, 512, generator=g) * 1e-2
    sd = synth.seeded_state_dict(synth.model_spec("video"), 61, "strong")
    trunk = E.ResNet18Trunk()
    trunk.load_train(sd, "cuda")
    feat, tape = trunk.forward_tape(frames.cuda(), None)
    saved = E.ResNet18Trunk.tape_tensors(tape, n)
    saved = {k: ([t.cpu() for t in v] if isinstance(v, list) else v.cpu()) for k, v in saved.items()}
    # the tape is self-consistent: stored statistics are those of the stored raw tensors, features = mean of the last map
    raw19 = saved["raw"][19].float()
    assert torch.allclose(saved["stats"][19, :512], raw19.mean((0, 1, 2)), atol=2e-3)
    assert torch.allclose(feat.cpu(), saved["out"][7].float().mean((1, 2)), atol=1e-5)
    dw, dg, db = trunk.backward(frames.cuda(), tape, dfeat.cuda())
    ref = trunk_backward_from_tape(frames, saved, sd, dfeat)
    rep = {}
    for i, (ck, bk) in enumerate(E.RESNET_LAYER_KEYS):
        for key, got in ((ck + ".weight", dw[i]), (bk + ".weight", dg[i]), (bk + ".bias", db[i])):
            r = ref["features." + key]
            rep[key] = float((got.cpu() - r).norm() / r.norm())
    print("trunk backward vs from-tape oracle:", {k: round(e, 4) for k, e in rep.items()})
    bad = {k: e for k, e in rep.items() if e > CONV_TOL}
    assert not bad, bad


def test_video_net_trainable_trunk_gradients_match_oracle_autograd():
    from packages.models.Video_Net import DeepVAD_video
    B, T = 4, 10
    lens = [10, 8, 10, 5]
    g = torch.Generator().manual_seed(21)
    v = torch.randn(B, T, 67, 67, generator=g)
    y = (torch.rand(B, T, 1, generator=g) > 0.5).float()
    sd = synth.seeded_state_dict(synth.model_spec("video"), 61, "strong")
    ref_logits, ref_loss, p = _oracle_step(
        lambda q: om.deepvad_video_forward(v, lens, q, training=True, quant=om.bf16_ste), sd, lens, y)
    _, _, p32 = _oracle_step(lambda q: om.deepvad_video_forward(v, lens, q, training=True), sd, lens, y)
    m = DeepVAD_video(2, 1024, 1)
    m.load_state_dict(sd)
    m = m.cuda().train()
    logits = m(v.cuda(), torch.tensor(lens).cuda())
    assert logits.requires_grad
    st = err_stats(logits.detach().cpu().numpy(), ref_logits.numpy())
    assert st["rel_fro"] < 3e-2, st
    loss, _, dl = E.batch_bce(logits, y.cuda(), lens, 1e-8, want_grad=True)
    assert abs(loss.item() - ref_loss) < 2e-2 * max(1.0, abs(ref_loss)), (loss.item(), ref_loss)
    logits.backward(dl)
    rep = _report(m.named_parameters(), p)
    print("trunk gradient rel errors:", {k: round(e, 4) for k, e in rep.items()})
    assert len([k for k in rep if k.startswith("features.")]) == 60
    # LSTM / head: tight.  Trunk: the end-to-end gradient is chaotic w.r.t. rounding (the bf16_ste oracle evaluated in fp32
    # and in fp64 arithmetic differs from ITSELF by 14-25 % per conv layer, oracle/trunk_backward.py), so here only its
    # direction is asserted; the tight check of the backward kernels is the from-tape test above.
    bad = {k: e for k, e in rep.items() if not k.startswith("features.") and e > 3e-2}
    assert not bad, bad
    assert max(e for k, e in rep.items() if k.startswith("features.")) < 0.5
    # against the gradient of the pure fp32 forward: same direction (what the optimiser needs), distance reported
    cos = {k: float(torch.nn.functional.cosine_similarity(q.grad.flatten().cpu(), p32[k].grad.flatten(), dim=0))
           for k, q in m.named_parameters()}
    print("cosine vs pure-fp32 gradients: min %.3f (%s)" % (min(cos.values()), min(cos, key=cos.get)))
    assert min(cos.values()) > 0.9, {k: c for k, c in cos.items() if c <= 0.9}
    # running statistics of every BatchNorm2d layer were updated like nn.BatchNorm2d does (momentum 0.1, unbiased var)
    with torch.no_grad():
        _, inter = om.resnet18_trunk(v.reshape(-1, 67, 67), sd, training=True, return_intermediates=True)
    bn1 = m.features[1]
    assert int(bn1.num_batches_tracked) == 1
    x0 = torch.nn.functional.conv2d(v.reshape(-1, 1, 67, 67).repeat(1, 3, 1, 1), sd["features.0.weight"], None, 2, 3)
    want_mean = 0.9 * sd["features.1.running_mean"] + 0.1 * x0.mean((0, 2, 3))
    assert torch.allclose(bn1.running_mean.cpu(), want_mean, atol=2e-3)


def test_video_net_training_step_matches_reference_module_digest():
    """The reference's own DeepVAD_video training step (train(), trunk trainable, pure fp32), B=2 x T=6.  Logits, loss and
    BatchNorm running statistics are compared directly; the gradients -- which for ANY bf16 forward sit 18-36 % from the
    fp32 ones (oracle.models.bf16_ste) -- by the cosine of the reference's stored strided samples and by their norms."""
    from packages.models.Video_Net import DeepVAD_video
    gs, gref = golden("ref_strong.npz"), ref_models()
    v, lens = torch.tensor(gref["av_video"]), gref["av_len"].tolist()
    y = torch.tensor(gs["train_target"])
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=47, family="strong").cuda().train()
    logits = m(v.cuda(), torch.tensor(lens).cuda())
    st = err_stats(logits.detach().cpu().numpy(), gs["train_video_logits"])
    assert st["rel_fro"] < 5e-2, st
    loss, _, dl = E.batch_bce(logits, y.cuda(), lens, 1e-8, want_grad=True)
    assert abs(loss.item() - float(gs["train_video_loss"])) < 3e-2 * float(gs["train_video_loss"])
    logits.backward(dl)
    cos, nrm = {}, {}
    for k, q in m.named_parameters():
        norm, sample = grad_digest_of(q.grad)
        rn, rs = float(gs[f"train_video/{k}/norm"]), gs[f"train_video/{k}/sample"]
        cos[k] = float(np.dot(sample, rs) / (np.linalg.norm(sample) * np.linalg.norm(rs) + 1e-30))
        nrm[k] = norm / rn
    print("vs reference digests: min cosine %.3f (%s), norm ratio %.2f .. %.2f" % (
        min(cos.values()), min(cos, key=cos.get), min(nrm.values()), max(nrm.values())))
    assert min(cos.values()) > 0.8, {k: c for k, c in cos.items() if c <= 0.8}
    assert 0.7 < min(nrm.values()) and max(nrm.values()) < 1.4, nrm
    lstm = [c for k, c in cos.items() if not k.startswith("features.")]
    assert min(lstm) > 0.999
    for k, t in m.state_dict().items():
        if k.startswith("features.") and (k.endswith("running_mean") or k.endswith("running_var")):
            ref = gs["train_video/" + k]
            assert np.abs(t.cpu().numpy() - ref).max() < 2e-2 * max(1.0, np.abs(ref).max()), k


def test_av_concat_trainable_trunk_gradients_match_oracle_autograd():
    from packages.models.AV_Net import DeepVAD_AV
    B, T = 3, 8
    lens = [8, 5, 8]
    g = torch.Generator().manual_seed(22)
    a = torch.randn(B, T, 513, generator=g)
    v = torch.randn(B, T, 67, 67, generator=g)
    y = (torch.rand(B, T, 1, generator=g) > 0.5).float()
    sd = synth.seeded_state_dict(synth.model_spec("av"), 62, "strong")
    _, ref_loss, p = _oracle_step(lambda q: om.deepvad_av_forward(a, v, lens, q, training=True, quant=om.bf16_ste), sd,
                                  lens, y, trainable=lambda k: not k.startswith("bn."))
    m = DeepVAD_AV(2, 1024, 1, use_mcb=False)
    m.load_state_dict(sd)
    m = m.cuda().train()
    logits = m(a.cuda(), v.cuda(), torch.tensor(lens).cuda())
    loss, _, dl = E.batch_bce(logits, y.cuda(), lens, 1e-8, want_grad=True)
    assert abs(loss.item() - ref_loss) < 2e-2 * max(1.0, abs(ref_loss))
    logits.backward(dl)
    rep = _report([(k, q) for k, q in m.named_parameters() if not k.startswith("bn.")], p)
    print("AV concat, trainable trunk:", {k: round(e, 4) for k, e in rep.items() if "conv" in k or "lstm" in k})
    bad = {k: e for k, e in rep.items() if not k.startswith("features.") and e > 4e-2}
    assert not bad, bad
    assert max(e for k, e in rep.items() if k.startswith("features.")) < 0.5   # see the video-net test above


def test_av_mcb_trainable_trunk_gradients_match_oracle_autograd():
    """train_AV_net.py with `features` left trainable under MCB fusion: the LSTM's input gradient goes back through
    BatchNorm1d (batch statistics), the detached whole-tensor L2 norm, the signed sqrt and the compact-bilinear pooling
    (device FFT kernels) into the device ResNet backward."""
    from packages.models.AV_Net import DeepVAD_AV
    B, T = 3, 8
    lens = [8, 5, 8]
    g = torch.Generator().manual_seed(24)
    a = torch.randn(B, T, 513, generator=g)
    v = torch.randn(B, T, 67, 67, generator=g)
    y = (torch.rand(B, T, 1, generator=g) > 0.5).float()
    sd = synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 64, "strong")
    _, ref_loss, p = _oracle_step(
        lambda q: om.deepvad_av_forward(a, v, lens, q, use_mcb=True, training=True, quant=om.bf16_ste), sd, lens, y,
        trainable=lambda k: not k.startswith("bn.") and not k.startswith("mcb."))
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True)
    m.load_state_dict(sd)
    m = m.cuda().train()
    logits = m(a.cuda(), v.cuda(), torch.tensor(lens).cuda())
    loss, _, dl = E.batch_bce(logits, y.cuda(), lens, 1e-8, want_grad=True)
    assert abs(loss.item() - ref_loss) < 2e-2 * max(1.0, abs(ref_loss))
    logits.backward(dl)
    named = [(k, q) for k, q in m.named_parameters() if not k.startswith("bn.")]
    rep = _report(named, p)
    print("AV MCB, trainable trunk:", {k: round(e, 4) for k, e in rep.items() if "conv" in k or "lstm" in k or "mcb" in k})
    assert any(k.startswith("features.") for k in rep) and "mcb_bn.weight" in rep
    bad = {k: e for k, e in rep.items() if not k.startswith("features.") and e > 6e-2}
    assert not bad, bad
    # trunk: direction and size (the end-to-end trunk gradient is chaotic w.r.t. bf16 rounding, see the video-net test)
    cos = {}
    for k, q in named:
        if k.startswith("features.") and k.endswith("weight") and ("conv" in k or k == "features.0.weight"):
            r = p[k].grad
            cos[k] = float((q.grad.cpu().flatten() @ r.flatten()) / (q.grad.cpu().norm() * r.norm() + 1e-30))
    print("trunk gradient cosines:", {k: round(c, 3) for k, c in cos.items()})
    # Direction only.  The fusion's signed square root has the derivative 0.5 / sqrt(|m| + 1e-8): pooled values near zero
    # dominate the gradient w.r.t. the video features and differ between two FFT implementations by more than their
    # own size, so even the last trunk layer agrees with the oracle's autograd to a cosine of ~0.7 only (measured
    # 0.69-0.71 over all convolutions); the pooling backward itself is pinned against the reference's hand-written
    # backward in tests/test_gpu_strong.py, BatchNorm1d / sqrt / norm are PyTorch ops.
    assert min(cos.values()) > 0.5, cos


def test_video_net_optimiser_steps_with_torch_adam_reduce_the_loss():
    """scripts/train_video_net.py as it is written: torch.optim.Adam over model.parameters(), loss.backward()."""
    from packages.models.Video_Net import DeepVAD_video
    from packages.models.utils import binary_cross_entropy
    B, T = 2, 8
    lens = torch.tensor([8, 6])
    g = torch.Generator().manual_seed(23)
    v = torch.randn(B, T, 67, 67, generator=g).cuda()
    y = (torch.rand(B, T, 1, generator=g) > 0.5).long().cuda()
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=63).cuda()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, betas=(0.9, 0.999))
    w0 = m.features[0].weight.detach().clone()
    losses = []
    for _ in range(5):
        m.train()
        out = m(v, lens.cuda())
        loss = 0.
        for length, pred, target in zip(lens, out, y):
            loss += binary_cross_entropy(pred[:length], target[:length], 1e-8)
        loss.backward()
        opt.step()
        opt.zero_grad()
        losses.append(loss.item())
    assert losses[-1] < losses[0], losses
    assert not torch.equal(w0, m.features[0].weight.detach())      # conv1 really is being trained


def test_weight_gradient_chunking_is_invisible(tmp_path):
    """The weight-gradient GEMMs run over chunks of <= 2^19 pixels and accumulate; with AVVAD_WGRAD_PIXELS=2048 the
    44-frame test input is split into up to 7 chunks per layer (and the last one is ragged).  Both settings must give the
    same gradients (fp32 accumulation order differs only across the split-K partials)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys; sys.path[:0] = [%r, %r]\n"
        "import torch\n"
        "from avvad import engine as E, synth\n"
        "g = torch.Generator().manual_seed(5)\n"
        "frames = torch.randn(44, 67, 67, generator=g).cuda()\n"
        "dfeat = (torch.randn(44, 512, generator=g) * 1e-2).cuda()\n"
        "sd = synth.seeded_state_dict(synth.model_spec('video'), 61, 'strong')\n"
        "t = E.ResNet18Trunk(); t.load_train(sd, 'cuda')\n"
        "feat, tape = t.forward_tape(frames, None)\n"
        "dw, dg, db = t.backward(frames, tape, dfeat)\n"
        "torch.save([x.cpu() for x in dw], sys.argv[1])\n"
    ) % (os.path.join(root, "audio-visual-vad_b200"), root)
    outs = []
    for px in ("524288", "2048"):
        path = str(tmp_path / f"wgrad_{px}.pt")
        subprocess.run([sys.executable, "-c", code, path], check=True, env=dict(os.environ, AVVAD_WGRAD_PIXELS=px))
        outs.append(torch.load(path))
    for i, (a, b) in enumerate(zip(*outs)):
        rel = float((a - b).norm() / b.norm())
        assert rel < 1e-5, (i, rel)
