"""GPU parity: ResNet trunk, MCB fusion, LSTM + head and the three reference-compatible modules,
against the golden outputs of the reference's own modules (tests/golden/ref_models.npz) and the CPU
oracle.  Tolerance (BASELINE.json north_star): frame posteriors within 1e-2 absolute, bf16 vs fp32."""
import numpy as np
import pytest
import torch

from oracle import models as om
from avvad import engine as E
from avvad import synth
from util import err_stats, ref_models

pytestmark = pytest.mark.gpu
POST_TOL = 1e-2


@pytest.fixture(scope="module")
def gref():
    return ref_models()


def _sd(kind, seed, **kw):
    return synth.seeded_state_dict(synth.model_spec(kind, **kw), seed)


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def test_trunk_layer_by_layer_vs_oracle(gref):
    sd = _sd("video", 12)
    frames = torch.tensor(gref["video_x"]).view(12, 67, 67)
    _, inter = om.resnet18_trunk(frames, sd, return_intermediates=True)
    trunk = E.ResNet18Trunk()
    trunk.load(sd, "cuda")
    checks = [(0, "pool", (17, 17, 64)), (2, "l1b0", (17, 17, 64)), (4, "l1b1", (17, 17, 64)),
              (6, "l2b0", (9, 9, 128)), (9, "l2b1", (9, 9, 128)), (11, "l3b0", (5, 5, 256)),
              (14, "l3b1", (5, 5, 256)), (16, "l4b0", (3, 3, 512)), (19, "l4b1", (3, 3, 512))]
    report = {}
    for upto, name, shape in checks:
        got = trunk.forward_upto(frames.cuda(), upto, shape).float().cpu().permute(0, 3, 1, 2).numpy()
        report[name] = err_stats(got, inter[name].numpy())
    print("trunk layer errors:", {k: round(v["rel_fro"], 4) for k, v in report.items()})
    for name, st in report.items():
        assert st["rel_fro"] < 3e-2, (name, st, report)


def test_trunk_features_match_reference_module(gref):
    sd = _sd("video", 12)
    trunk = E.ResNet18Trunk()
    trunk.load(sd, "cuda")
    feat = trunk.forward(torch.tensor(gref["video_x"]).view(12, 67, 67).cuda()).cpu().numpy()
    st = err_stats(feat, gref["video_feat"])
    assert st["rel_fro"] < 2e-2, st


def test_trunk_chunking_is_invisible():
    sd = _sd("video", 3)
    trunk = E.ResNet18Trunk()
    trunk.load(sd, "cuda")
    frames = torch.randn(37, 67, 67, generator=torch.Generator().manual_seed(0)).cuda()
    a = trunk.forward(frames)
    trunk.chunk = 8
    b = trunk.forward(frames)
    assert torch.equal(a, b)


def test_audio_module_matches_reference(gref):
    from packages.models.Audio_Net import DeepVAD_audio
    m = synth.fill_module_(DeepVAD_audio(2, 1024, 1), seed=11).cuda().eval()
    with torch.no_grad():
        logits, post, dec = m(torch.tensor(gref["audio_x"]).cuda(), gref["audio_len"].tolist(), return_posteriors=True)
    ref = gref["audio_out"]
    st = err_stats(_sigmoid(logits.cpu().numpy()), _sigmoid(ref))
    assert st["max"] < POST_TOL, st
    assert np.allclose(post.cpu().numpy(), _sigmoid(logits.cpu().numpy()), atol=1e-6)
    assert np.array_equal(dec.cpu().numpy(), (post.cpu().numpy() > 0.5).astype(np.int32))
    # padded steps: exactly the head bias
    bias = m.vad_audio.bias.item()
    assert np.all(logits.cpu().numpy()[2, 7:, 0] == np.float32(bias))


def test_audio_module_lengths_as_cuda_and_cpu_tensor(gref):
    from packages.models.Audio_Net import DeepVAD_audio
    m = synth.fill_module_(DeepVAD_audio(2, 1024, 1), seed=11).cuda().eval()
    x = torch.tensor(gref["audio_x"]).cuda()
    a = m(x, gref["audio_len"].tolist())
    b = m(x, torch.tensor(gref["audio_len"]))
    c = m(x, torch.tensor(gref["audio_len"]).cuda())
    assert torch.equal(a, b) and torch.equal(a, c)


def test_video_module_matches_reference(gref):
    from packages.models.Video_Net import DeepVAD_video
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=12).cuda().eval()
    x = torch.tensor(gref["video_x"]).cuda()
    out = m(x, gref["video_len"].tolist()).cpu().numpy()
    st = err_stats(_sigmoid(out), _sigmoid(gref["video_out"]))
    assert st["max"] < POST_TOL, st
    last = m(x, torch.tensor(gref["video_len"]), return_last=True).cpu().numpy()
    st = err_stats(_sigmoid(last), _sigmoid(gref["video_out_last"]))
    assert st["max"] < POST_TOL, st


@pytest.mark.parametrize("y_dim,seed,key", [(1, 13, "av_out"), (513, 14, "av513_out")])
def test_av_concat_module_matches_reference(gref, y_dim, seed, key):
    from packages.models.AV_Net import DeepVAD_AV
    m = synth.fill_module_(DeepVAD_AV(2, 1024, y_dim, use_mcb=False, eps=1e-8), seed=seed).cuda().eval()
    out = m(torch.tensor(gref["av_audio"]).cuda(), torch.tensor(gref["av_video"]).cuda(), gref["av_len"].tolist())
    st = err_stats(_sigmoid(out.cpu().numpy()), _sigmoid(gref[key]))
    assert st["max"] < POST_TOL, st


def _mcb_sd(seed, rows):
    sd = _sd("av", seed, use_mcb=True)
    # calibrate the BN running statistics to the scale the whole-tensor L2 norm produces
    sd["mcb_bn.running_mean"] = torch.zeros(1024)
    sd["mcb_bn.running_var"] = torch.full((1024,), 1.0 / (rows * 1024.0))
    return sd


def test_mcb_fusion_matches_oracle():
    rows = 24
    sd = _mcb_sd(21, rows)
    g = torch.Generator().manual_seed(3)
    a = torch.randn(2, 12, 513, generator=g)
    v = torch.randn(2, 12, 512, generator=g).abs()
    ref = om.mcb_fusion(a, v, sd, eps=1e-8).numpy().reshape(rows, 1024)
    mcb = E.Mcb()
    mcb.load(sd, "cuda", 1e-8)
    out = torch.empty(rows, 1024, device="cuda")
    outb = torch.zeros(rows, 1024, dtype=torch.bfloat16, device="cuda")
    mcb.forward(a.cuda(), v.cuda(), out_bf16=outb, out_f32=out)
    st = err_stats(out.cpu().numpy(), ref)
    assert st["max"] < 2e-3 * st["ref_absmax"], st
    assert err_stats(outb.float().cpu().numpy(), ref)["rel_fro"] < 5e-3


def test_av_mcb_module_matches_oracle(gref):
    from packages.models.AV_Net import DeepVAD_AV
    B, T = 2, 6
    sd = _mcb_sd(22, B * T)
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    a, v, lens = torch.tensor(gref["av_audio"]), torch.tensor(gref["av_video"]), gref["av_len"].tolist()
    ref = om.deepvad_av_forward(a, v, lens, sd, use_mcb=True, eps=1e-8).numpy()
    out = m(a.cuda(), v.cuda(), lens).cpu().numpy()
    st = err_stats(_sigmoid(out), _sigmoid(ref))
    assert st["max"] < POST_TOL, st


def test_av_larger_batch_decisions_agree_with_oracle():
    """B=6 ragged utterances, T up to 40, strong weight family: logits within 2e-2 relative, posteriors within 1e-2 and
    >= 99.9 % identical decisions over ALL valid frames."""
    from packages.models.AV_Net import DeepVAD_AV
    from util import check_logits
    B, T = 6, 40
    lens = [40, 33, 40, 17, 25, 9]
    sd = synth.seeded_state_dict(synth.model_spec("av"), 31, "strong")
    g = torch.Generator().manual_seed(9)
    a = torch.randn(B, T, 513, generator=g)
    v = torch.randn(B, T, 67, 67, generator=g)
    ref0 = om.deepvad_av_forward(a, v, lens, sd).numpy()
    nb = synth.decision_bias(ref0, lens, sd["vad_merged.bias"].numpy())
    ref = ref0 - sd["vad_merged.bias"].numpy() + nb.numpy()
    sd["vad_merged.bias"] = nb
    m = DeepVAD_AV(2, 1024, 1, use_mcb=False)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    logits, post, dec = m(a.cuda(), v.cuda(), torch.tensor(lens).cuda(), return_posteriors=True)
    check_logits(logits.cpu().numpy(), ref, lens, "AV concat B=6 ragged")
    assert np.array_equal(dec.cpu().numpy(), (post.cpu().numpy() > 0.5).astype(np.int32))


def _stem_reference(frames, sd):
    """fp32 torch: conv1 (3 identical channels) + BN(eval) + ReLU + maxpool, on bf16-rounded inputs."""
    import torch.nn.functional as F
    x = frames.to(torch.bfloat16).float()[:, None].repeat(1, 3, 1, 1)
    y = F.conv2d(x, sd["features.0.weight"], stride=2, padding=3)
    y = F.batch_norm(y, sd["features.1.running_mean"], sd["features.1.running_var"], sd["features.1.weight"],
                     sd["features.1.bias"], training=False, eps=1e-5)
    return F.max_pool2d(torch.relu(y), 3, 2, 1)


@pytest.mark.parametrize("n", [1, 2, 3, 37, 301])
def test_stem_image_as_operand_matches_fp32(n):
    """Every output pixel of the stem (incl. the edge tile's pooled column 16, odd batch tails and both frames of a
    batch) against fp32 conv+BN+ReLU+maxpool."""
    sd = _sd("video", 5)
    g = torch.Generator().manual_seed(n)
    frames = torch.randn(n, 67, 67, generator=g)
    ref = _stem_reference(frames, sd).permute(0, 2, 3, 1).numpy()
    trunk = E.ResNet18Trunk()
    trunk.load(sd, "cuda")
    got = trunk.forward_upto(frames.cuda(), 0, (17, 17, 64)).float().cpu().numpy()
    st = err_stats(got, ref)
    assert st["rel_fro"] < 8e-3, st
    assert st["max"] < 3e-2 * max(1.0, st["ref_absmax"]), st
    # per pooled column: a wrong anchor / shift mapping shows up as one bad column, not as noise
    col_err = np.abs(got - ref).max(axis=(0, 1, 3))
    assert col_err.max() < 3e-2 * max(1.0, st["ref_absmax"]), col_err


def test_trunk_from_u8_source_equals_gather_then_trunk():
    """avvad_resnet18_forward_u8 (gather + standardise + padding inside the stem) is bit-identical to
    avvad_upsample_gather followed by avvad_resnet18_forward, ragged lengths and chunking included."""
    sd = _sd("video", 9)
    trunk = E.ResNet18Trunk()
    trunk.load(sd, "cuda")
    B, F = 5, 23
    n_src = [23, 17, 1, 20, 0]
    t_max = 50
    n_out = [48, 35, 2, 50, 0]
    g = torch.Generator().manual_seed(3)
    src = torch.randint(0, 256, (B, F, 67, 67), generator=g, dtype=torch.uint8).cuda()
    frames = E.upsample_gather(src, n_src, n_out, t_max, synth.VIDEO_MEAN, synth.VIDEO_STD, 1e-8, True)
    for chunk in (2048, 64, 7):
        trunk.chunk = chunk
        a = trunk.forward(frames.view(B * t_max, 67, 67))
        b = trunk.forward_u8(src, n_src, n_out, t_max, synth.VIDEO_MEAN, synth.VIDEO_STD, 1e-8, True)
        assert torch.equal(a, b), (chunk, (a - b).abs().max().item())
