"""GPU parity with discriminating power (BASELINE.json north_star: posteriors within 1e-2, decisions identical on
>= 99.9 % of frames).

The default synthetic weights (PyTorch's init scale) produce logits within a few 1e-2 of the head bias, so a posterior
tolerance of 1e-2 cannot fail.  These tests use the "strong" weight family (avvad.synth.FAMILIES: logits span several
units) and assert on the LOGITS (relative Frobenius error <= 2e-2) in addition to posteriors and decisions, with NO
"unless close to 0.5" escape: decisions are compared on every valid frame.

References are outputs of the reference's own modules (tests/golden/ref_strong.npz, incl. the assembled use_mcb=True
forward executed through the legacy-FFT shim of tools/make_golden.py), and -- at the benchmarked shape B=256 x T=317 --
the CPU oracle on sampled utterances."""
import numpy as np
import pytest
import torch

from oracle import models as om
from oracle.reference_port import cpu_av_inputs
from avvad import engine as E
from avvad import synth
from avvad.pipeline import AVVADPipeline
from util import golden, ref_models, err_stats, check_logits, sigmoid as _sig, POST_TOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gs():
    return golden("ref_strong.npz")


@pytest.fixture(scope="module")
def gref():
    return ref_models()


def _with_bias(module, head, gs, key):
    """Head bias placed by synth.decision_bias at fixture time (tools/make_golden.py::ref_strong)."""
    with torch.no_grad():
        head.bias.copy_(torch.tensor(gs[key + "_bias"]))
    return module.cuda().eval()


def _long_av_inputs(gs):
    v = torch.tensor(np.random.default_rng(78).standard_normal((2, 40, 67, 67)).astype(np.float32))
    a = torch.tensor(np.random.default_rng(79).standard_normal((2, 40, 513)).astype(np.float32))
    return a, v, gs["av_long_len"].tolist()


def test_audio_strong_matches_reference_module(gs, gref):
    from packages.models.Audio_Net import DeepVAD_audio
    m = synth.fill_module_(DeepVAD_audio(2, 1024, 1), seed=41, family="strong")
    m = _with_bias(m, m.vad_audio, gs, "audio_long_out_strong")
    lens = gref["audio_len"].tolist()
    with torch.no_grad():
        out = m(torch.tensor(gref["audio_x"]).cuda(), lens).cpu().numpy()
    check_logits(out, gs["audio_out_strong"], lens, "audio B=3 T=20")
    # padded steps: exactly the head bias
    assert np.all(out[2, 7:, 0] == np.float32(m.vad_audio.bias.item()))


def test_audio_strong_long_ragged_matches_reference_module(gs):
    """317 recurrence steps, ragged: error growth through the bf16 recurrence is bounded on logits of O(1)."""
    from packages.models.Audio_Net import DeepVAD_audio
    m = synth.fill_module_(DeepVAD_audio(2, 1024, 1), seed=41, family="strong")
    m = _with_bias(m, m.vad_audio, gs, "audio_long_out_strong")
    x = torch.tensor(np.random.default_rng(77).standard_normal((4, 317, 513)).astype(np.float32))
    lens = gs["audio_long_len"].tolist()
    with torch.no_grad():
        out = m(x.cuda(), lens).cpu().numpy()
    ref = gs["audio_long_out_strong"]
    assert (ref < 0).any() and (ref > 0).any()
    check_logits(out, ref, lens, "audio B=4 T=317")


def test_video_strong_matches_reference_module(gs):
    from packages.models.Video_Net import DeepVAD_video
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=43, family="strong")
    m = _with_bias(m, m.vad_video, gs, "video_out_strong")
    _, v, lens = _long_av_inputs(gs)
    out = m(v.cuda(), lens).cpu().numpy()
    check_logits(out, gs["video_out_strong"], lens, "video B=2 T=40")


@pytest.mark.parametrize("y_dim,seed,key", [(1, 44, "av_out_strong"), (513, 45, "av513_out_strong")])
def test_av_concat_strong_matches_reference_module(gs, y_dim, seed, key):
    from packages.models.AV_Net import DeepVAD_AV
    m = synth.fill_module_(DeepVAD_AV(2, 1024, y_dim, use_mcb=False, eps=1e-8), seed=seed, family="strong")
    m = _with_bias(m, m.vad_merged, gs, key)
    a, v, lens = _long_av_inputs(gs)
    out = m(a.cuda(), v.cuda(), lens).cpu().numpy()
    if y_dim == 513:
        assert 0.4 < (gs[key] > 0).mean() < 0.6       # both decision classes, balanced
    check_logits(out, gs[key], lens, f"AV concat y_dim={y_dim}")


def test_av_mcb_strong_matches_reference_module(gs, gref):
    """The assembled use_mcb=True forward against the UNMODIFIED reference module's output."""
    from packages.models.AV_Net import DeepVAD_AV
    sd = synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 42, "strong"), 12)
    sd["vad_merged.bias"] = torch.tensor(gs["av_mcb_out_strong_bias"])
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    lens = gref["av_len"].tolist()
    out = m(torch.tensor(gref["av_audio"]).cuda(), torch.tensor(gref["av_video"]).cuda(), lens).cpu().numpy()
    check_logits(out, gs["av_mcb_out_strong"], lens, "AV MCB strong")


def test_av_mcb_default_family_matches_reference_module(gs, gref):
    """Default (PyTorch-scale) weights: logits are tiny, so the gate here is the relative error of (logit - bias)."""
    from packages.models.AV_Net import DeepVAD_AV
    sd = synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 22), 12)
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    lens = gref["av_len"].tolist()
    out = m(torch.tensor(gref["av_audio"]).cuda(), torch.tensor(gref["av_video"]).cuda(), lens).cpu().numpy()
    ref = gs["av_mcb_out_default"]
    bias = float(sd["vad_merged.bias"][0])
    mask = np.zeros(ref.shape[:2], dtype=bool)
    for b, n in enumerate(lens):
        mask[b, :n] = True
    rel = np.linalg.norm((out - ref)[mask]) / np.linalg.norm((ref - bias)[mask])
    assert rel < 3e-2, rel
    assert np.abs(_sig(out) - _sig(ref)).max() < POST_TOL


def test_standalone_mcb_matches_reference_function(gs):
    """CompactBilinearPooling as a stand-alone module (compact_bilinear_pooling.py:222-263) against the reference's own
    forward AND hand-written backward (:140-220)."""
    from packages.models.compact_bilinear_pooling import CompactBilinearPooling
    h1 = synth.seeded_tensor("mcb.sketch1.h", (513,), torch.int64, 15)
    s1 = synth.seeded_tensor("mcb.sketch1.s", (513,), torch.float32, 15)
    h2 = synth.seeded_tensor("mcb.sketch2.h", (512,), torch.int64, 15)
    s2 = synth.seeded_tensor("mcb.sketch2.s", (512,), torch.float32, 15)
    cbp = CompactBilinearPooling(513, 512, 1024, h1=h1, s1=s1, h2=h2, s2=s2).cuda()
    x = torch.tensor(gs["cbp_x"]).cuda().requires_grad_(True)
    y = torch.tensor(gs["cbp_y"]).cuda().requires_grad_(True)
    out = cbp(x, y)
    assert out.shape == (2, 5, 1024)
    st = err_stats(out.detach().cpu().numpy(), gs["cbp_out"])
    assert st["rel_fro"] < 1e-5, st
    out.backward(torch.tensor(gs["cbp_go"]).cuda())
    assert err_stats(x.grad.cpu().numpy(), gs["cbp_gx"])["rel_fro"] < 1e-4
    assert err_stats(y.grad.cpu().numpy(), gs["cbp_gy"])["rel_fro"] < 1e-4


def test_standalone_count_sketch_matches_reference_function(gref):
    """CountSketch stand-alone (compact_bilinear_pooling.py:59-113) vs the reference's CountSketchFn_forward; backward is
    the exact transpose (grad_x[i] = s_i * grad_out[h_i], :29-41)."""
    from packages.models.compact_bilinear_pooling import CountSketch
    h1 = synth.seeded_tensor("mcb.sketch1.h", (513,), torch.int64, 15)
    s1 = synth.seeded_tensor("mcb.sketch1.s", (513,), torch.float32, 15)
    cs = CountSketch(513, 1024, h1, s1).cuda()
    x = torch.tensor(gref["sketch_x"]).cuda().requires_grad_(True)
    out = cs(x)
    assert np.allclose(out.detach().cpu().numpy(), gref["sketch_out"], atol=1e-6)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(1)).cuda()
    out.backward(go)
    want = s1.cuda() * go[..., h1.cuda()]
    assert torch.equal(x.grad, want)


# ------------------------------------------------------------------------------------------------------------------
# the benchmarked shape: B = 256 utterances x T = 317 frames, use_mcb=True, raw inputs (bench.py's workload)
# ------------------------------------------------------------------------------------------------------------------
def test_benchmark_shape_pipeline_matches_oracle():
    """AVVADPipeline.infer_device at B=256 x T=317 (four 24,576-frame trunk passes, two 128-row recurrence slices x 317
    steps) against the CPU oracle on 8 sampled utterances (every trunk piece, both recurrence slices).

    The MCB branch divides by the L2 norm of the WHOLE (B,T,1024) tensor (AV_Net.py:117).  The oracle's norm is computed
    in float64 with the oracle's formula over all 81,152 rows; for the 248 utterances whose trunk features the CPU cannot
    afford to recompute (70 s of ResNet-18), the device's audio/video features are the input of that one scalar -- every
    feature error that matters shows up in the directly compared rows of the sampled utterances."""
    B, T = 256, 317
    wave, vid, mean, std = synth.batch_inputs(B, seed=1234)
    sd = synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 51, "strong"), B * T)
    ns, nf = [wave.shape[1]] * B, [vid.shape[1]] * B
    wave_d, vid_d = wave.cuda(), vid.cuda()
    pipe = AVVADPipeline(sd, mean, std, synth.VIDEO_MEAN, synth.VIDEO_STD, use_mcb=True)
    logits0 = pipe.infer_device(wave_d, ns, vid_d, nf)[0].cpu().numpy()
    audio_dev = pipe._bufs["audio"][: B * T * 513].view(B, T, 513)
    feat_dev = pipe._bufs["feat"][: B * T * 512].view(B, T, 512)

    sample = [0, 37, 63, 64, 127, 128, 200, 255]
    a_s, v_s, lens_s = cpu_av_inputs([wave[i].numpy() for i in sample], [vid[i].numpy() for i in sample], mean, std,
                                     synth.VIDEO_MEAN, synth.VIDEO_STD)
    assert lens_s == [T] * len(sample)
    torch.set_num_threads(max(1, torch.get_num_threads()))
    with torch.no_grad():
        f_s = om.resnet18_trunk(v_s.reshape(-1, 67, 67), sd).view(len(sample), T, 512)

    # (1) front end and trunk features of the sampled utterances
    st = err_stats(audio_dev[sample].cpu().numpy(), a_s.numpy())
    assert st["max"] < 2e-3, st       # log-power of near-zero bins amplifies fp32 FFT rounding; see test_gpu_frontend
    st = err_stats(feat_dev[sample].cpu().numpy(), f_s.numpy())
    print("trunk features B=256:", st)
    assert st["rel_fro"] < 2e-2, st

    # (2) whole-tensor L2 norm, float64, oracle formula (count sketch -> FFT product -> signed sqrt)
    with torch.no_grad():
        sd_dev = {k: v.cuda() for k, v in sd.items() if k.startswith("mcb.")}
        nsq = 0.0
        for r0 in range(0, B, 32):
            y = om.mcb(audio_dev[r0:r0 + 32].double(), feat_dev[r0:r0 + 32].double(),
                       {k: (v.double() if v.is_floating_point() else v) for k, v in sd_dev.items()})
            nsq += float((y.abs() + 1e-8).sum())    # |sign(y) sqrt(|y|+eps)|^2
        y_s = om.mcb(a_s, f_s, sd)
        # the sampled utterances' own contribution to the norm, oracle features vs device features, must agree as well
        y_sd = om.mcb(audio_dev[sample].cpu(), feat_dev[sample].cpu(), sd)
        assert abs(float((y_sd.abs() + 1e-8).sum()) / float((y_s.abs() + 1e-8).sum()) - 1) < 2e-3
        y_s = torch.sign(y_s) * torch.sqrt(y_s.abs() + 1e-8)
        y_s = y_s / (nsq ** 0.5)
        y_s = torch.nn.functional.batch_norm(y_s.permute(1, 2, 0).contiguous(), sd["mcb_bn.running_mean"],
                                             sd["mcb_bn.running_var"], sd["mcb_bn.weight"], sd["mcb_bn.bias"], False,
                                             0.1, 1e-8).permute(2, 0, 1).contiguous()
        # (3) LSTM + head on the sampled utterances
        ref = om.head(om.lstm_packed(y_s, lens_s, sd, "lstm_merged"), sd, "vad_merged").numpy()
    # head bias placed from the ORACLE's logits (synth.decision_bias; logits are affine in the bias), second device pass
    b0 = sd["vad_merged.bias"].clone()
    sd["vad_merged.bias"] = synth.decision_bias(ref, lens_s, b0.numpy())
    ref = ref - b0.numpy() + sd["vad_merged.bias"].numpy()
    assert (ref < 0).any() and (ref > 0).mean() > 0.9
    pipe = AVVADPipeline(sd, mean, std, synth.VIDEO_MEAN, synth.VIDEO_STD, use_mcb=True)
    logits, post, dec = pipe.infer_device(wave_d, ns, vid_d, nf)
    assert logits.shape == (B, T, 1)
    logits, post, dec = logits.cpu().numpy(), post.cpu().numpy(), dec.cpu().numpy()
    assert np.allclose(logits - logits0, float(sd["vad_merged.bias"][0] - b0[0]), atol=1e-5)
    check_logits(logits[sample], ref, lens_s, "pipeline B=256 T=317 MCB (8 sampled utterances)")
    assert np.array_equal(dec, (post > 0.5).astype(np.int32))
    assert np.allclose(post, _sig(logits), atol=1e-6)
    # every utterance saw a distinct input: no two logit rows coincide (a slice mix-up would duplicate rows)
    flat = logits[:, :, 0]
    assert len({flat[i].tobytes() for i in range(B)}) == B
