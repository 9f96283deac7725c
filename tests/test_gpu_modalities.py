"""GPU: the audio-only and video-only models on the raw-input entry points.

- The bf16 output mode of the register-FFT front end is bit-identical to the fp32 front end followed by
  pack_rows_bf16(zero_tail=True), and leaves the columns before col_off alone.
- AVVADPipeline(modality="audio" / "video") runs the kernels of DeepVAD_audio / DeepVAD_video, so its logits,
  posteriors and decisions are bit-identical to the modules' on the same features / frames.
- Against the CPU oracle (strong weight family, head bias placed by synth.decision_bias): the three parity gates of
  tests/util.check_logits, on ragged batches and on the golden utterance test/34M/sa1.
- The sharded evaluation returns bit-identical posteriors for any grouping of the utterances into calls."""
import numpy as np
import pytest
import torch

from avvad import engine as E
from avvad import synth
from avvad.evaluate import evaluate_shard, evaluate_sharded
from avvad.pipeline import AVVADPipeline
from oracle import frontend as ofe
from oracle import models as om
from oracle import video as ov
from util import check_logits, golden

pytestmark = pytest.mark.gpu


def _waves(B, seed, lo=3000, hi=30000):
    rng = np.random.default_rng(seed)
    ns = [int(n) for n in rng.integers(lo, hi, B)]
    ns[0] = hi                                     # one utterance that sets t_max
    wave = torch.zeros(B, hi + 777)                # wave_stride > every length
    for b, n in enumerate(ns):
        wave[b, :n] = torch.from_numpy(synth.synth_wave(n, seed + b)) if B <= 16 else 0.1 * torch.randn(n)
    return wave, ns


# ---- kernel --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 300])
@pytest.mark.parametrize("col_off,ld", [(0, 576), (0, 1088), (513, 1088)])
@pytest.mark.parametrize("normalise", [0, 1, 2])
def test_frontend_bf16_equals_fp32_then_pack(B, col_off, ld, normalise):
    torch.manual_seed(B + ld + normalise)
    wave, ns = _waves(B, 3 + normalise)
    wave = wave.cuda()
    full = [E.stft_num_frames(n) for n in ns]
    lens = [max(0, f - (b % 3) * 5) for b, f in enumerate(full)]    # trimmed below the STFT count for some rows
    t_max = max(full) + 6                                             # padding columns beyond every length
    mean, std = (torch.tensor(a).cuda() for a in synth.synth_audio_stats(0))
    peaks = (0.5 + torch.rand(B)).cuda() if normalise == 2 else None
    for stats in ((mean, std), (None, None)) if B == 1 else ((mean, std),):
        ref32 = E.frontend_logpower(wave, ns, lens, t_max, *stats, 1e-8, normalise > 0, peaks=peaks)
        sentinel = torch.randn(B * t_max, ld).to(torch.bfloat16).cuda()
        want = sentinel.clone()
        E.pack_rows_bf16(ref32.view(B * t_max, 513), want, col_off, True)
        got = sentinel.clone()
        out = E.frontend_logpower(wave, ns, lens, t_max, *stats, 1e-8, normalise > 0, peaks=peaks, out_bf16=got,
                                  col_off=col_off)
        assert out is got
        assert torch.equal(got.view(torch.int16), want.view(torch.int16)), (got != want).sum()
        assert torch.count_nonzero(got[:, col_off + 513:].float()) == 0      # the tail columns are exactly zero
        assert torch.equal(got[:, :col_off], sentinel[:, :col_off])


def test_frontend_bf16_argument_checks():
    wave, ns = _waves(2, 1)
    wave = wave.cuda()
    x = torch.zeros(2 * 10, 600, dtype=torch.bfloat16, device="cuda")
    for ld, col_off in ((600, 100), (1024, -1)):          # ld too small for col_off + 513; negative offset
        with pytest.raises(Exception):
            E.frontend_logpower(wave, ns, [10, 10], 10, None, None, out_bf16=x, ld=ld, col_off=col_off)
    with pytest.raises(Exception):                        # ld not a multiple of 8
        E.frontend_logpower(wave, ns, [10, 10], 10, None, None, out_bf16=torch.zeros(20, 514, dtype=torch.bfloat16,
                                                                                     device="cuda"))


# ---- pipeline == modules (same kernels) ----------------------------------------------------------------------------
def _video_batch(B, seed):
    nf = [12 + 9 * ((2 * b + 1) % B) for b in range(B)]   # ragged
    vid = torch.zeros(B, max(nf), 67, 67, dtype=torch.uint8)
    for b, f in enumerate(nf):
        vid[b, :f] = torch.from_numpy(synth.synth_video_u8(f, seed + b))
    return vid, nf


@pytest.mark.parametrize("y_dim", [1, 513])
def test_audio_pipeline_equals_module(y_dim):
    from packages.models.Audio_Net import DeepVAD_audio
    B = 5
    wave, ns = _waves(B, 21)
    wave = wave.cuda()
    mean, std = synth.synth_audio_stats(0)
    m = synth.fill_module_(DeepVAD_audio(2, 1024, y_dim), seed=61, family="strong").cuda().eval()
    pipe = AVVADPipeline.from_module(m, mean, std)
    assert pipe.modality == "audio" and pipe.trunk is None and pipe.lstm.ld == 576
    logits, post, dec = pipe.infer_device(wave, ns, None, None)
    lens = [E.stft_num_frames(n) for n in ns]
    assert logits.shape == (B, max(lens), y_dim)
    feat = E.frontend_logpower(wave, ns, lens, max(lens), torch.tensor(mean).cuda(), torch.tensor(std).cuda(), 1e-8,
                               True)
    with torch.no_grad():
        rl, rp, rd = m(feat, lens, return_posteriors=True)
    assert torch.equal(logits, rl) and torch.equal(post, rp) and torch.equal(dec, rd)
    # caller's lengths (the reference trims to the label length) and the host entry point
    cut = [max(1, t - 9) for t in lens]
    hp, hd = pipe.infer_host(wave.cpu().pin_memory(), ns, None, None, lengths=cut)
    feat = E.frontend_logpower(wave, ns, cut, max(cut), torch.tensor(mean).cuda(), torch.tensor(std).cuda(), 1e-8, True)
    with torch.no_grad():
        _, rp, rd = m(feat, cut, return_posteriors=True)
    assert torch.equal(hp, rp.cpu()) and torch.equal(hd, rd.cpu())


@pytest.mark.parametrize("y_dim", [1, 513])
@pytest.mark.parametrize("dedup", [False, True])
def test_video_pipeline_equals_module(y_dim, dedup):
    from packages.models.Video_Net import DeepVAD_video
    B = 5
    vid, nf = _video_batch(B, 31)
    vid = vid.cuda()
    m = synth.fill_module_(DeepVAD_video(2, 1024, y_dim), seed=62, family="strong").cuda().eval()
    pipe = AVVADPipeline.from_module(m, video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD)
    assert pipe.modality == "video" and pipe.lstm.ld == 512
    pipe.dedup_video = dedup
    pipe.piece = 2                                   # three trunk pieces
    lens = [E.upsampled_length(f) for f in nf]
    t_max = max(lens) + 3
    logits, post, dec = pipe.infer_device(None, None, vid, nf, t_max=t_max)
    frames = E.upsample_gather(vid, nf, lens, t_max, synth.VIDEO_MEAN, synth.VIDEO_STD, 1e-8, True)
    with torch.no_grad():
        rl = m(frames, lens)
    assert torch.equal(logits, rl)
    assert torch.equal(dec, (post > 0.5).int()) and torch.allclose(post, torch.sigmoid(rl), atol=1e-6)
    hp, hd = pipe.infer_host(None, None, vid.cpu().pin_memory(), nf, t_max=t_max)
    assert torch.equal(hp, post.cpu()) and torch.equal(hd, dec.cpu())
    # frames already at 62.5 fps (evaluate_video_net.py reads *_upsampled.h5): identity frame map
    up = torch.zeros(B, t_max, 67, 67, dtype=torch.uint8)
    for b in range(B):
        up[b, :lens[b]] = vid[b, E.upsample_index(nf[b], lens[b]).long()].cpu()
    pu = AVVADPipeline.from_module(m, video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD, upsampled_video=True)
    pu.dedup_video = dedup
    assert pu.lengths_of(None, lens) == lens
    lu, _, _ = pu.infer_device(None, None, up.cuda(), lens, t_max=t_max)
    assert torch.equal(lu, logits)


def test_single_modality_argument_errors():
    mean, std = synth.synth_audio_stats(0)
    pipe = AVVADPipeline(synth.seeded_state_dict(synth.model_spec("audio"), 1), mean, std, modality="audio")
    w = torch.zeros(1, 8000, device="cuda")
    with pytest.raises(ValueError, match="no MCB"):
        pipe.infer_device(w, [8000], None, None, per_utterance=True)
    with pytest.raises(ValueError, match="no MCB"):
        pipe.infer_device(w, [8000], None, None, mcb_norms_out=torch.zeros(1, device="cuda"))
    with pytest.raises(ValueError, match="video must be None"):
        pipe.infer_device(w, [8000], torch.zeros(1, 4, 67, 67, dtype=torch.uint8, device="cuda"), [4])


# ---- against the CPU oracle ----------------------------------------------------------------------------------------
def _placed(sd, head, ref0, lens):
    """Head bias from the oracle's logits (synth.decision_bias; logits are affine in the bias)."""
    nb = synth.decision_bias(ref0, lens, sd[head + ".bias"].numpy())
    ref = ref0 - sd[head + ".bias"].numpy() + nb.numpy()
    sd[head + ".bias"] = nb
    return ref


def test_audio_pipeline_matches_oracle_ragged():
    """About 1,400 valid frames, so that the >= 99.9 % decision gate tolerates one flip (a bf16 path flips about one frame
    in a thousand near the threshold)."""
    B = 6
    wave, ns = _waves(B, 41, lo=40000, hi=81920)
    mean, std = synth.synth_audio_stats(0)
    sd = synth.seeded_state_dict(synth.model_spec("audio"), 71, "strong")
    lens = [E.stft_num_frames(n) for n in ns]
    x = torch.zeros(B, max(lens), 513)
    for b, n in enumerate(ns):
        x[b, :lens[b]] = torch.from_numpy(ofe.frontend_features(wave[b, :n].numpy(), mean, std, dtype=np.float32))
    with torch.no_grad():
        ref = _placed(sd, "vad_audio", om.deepvad_audio_forward(x, lens, sd).numpy(), lens)
    pipe = AVVADPipeline(sd, mean, std, modality="audio")
    logits, _, _ = pipe.infer_device(wave.cuda(), ns, None, None)
    check_logits(logits.cpu().numpy(), ref, lens, "audio-only pipeline, ragged B=6")


def test_video_pipeline_matches_oracle_ragged():
    B = 3
    vid, nf = _video_batch(B, 43)
    sd = synth.seeded_state_dict(synth.model_spec("video"), 72, "strong")
    lens = [E.upsampled_length(f) for f in nf]
    x = torch.zeros(B, max(lens), 67, 67)
    for b, f in enumerate(nf):
        x[b, :lens[b]] = torch.from_numpy(ov.upsample_gather(vid[b, :f].numpy(), lens[b], synth.VIDEO_MEAN,
                                                             synth.VIDEO_STD))
    with torch.no_grad():
        ref = _placed(sd, "vad_video", om.deepvad_video_forward(x, lens, sd).numpy(), lens)
    pipe = AVVADPipeline(sd, video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD, modality="video")
    logits, _, _ = pipe.infer_device(None, None, vid.cuda(), nf)
    check_logits(logits.cpu().numpy(), ref, lens, "video-only pipeline, ragged B=3")


def test_golden_utterance_config0_audio_from_raw_waveform():
    g = golden("golden_frontend_34M.npz")
    wav = g["sa1_noisy_wav"].astype(np.float32) / 32768.0
    mean, std = g["audio_mean"][:, 0], g["audio_std"][:, 0]
    T = E.stft_num_frames(len(wav))
    x = torch.tensor(np.ascontiguousarray(ofe.frontend_features(wav, mean, std, dtype=np.float32)))[None]
    sd = synth.seeded_state_dict(synth.model_spec("audio"), 101, "strong")
    with torch.no_grad():
        ref = _placed(sd, "vad_audio", om.deepvad_audio_forward(x, [T], sd).numpy(), [T])
    pipe = AVVADPipeline(sd, mean, std, modality="audio")
    logits, post, dec = pipe.infer_device(torch.tensor(wav, device="cuda")[None], [len(wav)], None, None)
    assert logits.shape == (1, T, 1)
    check_logits(logits.cpu().numpy(), ref, [T], "config 0 through AVVADPipeline(modality='audio'), test/34M/sa1")
    assert torch.equal(dec, (post > 0.5).int())


def test_golden_utterance_config1_video_from_upsampled_frames():
    g, gf = golden("golden_upsample.npz"), golden("golden_frontend_34M.npz")
    frames_u8 = g["sa1_X_first24"]                                     # (24,67,67) from the shipped *_upsampled.h5
    vm, vs = float(gf["video_mean"][0, 0]), float(gf["video_std"][0, 0])
    x = torch.tensor((frames_u8.astype(np.float32) - np.float32(vm)) / (np.float32(vs) + np.float32(1e-8)))[None]
    sd = synth.seeded_state_dict(synth.model_spec("video"), 102, "strong")
    with torch.no_grad():
        ref = _placed(sd, "vad_video", om.deepvad_video_forward(x, [24], sd).numpy(), [24])
    pipe = AVVADPipeline(sd, video_mean=vm, video_std=vs, modality="video", upsampled_video=True)
    logits, _, _ = pipe.infer_device(None, None, torch.tensor(frames_u8)[None].cuda(), [24])
    check_logits(logits.cpu().numpy(), ref, [24], "config 1 through AVVADPipeline(modality='video'), test/34M/sa1")


# ---- sharded evaluation --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("modality", ["audio", "video"])
def test_evaluation_does_not_depend_on_the_call_grouping(modality):
    """One call, calls of three in list order, one utterance per call and three ranks: bit-identical posteriors (no MCB,
    per-row front end / trunk, recurrence and head), which is what lets the shard be sorted by length."""
    n = 7
    if modality == "audio":
        utts = [(synth.synth_wave(9000 + 2311 * ((5 * i + 3) % n), 90 + i), None) for i in range(n)]
        mean, std = synth.synth_audio_stats(0)
        pipe = AVVADPipeline(synth.seeded_state_dict(synth.model_spec("audio"), 51, "strong"), mean, std,
                             modality="audio")
    else:
        utts = [(None, synth.synth_video_u8(10 + 4 * ((5 * i + 3) % n), 90 + i)) for i in range(n)]
        pipe = AVVADPipeline(synth.seeded_state_dict(synth.model_spec("video"), 51, "strong"),
                             video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD, modality="video")
    a = evaluate_shard(pipe, utts, batch_size=n)
    b = evaluate_shard(pipe, utts, batch_size=3, sort_by_length=False)
    c = evaluate_shard(pipe, utts, batch_size=1)
    T = pipe.lengths_of([len(w) for w, _ in utts] if modality == "audio" else None,
                        [v.shape[0] for _, v in utts] if modality == "video" else None)
    for (sa, ha), (sb, hb), (sc, hc), t in zip(a, b, c, T):
        assert sa.shape == (t,)
        assert torch.equal(sa, sb) and torch.equal(ha, hb)
        assert torch.equal(sa, sc) and torch.equal(ha, hc)
    got = {}
    for rank in range(3):
        lo, hi, res = evaluate_sharded(pipe, utts, 3, rank, batch_size=2)
        got.update(zip(range(lo, hi), res))
    assert sorted(got) == list(range(n))
    for i, (s, h) in got.items():
        assert torch.equal(s, a[i][0]) and torch.equal(h, a[i][1])
