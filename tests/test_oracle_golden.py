"""CPU: pin the oracle against the reference's own golden artefacts and module outputs
(tests/golden/*.npz, built by tools/make_golden.py from /root/reference)."""
import os

import numpy as np
import pytest
import torch

from oracle import frontend as ofe
from oracle import models as om
from oracle import video as ov
from avvad import synth
from util import ref_models

G = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gfe():
    return np.load(os.path.join(G, "golden_frontend_34M.npz"))


@pytest.fixture(scope="module")
def gup():
    return np.load(os.path.join(G, "golden_upsample.npz"))


@pytest.fixture(scope="module")
def gref():
    return ref_models()


# ---- front end ---------------------------------------------------------------------------------
@pytest.mark.parametrize("utt,T,padded", [("sa1", 317, False), ("sa2", 283, True), ("si494", 277, False)])
def test_frame_count_and_pad_rule(gfe, utt, T, padded):
    n = len(gfe[utt + "_wav"])
    assert ofe.pad_at_end_fires(n) == padded
    assert ofe.num_frames(n) == T == gfe[utt + "_vad"].shape[1]


@pytest.mark.parametrize("utt", ["sa1", "sa2", "si494"])
@pytest.mark.parametrize("prec", ["f64", "torch_f32"])
def test_ibm_labels_bit_exact(gfe, utt, prec):
    """clean_speech_IBM(stft(clean/max)) reproduces the shipped *_ibm_labels.h5 on every cell."""
    wav = gfe[utt + "_wav"].astype(np.float32) / 32768.0  # torchaudio.load scaling
    x = ofe.peak_normalise(wav)
    S = ofe.stft_complex(x, dtype=np.float64) if prec == "f64" else ofe.stft_torch_fp32(x)
    mask = ofe.clean_speech_IBM(S)
    shape = tuple(gfe[utt + "_ibm_shape"])
    gold = np.unpackbits(gfe[utt + "_ibm_bits"])[: shape[0] * shape[1]].reshape(shape)
    assert mask.shape == shape
    assert int((mask != gold).sum()) == 0


@pytest.mark.parametrize("utt", ["sa1", "sa2", "si494"])
def test_vad_labels_bit_exact(gfe, utt):
    wav = gfe[utt + "_wav"].astype(np.float32) / 32768.0
    x = ofe.peak_normalise(wav)
    vad = ofe.clean_speech_VAD(x)
    assert np.array_equal(vad.astype(np.uint8), gfe[utt + "_vad"])


def test_logpower_f32_vs_f64(gfe):
    """Error profile of the fp32 library STFT the reference calls, against the float64 oracle:
    median ~1e-6, 99% < 1e-4, deep spectral nulls up to ~2e-3 abs on log-power.  The CUDA front
    end is held to the same profile (tests/test_gpu_frontend.py)."""
    x = ofe.peak_normalise(gfe["sa1_noisy_wav"].astype(np.float32) / 32768.0)
    S32 = ofe.stft_torch_fp32(x)
    lp32 = np.log(S32.real.astype(np.float32) ** 2 + S32.imag.astype(np.float32) ** 2 + np.float32(1e-8))
    lp64 = ofe.logpower(x, dtype=np.float64)
    d = np.abs(lp32 - lp64)
    assert np.quantile(d, 0.5) < 5e-6
    assert np.quantile(d, 0.99) < 1e-4
    assert d.max() < 2e-2


# ---- upsampling -------------------------------------------------------------------------------
def test_upsample_closed_form_matches_model():
    for F in (1, 2, 5, 6, 18, 131, 152, 192):
        assert np.array_equal(ov.upsample_index(F), ov.upsample_index_bruteforce(F)), F


def test_upsample_index_matches_reference_files(gup):
    for tag in gup["names"]:
        F, T = int(gup[tag + "_F"]), int(gup[tag + "_T"])
        assert T <= ov.upsampled_length(F)
        assert np.array_equal(ov.upsample_index(F, T), gup[tag + "_src"]), tag


def test_dct_decode_matches_reference_pixels(gup):
    rows = gup["sa1_mat_rows"]
    gold = gup["sa1_X_first24"].astype(np.int32)  # (24,67,67)
    src = np.stack([ov.roi_to_u8_per_frame(ov.dct_to_roi(r)) for r in rows])
    up = src[ov.upsample_index(152, 24)].astype(np.int32)
    d = np.abs(up - gold)
    assert d.max() <= 1
    assert (d == 0).mean() > 0.8


def test_idct_matrix_matches_scipy():
    sp = pytest.importorskip("scipy.fftpack")
    a = np.random.default_rng(0).standard_normal((67, 67))
    ref = sp.idct(sp.idct(a).T).T
    assert np.allclose(ov.dct_to_roi(a.ravel()), ref, rtol=1e-10, atol=1e-8)


# ---- models vs the reference's own modules ----------------------------------------------------
def _sd(kind, seed, **kw):
    return synth.seeded_state_dict(synth.model_spec(kind, **kw), seed)


def test_audio_forward_matches_reference(gref):
    sd = _sd("audio", 11)
    out = om.deepvad_audio_forward(torch.tensor(gref["audio_x"]), gref["audio_len"].tolist(), sd)
    assert np.allclose(out.numpy(), gref["audio_out"], atol=2e-5)
    # padded steps output the bias exactly (zeros from pad_packed_sequence through the Linear)
    assert np.allclose(out.numpy()[2, 7:, 0], sd["vad_audio.bias"].item(), atol=0)


def test_resnet_trunk_matches_reference(gref):
    sd = _sd("video", 12)
    f = om.resnet18_trunk(torch.tensor(gref["video_x"]).view(12, 67, 67), sd)
    assert np.allclose(f.numpy(), gref["video_feat"], atol=1e-4, rtol=1e-4)


def test_video_forward_matches_reference(gref):
    sd = _sd("video", 12)
    x = torch.tensor(gref["video_x"])
    out = om.deepvad_video_forward(x, gref["video_len"].tolist(), sd)
    assert np.allclose(out.numpy(), gref["video_out"], atol=5e-5)
    last = om.deepvad_video_forward(x, gref["video_len"].tolist(), sd, return_last=True)
    assert np.allclose(last.numpy(), gref["video_out_last"], atol=5e-5)


@pytest.mark.parametrize("y_dim,seed,key", [(1, 13, "av_out"), (513, 14, "av513_out")])
def test_av_concat_forward_matches_reference(gref, y_dim, seed, key):
    sd = _sd("av", seed, y_dim=y_dim)
    out = om.deepvad_av_forward(torch.tensor(gref["av_audio"]), torch.tensor(gref["av_video"]),
                                gref["av_len"].tolist(), sd, use_mcb=False)
    assert np.allclose(out.numpy(), gref[key], atol=5e-5)


def test_count_sketch_matches_reference_and_mcb_is_circular_convolution(gref):
    h = synth.seeded_tensor("mcb.sketch1.h", (513,), torch.int64, 15)
    s = synth.seeded_tensor("mcb.sketch1.s", (513,), torch.float32, 15)
    x = torch.tensor(gref["sketch_x"])
    px = om.count_sketch(x, h, s, 1024)
    assert np.array_equal(px.numpy(), gref["sketch_out"])
    # MCB == circular convolution of the two sketches (SURVEY §8a F2)
    sd = _sd("av", 15, use_mcb=True)
    a = torch.randn(1, 2, 513, dtype=torch.float64)
    v = torch.randn(1, 2, 512, dtype=torch.float64)
    sd64 = {k: (t.double() if t.is_floating_point() else t) for k, t in sd.items()}
    y = om.mcb(a, v, sd64)
    pa = om.count_sketch(a, sd["mcb.sketch1.h"], sd64["mcb.sketch1.s"], 1024)[0, 0].numpy()
    pv = om.count_sketch(v, sd["mcb.sketch2.h"], sd64["mcb.sketch2.s"], 1024)[0, 0].numpy()
    conv = np.array([np.dot(pa, np.roll(pv[::-1], k + 1)) for k in range(1024)])
    assert np.allclose(y[0, 0].numpy(), conv, atol=1e-10)


def test_loss_and_metrics_match_reference(gref):
    r, t = torch.tensor(gref["bce_r"]), torch.tensor(gref["bce_t"])
    assert np.allclose(om.binary_cross_entropy(r, t, 1e-8).numpy(), gref["bce_out"], rtol=1e-6)
    yh = (torch.sigmoid(r[:, 0]) > 0.5).int()
    vals = [v.item() for v in om.f1_loss(yh, t[:, 0].long(), 1e-8)]
    assert np.allclose(vals, gref["f1_out"], rtol=1e-6)


def test_wavenet_matches_reference(gref):
    from collections import OrderedDict
    dil = [1, 2, 4, 8, 1, 2, 4, 8]
    spec = OrderedDict()
    spec["en_dilation_layer_stack.0.weight"] = None  # placeholder to keep key order irrelevant
    spec.clear()
    shapes = {"en_causal_layer": (32, 16, 2), "bottleneck_layer": (16, 32, 1)}
    for i in range(len(dil)):
        shapes[f"en_dilation_layer_stack.{i}"] = (32, 32, 2)
        shapes[f"en_dense_layer_stack.{i}"] = (32, 32, 1)
    sd = {}
    for k, shp in shapes.items():
        sd[k + ".weight"] = synth.seeded_tensor(k + ".weight", shp, torch.float32, 16)
        sd[k + ".bias"] = synth.seeded_tensor(k + ".bias", (shp[0],), torch.float32, 16)
    out = om.wavenet_encode(torch.tensor(gref["wavenet_x"]), sd, dil, 10)
    assert np.allclose(out.numpy(), gref["wavenet_out"], atol=1e-5)
