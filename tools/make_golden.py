#!/usr/bin/env python
"""Build tests/golden/*.npz from the reference (run in the build container only).

  python tools/make_golden.py [/root/reference]

Two kinds of fixtures are produced (SURVEY §8c):
  A. golden_*.npz  -- the reference's OWN artefacts under data/subset (wavs, IBM/VAD label files,
     *_upsampled.h5, *.mat), reduced to what the parity tests need;
  B. ref_*.npz     -- outputs of the reference's own Python modules imported from
     <reference>/packages and run here on seeded inputs / seeded weights
     (avvad.synth.seeded_tensor), so the GPU box -- which never sees /root/reference -- can
     check the oracle and the CUDA path against the real implementation.
"""
from __future__ import annotations

import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(REPO, "audio-visual-vad_b200"))
sys.path.insert(0, REPO)

from avvad.h5min import H5File, read_wav_int16  # noqa: E402
from avvad import synth  # noqa: E402

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
OUT = os.path.join(REPO, "tests", "golden")
SUB = os.path.join(REF, "data", "subset")
os.makedirs(OUT, exist_ok=True)
warnings.filterwarnings("ignore")


def golden_frontend():
    """clean wavs + IBM/VAD label files of test/34M (the only split generated at 62.5 fps)."""
    d = {}
    base = os.path.join(SUB, "processed/ntcd_timit/Clean/test/34M")
    for utt in ("sa1", "sa2", "si494"):
        wav, fs = read_wav_int16(os.path.join(base, utt + ".wav"))
        assert fs == 16000
        ibm = H5File(os.path.join(base, utt + "_ibm_labels.h5"))["Y"]
        vad = H5File(os.path.join(base, utt + "_vad_labels.h5"))["Y"]
        assert set(np.unique(ibm)) <= {0.0, 1.0} and set(np.unique(vad)) <= {0.0, 1.0}
        d[utt + "_wav"] = wav
        d[utt + "_ibm_shape"] = np.asarray(ibm.shape)
        d[utt + "_ibm_bits"] = np.packbits(ibm.astype(np.uint8).ravel())
        d[utt + "_vad"] = vad.astype(np.uint8)
    # noisy file of the same utterance: what the AV model actually consumes
    noisy = os.path.join(SUB, "processed/ntcd_timit/Noisy/Babble/-5/test/34M/sa1.wav")
    if os.path.exists(noisy):
        d["sa1_noisy_wav"] = read_wav_int16(noisy)[0]
    st = H5File(os.path.join(SUB, "processed/ntcd_timit/Noisy/ntcd_timit_power_spec_statistics.h5"))
    d["audio_mean"] = st["X_train_mean"].astype(np.float32)
    d["audio_std"] = st["X_train_std"].astype(np.float32)
    sv = H5File(os.path.join(SUB, "processed/ntcd_timit/matlab_raw/ntcd_timit_statistics.h5"))
    d["video_mean"] = sv["X_train_mean"].astype(np.float32)
    d["video_std"] = sv["X_train_std"].astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "golden_frontend_34M.npz"), **d)
    print("golden_frontend_34M.npz", {k: v.shape for k, v in d.items()})


def golden_upsample():
    """Recover src(k) for every frame of every shipped *_upsampled.h5 by matching it to the
    inverse-DCT frames of the .mat it was made from (argmax correlation); keep a small pixel
    excerpt of test/34M/sa1 to pin the DCT->ROI decode."""
    from oracle.video import dct_to_roi, roi_to_u8_per_frame

    d = {}
    names = []
    for split, spk, utt in (("test", "34M", "sa1"), ("test", "34M", "sa2"), ("test", "34M", "si494"),
                            ("dev", "08F", "sa1"), ("train", "01M", "sa1")):
        up = os.path.join(SUB, f"processed/ntcd_timit/matlab_raw/{split}/{spk}/{utt}_upsampled.h5")
        mat = os.path.join(SUB, f"raw/ntcd_timit/matlab_raw/{split}/{spk}/{utt}.mat")
        if not (os.path.exists(up) and os.path.exists(mat)):
            continue
        X = H5File(up)["X"]  # (67,67,T)
        D = H5File(mat)["data"]  # (F,4489)
        src = np.stack([roi_to_u8_per_frame(dct_to_roi(row)) for row in D]).astype(np.float64)  # (F,67,67)
        Xf = np.moveaxis(X, -1, 0).astype(np.float64)  # (T,67,67)
        a = src.reshape(len(src), -1)
        b = Xf.reshape(len(Xf), -1)
        a0 = a - a.mean(1, keepdims=True)
        b0 = b - b.mean(1, keepdims=True)
        # frames are near-duplicates of neighbours: use mean |diff| (exact match ~0.3) not correlation
        idx = np.empty(len(b), dtype=np.int64)
        err = np.empty(len(b))
        for k in range(len(b)):
            lo = max(0, int(k * 12 / 25) - 3)
            hi = min(len(a), lo + 8)
            e = np.abs(a[lo:hi] - b[k][None]).mean(1)
            idx[k] = lo + int(np.argmin(e))
            err[k] = e.min()
        tag = f"{split}_{spk}_{utt}"
        names.append(tag)
        d[tag + "_F"] = np.asarray(D.shape[0])
        d[tag + "_T"] = np.asarray(X.shape[-1])
        d[tag + "_src"] = idx.astype(np.int32)
        d[tag + "_maxerr"] = np.asarray(err.max())
        print(tag, "F", D.shape[0], "T", X.shape[-1], "match err max", err.max(), "first", idx[:14])
        if tag == "test_34M_sa1":
            d["sa1_mat_rows"] = D[:12].astype(np.float32)  # DCT rows of source frames 0..11
            d["sa1_X_first24"] = np.moveaxis(X[:, :, :24], -1, 0).astype(np.uint8)  # integer-valued f32
            assert np.all(X[:, :, :24] == np.rint(X[:, :, :24]))
    d["names"] = np.asarray(names)
    np.savez_compressed(os.path.join(OUT, "golden_upsample.npz"), **d)


def ref_models():
    """Reference modules on seeded weights/inputs."""
    sys.path.insert(0, REF)
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models.Video_Net import DeepVAD_video
    from packages.models.AV_Net import DeepVAD_AV
    from packages.models.compact_bilinear_pooling import CountSketchFn_forward
    from packages.models.utils import binary_cross_entropy, f1_loss, method3
    from packages.models.wavenet_autoencoder import wavenet_autoencoder
    from packages.utils import collate_many2many_AV, collate_many2many_audio, collate_many2many_video

    d = {}
    g = torch.Generator().manual_seed(1234)
    mean_a, std_a = synth.synth_audio_stats(0)

    # ---- audio-only ----
    m = synth.fill_module_(DeepVAD_audio(2, 1024, 1), seed=11).eval()
    xa = torch.randn(3, 20, 513, generator=g)
    la = [20, 13, 7]
    with torch.no_grad():
        d["audio_x"], d["audio_len"], d["audio_out"] = xa.numpy(), np.asarray(la), m(xa, la).numpy()

    # ---- video-only ----
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=12).eval()
    xv = torch.randn(2, 6, 67, 67, generator=g)
    lv = [6, 4]
    with torch.no_grad():
        d["video_x"], d["video_len"], d["video_out"] = xv.numpy(), np.asarray(lv), m(xv, lv).numpy()
        d["video_out_last"] = m(xv, torch.tensor(lv), return_last=True).numpy()
        # trunk features for a handful of frames (pins the ResNet restatement layer by layer)
        f = m.features(xv.view(12, 1, 67, 67).repeat(1, 3, 1, 1)).squeeze()
        d["video_feat"] = f.numpy()

    # ---- AV, concat fusion (the only AV variant the reference can execute on torch 2.x) ----
    m = synth.fill_module_(DeepVAD_AV(2, 1024, 1, use_mcb=False, eps=1e-8), seed=13).eval()
    xa2 = torch.randn(2, 6, 513, generator=g)
    with torch.no_grad():
        d["av_audio"], d["av_len"] = xa2.numpy(), np.asarray(lv)   # video input: video_x (tests/util.py::ref_models)
        d["av_out"] = m(xa2, xv, lv).numpy()
    # y_dim = 513 (IBM variant, train_AV_net.py:65-66)
    m = synth.fill_module_(DeepVAD_AV(2, 1024, 513, use_mcb=False, eps=1e-8), seed=14).eval()
    with torch.no_grad():
        d["av513_out"] = m(xa2, xv, lv).numpy()

    # ---- count sketch (the part of MCB that still runs) ----
    h1 = synth.seeded_tensor("mcb.sketch1.h", (513,), torch.int64, 15)
    s1 = synth.seeded_tensor("mcb.sketch1.s", (513,), torch.float32, 15)
    xs = torch.randn(2, 5, 513, generator=g)
    d["sketch_x"], d["sketch_out"] = xs.numpy(), CountSketchFn_forward(h1, s1, 1024, xs).numpy()

    # ---- loss / metrics ----
    r = torch.randn(37, 1, generator=g) * 3
    t = (torch.rand(37, 1, generator=g) > 0.4).float()
    d["bce_r"], d["bce_t"] = r.numpy(), t.numpy()
    d["bce_out"] = binary_cross_entropy(r, t, 1e-8).numpy()
    yh = (torch.sigmoid(r[:, 0]) > 0.5).int()
    d["f1_out"] = np.asarray([v.item() for v in f1_loss(yh, t[:, 0].long(), 1e-8)], dtype=np.float32)

    # ---- collate ----
    batch = [(torch.randn(513, L, generator=g), torch.randn(67, 67, L, generator=g),
              (torch.rand(1, L, generator=g) > 0.5).float(), L) for L in (5, 3, 4)]
    lens, pa, pv, pt = collate_many2many_AV(batch)
    d["collate_in_a"] = np.concatenate([b[0].numpy().ravel() for b in batch])
    d["collate_in_v"] = np.concatenate([b[1].numpy().ravel() for b in batch])
    d["collate_in_t"] = np.concatenate([b[2].numpy().ravel() for b in batch])
    d["collate_lens"], d["collate_a"], d["collate_v"], d["collate_t"] = lens.numpy(), pa.numpy(), pv.numpy(), pt.numpy()

    # ---- WaveNet encoder (dead code, but named by north_star) ----
    wn = wavenet_autoencoder(filter_width=2, quantization_channel=16, dilations=[1, 2, 4, 8, 1, 2, 4, 8],
                             en_residual_channel=32, en_dilation_channel=32, en_bottleneck_width=16,
                             en_pool_kernel_size=10, use_bias=True)
    synth.fill_module_(wn, seed=16).eval()
    xw = torch.randn(2, 16, 400, generator=g)
    with torch.no_grad():
        d["wavenet_x"], d["wavenet_out"] = xw.numpy(), wn(xw).numpy()

    # ---- reference front-end library call (torch.stft is what stft_pytorch wraps) ----
    np.savez_compressed(os.path.join(OUT, "ref_models.npz"), **d)
    print("ref_models.npz", {k: v.shape for k, v in d.items()})


def install_legacy_fft_shim():
    """torch.rfft / torch.irfft were removed in torch 1.8; the reference's MCB (compact_bilinear_pooling.py:152-171,
    186-215) still calls them.  Two pure re-spellings through torch.fft restore the legacy signatures
    (rfft(x, 1) -> (..., N/2+1, 2) real view, un-normalised; irfft(X, 1, signal_sizes=(N,)) -> 1/N-normalised inverse),
    so the UNMODIFIED reference module executes here."""
    if not hasattr(torch, "rfft"):
        torch.rfft = lambda x, signal_ndim=1, normalized=False, onesided=True: torch.view_as_real(torch.fft.rfft(x))
    _new_irfft = torch.fft.irfft

    def _irfft(x, signal_ndim=1, normalized=False, onesided=True, signal_sizes=None):
        return _new_irfft(torch.view_as_complex(x.contiguous()), n=signal_sizes[0])
    if not hasattr(torch, "irfft"):
        torch.irfft = _irfft


def grad_digest(d, tag, named_params):
    """Compact, discriminating fingerprint of a gradient set: Frobenius norm and a strided sample of <= 2048 elements of
    every tensor (full gradients of the 11-28 M-parameter models are too large to commit)."""
    for k, p in named_params:
        if p.grad is None:
            continue
        g = p.grad.detach().reshape(-1)
        step = max(1, g.numel() // 2048)
        d[f"{tag}/{k}/norm"] = np.asarray(g.double().norm().item())
        d[f"{tag}/{k}/sample"] = g[::step][:2048].numpy().copy()


def ref_strong():
    """Second fixture file, all from the reference's own modules:
      * the assembled use_mcb=True forward (AV_Net.py:111-121) and the stand-alone CompactBilinearPooling forward /
        hand-written backward (compact_bilinear_pooling.py:140-220), executed through install_legacy_fft_shim();
      * every module on the "strong" weight family (avvad.synth.FAMILIES) whose logits span several units;
      * one training step (train() mode, loss as scripts/train_AV_net.py:298-301) of DeepVAD_AV(use_mcb=True) with the
        trunk frozen (train_AV_net.py:241-245) and of DeepVAD_video with the trunk trainable
        (train_video_net.py:145-173): loss + gradient digests, running-statistics of all 20 BatchNorm2d layers."""
    sys.path.insert(0, REF)
    install_legacy_fft_shim()
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models.Video_Net import DeepVAD_video
    from packages.models.AV_Net import DeepVAD_AV
    from packages.models.compact_bilinear_pooling import CompactBilinearPooling
    from packages.models.utils import binary_cross_entropy

    base = np.load(os.path.join(OUT, "ref_models.npz"))
    d = {}
    g = torch.Generator().manual_seed(4242)

    # ---- stand-alone MCB: forward + backward of the reference Function ----
    h1 = synth.seeded_tensor("mcb.sketch1.h", (513,), torch.int64, 15)
    s1 = synth.seeded_tensor("mcb.sketch1.s", (513,), torch.float32, 15)
    h2 = synth.seeded_tensor("mcb.sketch2.h", (512,), torch.int64, 15)
    s2 = synth.seeded_tensor("mcb.sketch2.s", (512,), torch.float32, 15)
    cbp = CompactBilinearPooling(513, 512, 1024, h1=h1, s1=s1, h2=h2, s2=s2)
    x = torch.randn(2, 5, 513, generator=g, requires_grad=True)
    y = torch.randn(2, 5, 512, generator=g).abs().requires_grad_(True)
    go = torch.randn(2, 5, 1024, generator=g)
    out = cbp(x, y)
    out.backward(go)
    d["cbp_x"], d["cbp_y"], d["cbp_go"] = x.detach().numpy(), y.detach().numpy(), go.numpy()
    d["cbp_out"], d["cbp_gx"], d["cbp_gy"] = out.detach().numpy(), x.grad.numpy(), y.grad.numpy()

    a6, v6, l6 = torch.tensor(base["av_audio"]), torch.tensor(base["video_x"]), base["av_len"].tolist()

    def strong_forward(m, head, key, *inputs, lengths):
        """Forward with the strong family, head bias placed by synth.decision_bias (stored as <key>_bias)."""
        m.eval()
        with torch.no_grad():
            out0 = m(*inputs, lengths).numpy()
            nb = synth.decision_bias(out0, lengths, head.bias.detach().numpy())
            head.bias.copy_(nb)
            d[key + "_bias"] = nb.numpy()
            d[key] = m(*inputs, lengths).numpy()
        return m

    # ---- assembled AV + MCB forward (seed 22 default family as in the GPU test; seed 42 strong family) ----
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 22), 12))
    m.eval()
    with torch.no_grad():
        d["av_mcb_out_default"] = m(a6, v6, l6).numpy()
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 42, "strong"), 12))
    strong_forward(m, m.vad_merged, "av_mcb_out_strong", a6, v6, lengths=l6)

    # ---- strong family, all modules ----
    # long ragged batch: exercises error growth over many recurrence steps
    # (input = numpy PCG64 stream, regenerated by the tests instead of being stored: 2.6 MB)
    xl = torch.tensor(np.random.default_rng(77).standard_normal((4, 317, 513)).astype(np.float32))
    ll = [317, 301, 158, 317]
    m = synth.fill_module_(DeepVAD_audio(2, 1024, 1), seed=41, family="strong")
    strong_forward(m, m.vad_audio, "audio_long_out_strong", xl, lengths=ll)
    d["audio_long_len"] = np.asarray(ll)
    xa, la = torch.tensor(base["audio_x"]), base["audio_len"].tolist()
    with torch.no_grad():   # same weights and (calibrated) bias on the short batch of ref_models.npz
        d["audio_out_strong"] = m(xa, la).numpy()
    # video / AV: 40 frames per utterance so that the bias placement has a distribution to work with
    vl = torch.tensor(np.random.default_rng(78).standard_normal((2, 40, 67, 67)).astype(np.float32))
    al = torch.tensor(np.random.default_rng(79).standard_normal((2, 40, 513)).astype(np.float32))
    lv = [40, 29]
    d["av_long_len"] = np.asarray(lv)
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=43, family="strong")
    strong_forward(m, m.vad_video, "video_out_strong", vl, lengths=lv)
    for y_dim, seed, key in ((1, 44, "av_out_strong"), (513, 45, "av513_out_strong")):
        m = synth.fill_module_(DeepVAD_AV(2, 1024, y_dim, use_mcb=False, eps=1e-8), seed=seed, family="strong")
        strong_forward(m, m.vad_merged, key, al, vl, lengths=lv)

    # ---- training step, AV + MCB, trunk frozen (reference loop: train_AV_net.py:241-245,253,293-305) ----
    tgt = (torch.rand(2, 6, 1, generator=g) > 0.5).float()
    d["train_target"] = tgt.numpy()
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 46, "strong"))
    for name, child in m.named_children():
        if name == "features":
            for p in child.parameters():
                p.requires_grad = False
    m.train()
    out = m(a6, v6, torch.tensor(l6))
    loss = 0.
    for length, pred, target in zip(l6, out, tgt.long()):
        loss = loss + binary_cross_entropy(pred[:length], target[:length], 1e-8)
    loss.backward()
    d["train_av_mcb_logits"], d["train_av_mcb_loss"] = out.detach().numpy(), np.asarray(loss.item())
    grad_digest(d, "train_av_mcb", m.named_parameters())
    d["train_av_mcb/mcb_bn.running_mean"] = m.mcb_bn.running_mean.numpy().copy()
    d["train_av_mcb/mcb_bn.running_var"] = m.mcb_bn.running_var.numpy().copy()

    # ---- training step, video-only, trunk TRAINABLE (train_video_net.py:145-173) ----
    m = synth.fill_module_(DeepVAD_video(2, 1024, 1), seed=47, family="strong")
    m.train()
    out = m(v6, torch.tensor(l6))
    loss = 0.
    for length, pred, target in zip(l6, out, tgt.long()):
        loss = loss + binary_cross_entropy(pred[:length], target[:length], 1e-8)
    loss.backward()
    d["train_video_logits"], d["train_video_loss"] = out.detach().numpy(), np.asarray(loss.item())
    grad_digest(d, "train_video", m.named_parameters())
    for k, v in m.state_dict().items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            d["train_video/" + k] = v.numpy().copy()

    np.savez_compressed(os.path.join(OUT, "ref_strong.npz"), **d)
    print("ref_strong.npz", len(d), "arrays;",
          {k: (round(float(np.min(d[k])), 2), round(float(np.max(d[k])), 2), round(float((d[k] > 0).mean()), 3))
           for k in d if k.endswith("_strong") or k.startswith("av_mcb_out")})


EVAL_SINGLE_LENS = [23, 9, 16, 31]


def eval_single_inputs():
    """Inputs of ref_eval_single(), regenerated by the tests from the same PCG64 streams instead of being stored."""
    B, T = len(EVAL_SINGLE_LENS), max(EVAL_SINGLE_LENS)
    a = np.random.default_rng(91).standard_normal((B, T, 513)).astype(np.float32)
    v = np.random.default_rng(92).standard_normal((B, T, 67, 67)).astype(np.float32)
    return a, v, list(EVAL_SINGLE_LENS)


def ref_eval_single():
    """The reference's evaluation call pattern (scripts/evaluate_AV_net.py:186-236): the UNMODIFIED DeepVAD_AV
    (use_mcb=True, eval()) called ONCE PER UTTERANCE with x[None], v[None], lengths = [T], so AV_Net.py:117's
    whole-tensor L2 norm is a per-utterance norm.  Strong weight family, head bias placed by synth.decision_bias over all
    utterances.  -> tests/golden/ref_eval_single.npz (logits padded to (B, Tmax, 1), bias)."""
    sys.path.insert(0, REF)
    install_legacy_fft_shim()
    from packages.models.AV_Net import DeepVAD_AV

    a, v, lens = eval_single_inputs()
    m = DeepVAD_AV(2, 1024, 1, use_mcb=True, eps=1e-8)
    m.load_state_dict(synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 43, "strong"), 20))
    m.eval()

    def run():
        out = np.zeros((len(lens), max(lens), 1), dtype=np.float32)
        with torch.no_grad():
            for b, n in enumerate(lens):
                out[b, :n] = m(torch.tensor(a[b:b + 1, :n]), torch.tensor(v[b:b + 1, :n]), [n]).numpy()[0]
        return out

    out0 = run()
    with torch.no_grad():
        nb = synth.decision_bias(out0, lens, m.vad_merged.bias.detach().numpy())
        m.vad_merged.bias.copy_(nb)
    out = run()
    with torch.no_grad():  # for contrast: ONE batched call of the same utterances (whole-call norm over the padded tensor)
        batched = m(torch.tensor(a), torch.tensor(v), lens).numpy()
    np.savez_compressed(os.path.join(OUT, "ref_eval_single.npz"), logits=out, bias=nb.numpy(), lens=np.asarray(lens),
                        batched_call_logits=batched)
    valid = np.concatenate([out[b, :n, 0] for b, n in enumerate(lens)])
    print("ref_eval_single.npz: logits range [%.2f, %.2f] std %.2f; batched-call logits differ by up to %.2f" %
          (valid.min(), valid.max(), valid.std(),
           max(np.abs(out[b, :n] - batched[b, :n]).max() for b, n in enumerate(lens))))


def golden_h5():
    """Two small files of the reference copied verbatim (data, 4 KB + 9 KB) and the first LZF chunks of a video file:
    they pin the HDF5 writer (message bytes, chunk shapes) and the LZF encoder (stored bytes) of avvad/h5min.py."""
    import shutil
    import struct
    os.makedirs(os.path.join(OUT, "h5"), exist_ok=True)
    base = os.path.join(SUB, "processed/ntcd_timit")
    shutil.copyfile(os.path.join(base, "Clean/test/34M/sa1_vad_labels.h5"), os.path.join(OUT, "h5", "sa1_vad_labels.h5"))
    shutil.copyfile(os.path.join(base, "matlab_raw/ntcd_timit_statistics.h5"), os.path.join(OUT, "h5", "ntcd_timit_statistics.h5"))
    h = H5File(os.path.join(base, "matlab_raw/test/34M/sa1_upsampled.h5"))
    layout = [d for t, d in h._messages(h.datasets["/X"]) if t == 0x08][0]
    ndim = layout[2]
    btree = struct.unpack_from("<Q", layout, 3)[0]
    found = []

    def walk(addr):
        b = h.buf
        _, level, used = struct.unpack_from("<BBH", b, addr + 4)
        p, ks = addr + 24, 8 + 8 * ndim
        for _ in range(used):
            nbytes, fmask = struct.unpack_from("<II", b, p)
            child = struct.unpack_from("<Q", b, p + ks)[0]
            p += ks + 8
            if level > 0:
                walk(child)
            else:
                found.append((child, nbytes, fmask))
    walk(btree)
    found.sort()
    d = {"chunk_dims": np.asarray(struct.unpack_from("<" + "I" * ndim, layout, 11)), "n_chunks_in_file": np.asarray(len(found))}
    for i, (a, n, m) in enumerate(found[:12]):   # in file (= write) order, from the start of the file
        assert m == 0
        d[f"chunk{i}"] = np.frombuffer(h.buf[a:a + n], dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, "golden_lzf_chunks.npz"), **d)
    print("golden_lzf_chunks.npz", len(found), "chunks in file, stored", min(12, len(found)))


def ref_helpers():
    """Host-level helpers of packages/models/utils.py:57-162 and packages/utils.py:9-40 on seeded inputs (a separate,
    small file so that ref_models.npz does not have to be regenerated)."""
    sys.path.insert(0, REF)
    import packages.models.utils as mu
    import packages.utils as pu
    g = torch.Generator().manual_seed(4321)
    x = torch.rand(6, 5, generator=g) + 0.1
    r = torch.rand(6, 5, generator=g) + 0.1
    mu_, lv = torch.randn(6, 4, generator=g), torch.randn(6, 4, generator=g)
    y = torch.rand(3, 2, generator=g)
    t = (x > 0.5).float()
    eps = 1e-8
    d = {"x": x, "r": r, "mu": mu_, "logvar": lv, "y": y}
    d["enumerate"] = mu.enumerate_discrete(torch.zeros(3, 7), 4)
    d["onehot_5_2"], d["onehot_3_7"] = mu.onehot(5)(2), mu.onehot(3)(7)
    d["lse"], d["lse_mean0"] = mu.log_sum_exp(x), mu.log_sum_exp(x, 0, torch.mean)
    d["bce2"] = mu.binary_cross_entropy_2classes(x, r, t, eps)
    d["isd"] = mu.ikatura_saito_divergence(r, x, eps)
    for k, v in zip(("elbo0", "elbo1", "elbo2"), mu.elbo(x, r, mu_, lv, eps)):
        d[k] = v
    for k, v in zip(("L0", "L1", "L2"), mu.L_loss(x, r, mu_, lv, eps)):
        d[k] = v
    for k, v in zip(("U0", "U1", "U2", "U3"), mu.U_loss(x, r, mu_, lv, y, eps)):
        d[k] = v
    d["mse_signal"], d["mse_mask"] = mu.mean_square_error_signal(x, r, x * 0.5), mu.mean_square_error_mask(x, r)
    d["msa"] = mu.magnitude_spectrum_approxiamation_loss(torch.complex(x, r), torch.complex(r, x), x)
    vids = [torch.rand(4, 5, 3, T, generator=g) for T in (6, 4, 5)]
    for i, v in enumerate(vids):
        d[f"collate_in{i}"] = v
    lens, data, target = pu.my_collate([(v, torch.tensor(float(i % 2)), v.shape[-1]) for i, v in enumerate(vids)])
    d["collate_len"], d["collate_data"], d["collate_target"] = lens, data, target
    d = {k: np.asarray(v) for k, v in d.items()}
    np.savez_compressed(os.path.join(OUT, "ref_helpers.npz"), **d)
    print("ref_helpers.npz", {k: v.shape for k, v in d.items()})


def ref_target_masks():
    """Threshold-based masks of packages/processing/target.py:110-251 on a seeded complex spectrogram pair.  The module
    imports librosa at its top (absent here; only clean_speech_VAD uses it), so an empty stand-in is registered."""
    import importlib.util
    import types
    for name in ("librosa", "librosa.util"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["librosa"].util = sys.modules["librosa.util"]
    spec = importlib.util.spec_from_file_location("ref_target", os.path.join(REF, "packages/processing/target.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    rng = np.random.default_rng(3)
    X = (rng.standard_normal((7, 513)) + 1j * rng.standard_normal((7, 513))) * rng.uniform(0.01, 5, (7, 513))
    N = (rng.standard_normal((7, 513)) + 1j * rng.standard_normal((7, 513))) * rng.uniform(0.01, 5, (7, 513))
    voiced, unvoiced = ref._voiced_unvoiced_split_characteristic(513)
    speech, noise = ref.noise_aware_IBM(X, N)
    np.savez_compressed(os.path.join(OUT, "ref_target_masks.npz"), X=X, N=N, voiced=voiced, unvoiced=unvoiced,
                        speech=speech, noise=noise, thresh=ref.threshold_IBM(X))
    print("ref_target_masks.npz", speech.mean(), noise.mean())


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[2] == "h5":
        golden_h5()
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[2] == "strong":
        ref_strong()
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[2] == "eval_single":
        ref_eval_single()
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[2] == "helpers":
        ref_helpers()
        ref_target_masks()
        sys.exit(0)
    golden_frontend()
    golden_upsample()
    ref_models()
    ref_strong()
    ref_eval_single()
    golden_h5()
    ref_helpers()
    ref_target_masks()
