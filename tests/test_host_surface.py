"""CPU: the host-side part of the reference-compatible surface (imports, path builders, label generation, collate,
metrics) -- what scripts/train_*_net.py and scripts/evaluate_*_net.py import at module top must import cleanly."""
import os

import numpy as np
import pytest
import torch

G = os.path.join(os.path.dirname(__file__), "golden")


def test_script_level_imports_resolve():
    from packages.models.utils import f1_loss, binary_cross_entropy  # noqa: F401
    from packages.processing.stft import stft_pytorch  # noqa: F401
    from packages.models.AV_Net import DeepVAD_AV  # noqa: F401
    from packages.models.Audio_Net import DeepVAD_audio  # noqa: F401
    from packages.models.Video_Net import DeepVAD_video  # noqa: F401
    from packages.visualization import display_multiple_signals  # noqa: F401
    from packages.dataset.ntcd_timit import proc_noisy_clean_pair_dict, speech_list, proc_video_audio_pair_dict  # noqa: F401
    from packages.data_handling import (AudioVisualSequenceLabeledFrames, NoisyWavWholeSequenceSpectrogramLabeledFrames,  # noqa: F401
                                        WavWholeSequenceSpectrogramLabeledFrames)
    from packages.utils import count_parameters, collate_many2many_AV, collate_many2many_audio, collate_many2many_video  # noqa: F401
    from packages.models.wavenet_autoencoder import wavenet_autoencoder  # noqa: F401
    import packages.metrics  # noqa: F401


def test_state_dict_keys_match_the_reference_layout():
    from avvad import synth
    from packages.models.AV_Net import DeepVAD_AV
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models.Video_Net import DeepVAD_video
    for mod, kind, kw in ((DeepVAD_AV(2, 1024, 1, use_mcb=True), "av", {"use_mcb": True}),
                          (DeepVAD_AV(2, 1024, 1, use_mcb=False), "av", {"use_mcb": False}),
                          (DeepVAD_audio(2, 1024, 1), "audio", {}), (DeepVAD_video(2, 1024, 1), "video", {})):
        sd = mod.state_dict()
        spec = synth.model_spec(kind, **kw)
        assert list(sd.keys()) == list(spec.keys()) or set(sd.keys()) == set(spec.keys())
        for k, (shape, dtype) in spec.items():
            assert tuple(sd[k].shape) == tuple(shape) and sd[k].dtype == dtype, k
    assert len(DeepVAD_AV(2, 1024, 1, use_mcb=True).state_dict()) == 144
    assert "features" in dict(DeepVAD_AV(2, 1024, 1).named_children())


def test_labels_reproduce_reference_files():
    from packages.processing import target as tg
    g = np.load(os.path.join(G, "golden_frontend_34M.npz"))
    for utt in ("sa1", "sa2", "si494"):
        x = g[utt + "_wav"].astype(np.float32) / 32768.0
        x = x / np.abs(x).max()
        vad = tg.clean_speech_VAD(x, fs=16000, wlen_sec=0.064, hop_percent=0.25, center=False)
        assert np.array_equal(vad.astype(np.uint8), g[utt + "_vad"])


def test_collate_matches_reference_golden():
    from packages.utils import collate_many2many_AV
    g = np.load(os.path.join(G, "ref_models.npz"))
    a, v, t = g["collate_in_a"], g["collate_in_v"], g["collate_in_t"]
    batch, oa, ov, ot = [], 0, 0, 0
    for L in (5, 3, 4):
        batch.append((torch.tensor(a[oa:oa + 513 * L]).view(513, L), torch.tensor(v[ov:ov + 4489 * L]).view(67, 67, L),
                      torch.tensor(t[ot:ot + L]).view(1, L), L))
        oa, ov, ot = oa + 513 * L, ov + 4489 * L, ot + L
    lens, pa, pv, pt = collate_many2many_AV(batch)
    assert np.array_equal(lens.numpy(), g["collate_lens"]) and np.array_equal(pa.numpy(), g["collate_a"])
    assert np.array_equal(pv.numpy(), g["collate_v"]) and np.array_equal(pt.numpy(), g["collate_t"])


def test_path_builders_on_the_reference_subset(tmp_path):
    """The test/34M part of the reference's data/subset/processed tree (SURVEY appendix A): sa1's label file verbatim
    (tests/golden/h5), the other label files from the golden labels, upsampled ROI videos at the shipped shapes, and
    files of the same directories that the builders must not pick up."""
    import shutil
    from avvad import h5min, synth
    from oracle import video as ov
    from packages.dataset.ntcd_timit import proc_noisy_clean_pair_dict, proc_video_audio_pair_dict
    from packages.data_handling import WavWholeSequenceSpectrogramLabeledFrames
    g = np.load(os.path.join(G, "golden_frontend_34M.npz"))
    clean = tmp_path / "ntcd_timit" / "Clean" / "test" / "34M"
    video = tmp_path / "ntcd_timit" / "matlab_raw" / "test" / "34M"
    for d in (clean, video):
        d.mkdir(parents=True)
    shutil.copyfile(os.path.join(G, "h5", "ntcd_timit_statistics.h5"), video.parent.parent / "ntcd_timit_statistics.h5")
    frames = {}
    for k, (utt, F) in enumerate((("sa1", 152), ("sa2", 136), ("si494", 134))):
        T = g[utt + "_vad"].shape[1]
        if utt == "sa1":
            shutil.copyfile(os.path.join(G, "h5", "sa1_vad_labels.h5"), clean / "sa1_vad_labels.h5")
        else:
            h5min.write_h5(str(clean / f"{utt}_vad_labels.h5"),
                           {"Y": (g[utt + "_vad"].astype(np.float32), dict(maxshape=(1, None), creation_shape=(1, 0)))})
        src = synth.synth_video_u8(F, k).astype(np.float32)
        frames[utt] = np.ascontiguousarray(np.moveaxis(src[ov.upsample_index(F, T)], 0, -1))    # (67,67,T)
        h5min.write_h5(str(video / f"{utt}_upsampled.h5"),
                       {"X": (frames[utt], dict(maxshape=(67, 67, None), creation_shape=(67, 67, 0)))})
        (clean / f"{utt}_ibm_labels.h5").touch()
        (video / f"{utt}.mat").touch()
    root = str(tmp_path) + "/"
    pairs = proc_noisy_clean_pair_dict(root, "test", "subset", "vad_labels", upsampled=False)
    assert list(pairs.items())[0] == ("ntcd_timit/Noisy/Babble/-5/test/34M/sa1.wav", "ntcd_timit/Clean/test/34M/sa1_vad_labels.h5")
    v, a = proc_video_audio_pair_dict(root, "test", "vad_labels", upsampled=True)
    assert len(v) == 3 and v[0].endswith("sa1_upsampled.h5") and a[0].endswith("sa1_vad_labels.h5")
    x, y, n = WavWholeSequenceSpectrogramLabeledFrames(root, "test", labels="vad_labels", upsampled=True)[0]
    assert tuple(x.shape) == (67, 67, 317) and tuple(y.shape) == (1, 317) and n == 317
    assert np.array_equal(x.numpy(), frames["sa1"]) and np.array_equal(y.numpy(), g["sa1_vad"])


def test_metrics_helpers():
    from packages.metrics import energy_ratios, mean_confidence_interval
    rng = np.random.default_rng(0)
    s, n = rng.standard_normal(1000), 0.1 * rng.standard_normal(1000)
    sdr, sir, sar = energy_ratios(s + n, s, n)
    assert sdr > 15 and sir > 15
    m, h = mean_confidence_interval([1.0, 2.0, 3.0, 4.0])
    assert m == 2.5 and h > 0


def test_compute_stats_has_the_reference_signature(capsys):
    """packages/metrics.py:62-68: (metrics_keys, all_metrics, model_data_dir, confidence, all_snr_db, all_noise_types,
    all_speakers) -- the scripts pass all_speakers=... by keyword; unknown keywords must raise, nothing is written."""
    import inspect
    from packages.metrics import compute_stats
    assert list(inspect.signature(compute_stats).parameters) == [
        "metrics_keys", "all_metrics", "model_data_dir", "confidence", "all_snr_db", "all_noise_types", "all_speakers"]
    rows = [(0.9, 0.8), (0.7, 0.6), (0.5, 0.4), (0.3, 0.2)]
    compute_stats(["acc", "f1"], rows, "/nonexistent/dir/", 0.95, all_snr_db=np.array([-5, -5, 0, 0]),
                  all_noise_types=["Babble", "Cafe", "Babble", "Cafe"], all_speakers=["34M", "34M", "08F", "08F"])
    out = capsys.readouterr().out
    assert "Input SNR = -5.00" in out and "Noise type = Cafe" in out and "Speaker = 08F" in out
    assert out.count("METRIC") == 1 + 2 + 2 + 2
    with pytest.raises(TypeError):
        compute_stats(["acc"], [(1.0,)], "", 0.95, all_speaker_ids=["x"])


def test_full_state_dict_inside_dataparallel_replica():
    """torch.nn.parallel.replicate strips nn.Parameters from replicas (plain tensor attributes + `_former_parameters`);
    the engines must still find every weight (scripts/train_AV_net.py:193 wraps the model in nn.DataParallel).  The
    replication is emulated here on the CPU exactly as torch/nn/parallel/replicate.py does it."""
    from collections import OrderedDict
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models._engine import all_parameters, full_state_dict
    m = DeepVAD_audio(2, 1024, 1)
    reps = {mod: mod._replicate_for_data_parallel() for mod in m.modules()}
    for mod, rep in reps.items():
        rep._former_parameters = OrderedDict()
        for k, child in mod._modules.items():
            setattr(rep, k, reps[child])
        for k, p in mod._parameters.items():
            c = p.detach().clone().requires_grad_(p.requires_grad)
            setattr(rep, k, c)
            rep._former_parameters[k] = c
    r = reps[m]
    ref = m.state_dict()
    assert len(r.state_dict()) < len(ref)            # what broke the engines: parameters are gone
    sd = full_state_dict(r)
    assert set(sd.keys()) == set(ref.keys())
    assert all(torch.equal(sd[k], ref[k]) for k in ref)
    assert len(all_parameters(r)) == len(list(m.parameters())) and any(p.requires_grad for p in all_parameters(r))


def test_modules_survive_pickle_and_deepcopy():
    """scripts/evaluate_AV_net.py:332-339 hands the classifier to a spawn-context process pool (pickle); the engine
    cache (ctypes handles) must not travel and must be re-created empty on the other side."""
    import copy
    import pickle
    from packages.models.AV_Net import DeepVAD_AV
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models.Video_Net import DeepVAD_video
    for m in (DeepVAD_AV(2, 1024, 1, use_mcb=True), DeepVAD_audio(2, 1024, 1), DeepVAD_video(2, 1024, 1)):
        ref = m.state_dict()
        for clone in (pickle.loads(pickle.dumps(m)), copy.deepcopy(m)):
            sd = clone.state_dict()
            assert list(sd.keys()) == list(ref.keys())
            assert all(torch.equal(sd[k], ref[k]) for k in ref)
            assert clone._engines is not m._engines and clone._engines.by_device == {}


def test_host_helpers_match_reference_outputs():
    """packages/models/utils.py:57-162 and packages/utils.py:9-40 (imported by scripts/train_video_net.py:18-19):
    our restatements against outputs of the reference's own functions (tests/golden/ref_helpers.npz,
    tools/make_golden.py:ref_helpers)."""
    import packages.models.utils as mu
    import packages.utils as pu
    from util import golden
    g = golden("ref_helpers.npz")
    t = lambda k: torch.tensor(g[k])  # noqa: E731
    x, r, mu_, lv, y = t("x"), t("r"), t("mu"), t("logvar"), t("y")
    eps = 1e-8

    def close(a, k):
        assert np.allclose(np.asarray(a), g[k], atol=1e-6, rtol=1e-5), k

    close(mu.enumerate_discrete(torch.zeros(3, 7), 4), "enumerate")
    close(mu.onehot(5)(2), "onehot_5_2")
    close(mu.onehot(3)(7), "onehot_3_7")
    close(mu.log_sum_exp(x), "lse")
    close(mu.log_sum_exp(x, 0, torch.mean), "lse_mean0")
    close(mu.binary_cross_entropy_2classes(x, r, (x > 0.5).float(), eps), "bce2")
    close(mu.ikatura_saito_divergence(r, x, eps), "isd")
    for k, v in zip(("elbo0", "elbo1", "elbo2"), mu.elbo(x, r, mu_, lv, eps)):
        close(v, k)
    for k, v in zip(("L0", "L1", "L2"), mu.L_loss(x, r, mu_, lv, eps)):
        close(v, k)
    for k, v in zip(("U0", "U1", "U2", "U3"), mu.U_loss(x, r, mu_, lv, y, eps)):
        close(v, k)
    close(mu.mean_square_error_signal(x, r, x * 0.5), "mse_signal")
    close(mu.mean_square_error_mask(x, r), "mse_mask")
    close(mu.magnitude_spectrum_approxiamation_loss(torch.complex(x, r), torch.complex(r, x), x), "msa")
    vids = [t(f"collate_in{i}") for i in range(3)]
    lens, data, target = pu.my_collate([(v, torch.tensor(float(i % 2)), v.shape[-1]) for i, v in enumerate(vids)])
    assert lens.dtype == torch.int64 and lens.tolist() == g["collate_len"].tolist()
    close(data, "collate_data")
    close(target, "collate_target")


def test_remaining_script_imports_resolve():
    """Names imported at module top by scripts/train_video_net.py:18-19, scripts/reconstruct_dnn_classif.py and
    scripts/visualization_audio.py:16-19 (third-party imports such as h5py / librosa / ffmpeg are the scripts' own)."""
    from packages.models.utils import binary_cross_entropy, binary_cross_entropy_2classes, f1_loss  # noqa: F401
    from packages.utils import count_parameters, my_collate, collate_many2many_video  # noqa: F401
    from packages.processing.stft import stft, istft, stft_pytorch  # noqa: F401
    from packages.processing.target import clean_speech_VAD, clean_speech_IBM, noise_robust_clean_speech_IBM  # noqa: F401
    from packages.visualization import (display_wav_spectro_mask, display_waveplot, display_spectrogram,  # noqa: F401
                                        display_power_spectro, display_multiple_signals, display_multiple_spectro)


@pytest.mark.parametrize("n", [16000, 81920, 70000])
@pytest.mark.parametrize("center", [True, False])
def test_numpy_stft_istft_against_torch(n, center):
    """packages/processing/stft.py:13-99 wraps librosa.core.stft / istft; ours is plain numpy.  Checked against
    torch.stft / torch.istft (the same transform: periodic Hann, reflect centre padding, window-sum-square
    normalisation) and through the analysis -> synthesis round trip."""
    import math
    from packages.processing.stft import stft, istft
    rng = np.random.default_rng(n)
    x = (rng.standard_normal(n) * 0.1).astype(np.float32)
    S = stft(x, 16e3, 64e-3, 'hann', 0.25, center, 'reflect', True)
    padded = math.ceil(n / 16e3 / 64e-3 / 0.25) != int(n / 16e3 / 64e-3 / 0.25)   # the reference's pad-at-end rule
    xp = np.pad(x, (0, 256)) if padded else x
    R = torch.stft(torch.tensor(xp), 1024, 256, window=torch.hann_window(1024), center=center, pad_mode='reflect',
                   return_complex=True).numpy()
    assert S.dtype == np.complex64 and S.shape == R.shape
    assert np.abs(S - R).max() < 1e-5
    if center:
        y = istft(S, 16000, 64e-3, 'hann', 0.25, True, 'float32', max_len=n)
        yr = torch.istft(torch.tensor(R), 1024, 256, window=torch.hann_window(1024), center=True, length=n).numpy()
        assert y.dtype == np.float32 and y.shape == (n,)
        assert np.abs(y - yr).max() < 1e-6 and np.abs(y - x).max() < 1e-6


def test_raw_corpus_listers(tmp_path):
    """packages/dataset/ntcd_timit.py:57-96,193-381 (imported by scripts/create_audio_train_files.py:27 and
    scripts/create_video_train_files_upsampled.py:27).  Expected mappings were checked against the reference's own
    functions on the same synthetic tree in the build container."""
    from packages.dataset.ntcd_timit import kaldi_list, noisy_clean_pair_dict, noisy_speech_dict
    root = str(tmp_path) + '/'
    for split in ('train', 'dev', 'test'):
        for spk in ('01M', '08F'):
            for utt in ('sa1', 'si494'):
                for sub, exts in (('matlab_raw', ('.mat',)), ('kaldi_fMLLR', ('.ark', '.scp'))):
                    d = os.path.join(root, 'ntcd_timit', sub, split, spk)
                    os.makedirs(d, exist_ok=True)
                    for e in exts:
                        open(os.path.join(d, utt + e), 'w').close()
    noisy = 'ntcd_timit/u/drspeech/data/TCDTIMIT/Noisy_TCDTIMIT/'
    sub = noisy_clean_pair_dict(root, 'test', 'subset')
    assert list(sub.items()) == [
        (noisy + 'Babble/-5/volunteers/01M/straightcam/sa1.wav', 'ntcd_timit/Clean/test/01M/sa1.wav'),
        (noisy + 'Babble/-5/volunteers/01M/straightcam/si494.wav', 'ntcd_timit/Clean/test/01M/si494.wav'),
        (noisy + 'Babble/-5/volunteers/08F/straightcam/sa1.wav', 'ntcd_timit/Clean/test/08F/sa1.wav'),
        (noisy + 'Babble/-5/volunteers/08F/straightcam/si494.wav', 'ntcd_timit/Clean/test/08F/si494.wav')]
    full = noisy_clean_pair_dict(root, 'validation')
    assert len(full) == 6 * 3 * 4 and full[noisy + 'White/5/volunteers/08F/straightcam/si494.wav'] == \
        'ntcd_timit/Clean/dev/08F/si494.wav'
    out = noisy_speech_dict(root, 'train', 'subset')
    assert out[noisy + 'Babble/-5/volunteers/01M/straightcam/sa1.wav'] == 'ntcd_timit/Noisy/Babble/-5/train/01M/sa1.wav'
    assert len(noisy_speech_dict(root, 'train')) == 72
    ark, scp = kaldi_list(root, 'test')
    assert ark == ['ntcd_timit/kaldi_fMLLR/test/01M/sa1.ark', 'ntcd_timit/kaldi_fMLLR/test/01M/si494.ark',
                   'ntcd_timit/kaldi_fMLLR/test/08F/sa1.ark', 'ntcd_timit/kaldi_fMLLR/test/08F/si494.ark']
    assert [p[:-4] for p in scp] == [p[:-4] for p in ark]


def test_csr1_pickle_round_trip(tmp_path, capsys):
    from packages.dataset.csr1_wjs0 import read_dataset, write_dataset
    root = str(tmp_path) + '/'
    data = {"x": np.arange(6).reshape(2, 3), "names": ["a", "b"]}
    write_dataset(data, root, 'validation', suffix='frames')
    assert os.path.exists(root + 'CSR-1-WSJ-0/si_dt_05_frames.p')
    back = read_dataset(root, 'validation', suffix='frames')
    assert back["names"] == data["names"] and np.array_equal(back["x"], data["x"])
    assert "data is stored in" in capsys.readouterr().out


def test_legacy_hdf5_datasets(monkeypatch):
    """data_handling.py:51-189: frame, trailing-sequence and block views over one (F, N) / (y, N) array pair."""
    import packages.data_handling as dh
    X = np.arange(3 * 10, dtype=np.float32).reshape(3, 10)
    Y = (np.arange(10, dtype=np.float32) % 2)[None]
    monkeypatch.setattr(dh, "read_h5", lambda path, key: {"X_train": X, "Y_train": Y}[key])
    a = dh.HDF5SpectrogramLabeledFrames("f.h5", "train", 1, 1)
    assert len(a) == 10 and np.array_equal(a[4][0], X[:, 4]) and np.array_equal(a[4][1], Y[:, 4])
    b = dh.HDF5SequenceSpectrogramLabeledFrames("f.h5", "train", 1, 1, seq_length=4)
    d, l, n = b[2]
    assert n == 3 and torch.equal(d, torch.tensor(X[:, :3])) and torch.equal(l, torch.tensor(Y[:, 2:3]))
    d, l, n = b[7]
    assert n == 4 and torch.equal(d, torch.tensor(X[:, 4:8])) and torch.equal(l, torch.tensor(Y[:, 7:8]))
    c = dh.HDF5WholeSequenceSpectrogramLabeledFrames("f.h5", "train", 1, 1, seq_length=4)
    assert len(c) == 3
    d, l, n = c[2]
    assert n == 2 and torch.equal(d, torch.tensor(X[:, 8:])) and torch.equal(l, torch.tensor(Y[:, 8:]))
    assert len(dh.VideoFrames(["01M/sa1", "01M/sa2"], 5)) == 2


def test_threshold_masks_match_reference_outputs():
    """packages/processing/target.py:110-251 against outputs of the reference's own functions
    (tests/golden/ref_target_masks.npz, tools/make_golden.py:ref_target_masks): tables and masks bit-exact."""
    from packages.processing.target import _voiced_unvoiced_split_characteristic, noise_aware_IBM, threshold_IBM
    from util import golden
    g = golden("ref_target_masks.npz")
    voiced, unvoiced = _voiced_unvoiced_split_characteristic(513)
    assert np.array_equal(voiced, g["voiced"]) and np.array_equal(unvoiced, g["unvoiced"])
    speech, noise = noise_aware_IBM(g["X"], g["N"])
    assert np.array_equal(speech, g["speech"]) and np.array_equal(noise, g["noise"])
    assert np.array_equal(threshold_IBM(g["X"]), g["thresh"])
    assert 0.2 < speech.mean() < 0.6  # the fixture is not degenerate
