"""Host side of the audio-only and video-only entry points, without a GPU: the frame accounting of a stream for each
model (avvad.stream.FramePlan), the argument rules of the pipeline and its modality detection, and the sharded
evaluation loop over audio-only and video-only items with a stub in place of the device pipeline."""
import random

import numpy as np
import pytest
import torch

from avvad import engine as E
from avvad import synth
from avvad.evaluate import evaluate_shard, evaluate_sharded
from avvad.pipeline import AVVADPipeline, check_inputs, check_state_dict, modality_lengths, modality_of
from avvad.stream import FramePlan, audio_full_frames, source_index


def _split(total, rng):
    out = []
    while total > 0:
        n = min(total, 1 if rng.random() < 0.3 else rng.randint(1, max(1, total // 3)))
        out.append(n)
        total -= n
    return out


@pytest.mark.parametrize("seed", range(20))
@pytest.mark.parametrize("modality", ["audio", "video"])
def test_frame_plan_single_modality(modality, seed):
    """Ragged pushes of one input: a frame emitted before close is final (its window / source frame has arrived), and
    the frames emitted in all are the offline count of that model."""
    rng = random.Random(seed)
    hears = modality == "audio"
    total_in = rng.randint(1000, 110000) if hears else rng.randint(1, 200)
    T = E.stft_num_frames(total_in) if hears else E.upsampled_length(total_in)
    assert modality_lengths(modality, [total_in] if hears else None, None if hears else [total_in]) == [T]
    plan = FramePlan(audio=hears, video=not hears)
    for n in _split(total_in, rng):
        plan.push(n, 0) if hears else plan.push(0, n)
        k0 = plan.emitted
        c = plan.take(rng.choice([1, 3, 16, 64, 10 ** 6]))
        for k in range(k0, k0 + c):
            if hears:
                assert k * 256 + 1024 <= plan.n_samples, (seed, k)
            else:
                assert source_index(k) <= plan.n_src - 1, (seed, k)
        # before close the audio model waits for whole windows only; the video model's rule does not change at close
        assert plan.ready() == (audio_full_frames(plan.n_samples) if hears else E.upsampled_length(plan.n_src))
    plan.close()
    while not plan.finished():
        assert plan.take(rng.choice([1, 7, 64])) > 0
    assert plan.emitted == plan.total() == T


def test_frame_plan_av_rule_unchanged():
    plan = FramePlan()
    plan.push(20000, 10)
    assert plan.ready() == min(audio_full_frames(20000), E.upsampled_length(10))
    plan.close()
    assert plan.total() == AVVADPipeline.frame_counts([20000], [10])[0]
    with pytest.raises(ValueError):
        FramePlan(audio=False, video=False)


def test_input_rules():
    w, v = torch.zeros(1, 4000), torch.zeros(1, 4, 67, 67, dtype=torch.uint8)
    check_inputs("av", True, w, v, True, torch.zeros(1))
    check_inputs("av", False, w, v, True, None)        # the AV model without MCB ignores per_utterance, as before
    check_inputs("audio", False, w, None)
    check_inputs("video", False, None, v)
    for args in [("audio", w, v), ("audio", None, None), ("video", w, v), ("video", None, None), ("av", w, None),
                 ("av", None, v)]:
        with pytest.raises(ValueError):
            check_inputs(args[0], False, args[1], args[2])
    with pytest.raises(ValueError, match="no MCB"):
        check_inputs("audio", False, w, None, per_utterance=True)
    with pytest.raises(ValueError, match="no MCB"):
        check_inputs("video", False, None, v, mcb_norms_out=torch.zeros(1))


def _sd(kind, **kw):
    return {k: torch.zeros(s, dtype=d) for k, (s, d) in synth.model_spec(kind, hidden=64, **kw).items()}


def test_state_dict_keys_are_checked_before_any_device_work():
    check_state_dict(_sd("audio"), "audio", False, 2, 64, 1)
    check_state_dict(_sd("video", y_dim=513), "video", False, 2, 64, 513)
    check_state_dict(_sd("av", use_mcb=True), "av", True, 2, 64, 1)
    with pytest.raises(KeyError, match="lstm_video"):
        check_state_dict(_sd("audio"), "video", False, 2, 64, 1)
    with pytest.raises(KeyError, match="features"):
        check_state_dict({k: v for k, v in _sd("video").items() if not k.startswith("features.")}, "video", False, 2,
                         64, 1)
    with pytest.raises(ValueError, match="needs"):
        check_state_dict(_sd("audio"), "audio", False, 2, 64, 513)        # head of another y_dim
    with pytest.raises(KeyError, match="mcb"):
        check_state_dict(_sd("av", use_mcb=False), "av", True, 2, 64, 1)  # a concat checkpoint where MCB is expected
    # the constructor rejects a wrong checkpoint, a modality name and missing statistics before it needs a GPU
    mean, std = synth.synth_audio_stats(0)
    with pytest.raises(KeyError):
        AVVADPipeline(_sd("video"), mean, std, hidden=64, modality="audio")
    with pytest.raises(ValueError, match="modality"):
        AVVADPipeline(_sd("audio"), mean, std, hidden=64, modality="speech")
    with pytest.raises(ValueError, match="video_mean"):
        AVVADPipeline(_sd("video"), hidden=64, modality="video")
    with pytest.raises(ValueError, match="audio_mean"):
        AVVADPipeline(_sd("audio"), hidden=64, modality="audio", video_mean=0.0, video_std=1.0)
    with pytest.raises(ValueError, match="upsampled_video"):
        AVVADPipeline(_sd("audio"), mean, std, hidden=64, modality="audio", upsampled_video=True)


def test_modality_of_module_class():
    from packages.models.AV_Net import DeepVAD_AV
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models.Video_Net import DeepVAD_video
    assert modality_of(DeepVAD_audio(1, 16, 1)) == "audio"
    assert modality_of(DeepVAD_video(1, 16, 1)) == "video"
    assert modality_of(DeepVAD_AV(1, 16, 1, use_mcb=False)) == "av"
    with pytest.raises(TypeError):
        modality_of(torch.nn.LSTM(4, 4))


# ---- the evaluation loop over single-modality items, with a stub pipeline -------------------------------------------
class _StubPipeline:
    """infer_host of a single-modality pipeline: the posterior of frame t of an utterance is a fixed function of that
    utterance's own input only, so a wrong row order, a length attached to the wrong utterance or stale staging
    contents change the result."""

    def __init__(self, modality):
        self.modality = modality
        self.video_rate = (E.FPS_NUM, E.FPS_DEN)
        self.calls = []

    def infer_host(self, wave, n_samples, video, n_src, lengths=None, per_utterance=None, t_max=None):
        check_inputs(self.modality, False, wave, video, per_utterance)
        B, T = len(lengths), max(lengths)
        self.calls.append((B, T))
        post = torch.full((B, T, 1), 0.5)
        for b in range(B):
            x = wave[b, : n_samples[b]].double() if wave is not None else video[b, : n_src[b]].double()
            key = float(x.sum()) * 1e-3 + float(x.mean()) * 1e-2
            t = torch.arange(lengths[b], dtype=torch.float64)
            post[b, : lengths[b], 0] = torch.sigmoid(torch.sin(key + 0.1 * t)).float()
        return post, (post > 0.5).int()


def _items(modality, n):
    out = []
    for i in range(n):
        rng = np.random.default_rng(500 + i)
        if modality == "audio":
            out.append((rng.standard_normal(int(rng.integers(2000, 9000))).astype(np.float32), None))
        else:
            out.append((None, rng.integers(0, 256, (int(rng.integers(2, 30)), 67, 67), dtype=np.uint8)))
    return out


@pytest.mark.parametrize("modality", ["audio", "video"])
def test_evaluate_shard_single_modality_items(modality):
    utts = _items(modality, 11)
    one = evaluate_shard(_StubPipeline(modality), utts, batch_size=1, sort_by_length=False)
    pipe = _StubPipeline(modality)
    batched = evaluate_shard(pipe, utts, batch_size=4)
    assert len(pipe.calls) == 3
    T = modality_lengths(modality, [len(w) for w, _ in utts] if modality == "audio" else None,
                         [v.shape[0] for _, v in utts] if modality == "video" else None)
    for (s1, h1), (s2, h2), t in zip(one, batched, T):
        assert s1.shape == (t,) and torch.equal(s1, s2) and torch.equal(h1, h2)
    parts = [evaluate_sharded(_StubPipeline(modality), utts, 3, r, batch_size=2) for r in range(3)]
    assert [p[0] for p in parts] == [0, 4, 8] and parts[-1][1] == 11
    merged = [x for p in parts for x in p[2]]
    assert all(torch.equal(a[0], b[0]) for a, b in zip(merged, one))
    other = "video" if modality == "audio" else "audio"
    with pytest.raises(ValueError, match="item 0"):
        evaluate_shard(_StubPipeline(other), utts)
