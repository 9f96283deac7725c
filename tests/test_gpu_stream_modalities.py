"""GPU: AVVADStream on audio-only and video-only pipelines against one offline call.  Ragged synthetic utterances
("strong" weights) are streamed through a few slots in irregular blocks -- slots opened at different steps, closed,
reused for the next utterance, steps in which some slots have no ready frame -- at 1, 7, 16 and 64 frames per step.
Concatenated per utterance, the streamed logits, posteriors and decisions must be bit-identical to
AVVADPipeline.infer_device on the whole utterances.  The audio stream divides by the given peaks (normalise 2), the
offline call by max|x| of each utterance (normalise 1)."""
import random

import numpy as np
import pytest
import torch

from avvad import synth
from avvad.pipeline import AVVADPipeline
from avvad.stream import AVVADStream

pytestmark = pytest.mark.gpu

_PIPES = {}


def _pipeline(modality):
    if modality not in _PIPES:
        sd = synth.seeded_state_dict(synth.model_spec(modality), 52, "strong")
        mean, std = synth.synth_audio_stats(0)
        if modality == "audio":
            _PIPES[modality] = AVVADPipeline(sd, mean, std, modality="audio")
        else:
            _PIPES[modality] = AVVADPipeline(sd, video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD,
                                             modality="video")
    return _PIPES[modality]


def _utterances(modality, rng, n):
    if modality == "audio":
        return [synth.synth_wave(rng.randint(9000, 30000), 80 + i) for i in range(n)]
    return [synth.synth_video_u8(rng.randint(14, 50), 80 + i) for i in range(n)]


def _offline(pipe, utts):
    B = len(utts)
    if pipe.modality == "audio":
        ns = [len(w) for w in utts]
        wave = torch.zeros(B, max(ns))
        for i, w in enumerate(utts):
            wave[i, :len(w)] = torch.from_numpy(w)
        lg, post, dec = pipe.infer_device(wave.cuda(), ns, None, None)
        T = pipe.lengths_of(ns, None)
    else:
        nf = [v.shape[0] for v in utts]
        vid = torch.zeros(B, max(nf), 67, 67, dtype=torch.uint8)
        for i, v in enumerate(utts):
            vid[i, :v.shape[0]] = torch.from_numpy(v)
        lg, post, dec = pipe.infer_device(None, None, vid.cuda(), nf)
        T = pipe.lengths_of(None, nf)
    return [(lg[i, :t].clone(), post[i, :t].clone(), dec[i, :t].clone()) for i, t in enumerate(T)], T


@pytest.mark.parametrize("max_step", [1, 7, 16, 64])
@pytest.mark.parametrize("modality", ["audio", "video"])
def test_single_modality_stream_equals_offline(modality, max_step):
    rng = random.Random(max_step)
    utts = _utterances(modality, rng, 5)
    pipe = _pipeline(modality)
    ref, T = _offline(pipe, utts)
    slots = 3
    st = AVVADStream(pipe, slots, max_samples=16000, max_frames=40, max_step=max_step)
    assert (st.wave is None) == (modality == "video") and (st.video is None) == (modality == "audio")
    queue = list(range(len(utts)))
    live = {}                                   # slot -> [utterance, input pushed, step it opened]
    got = {u: [] for u in range(len(utts))}
    opened = mixed_steps = step_no = 0
    while queue or live:
        # slot s first opens at step 3 s; a freed slot takes the next utterance at once.  A slot's first input
        # arrives one step after it opened, so that step has a live slot without frames.
        for s in range(slots):
            if s not in live and queue and step_no >= 3 * s:
                u = queue.pop(0)
                st.open(s, float(np.abs(utts[u]).max()) if modality == "audio" else None)
                live[s] = [u, 0, step_no]
                opened += 1
        for s, rec in live.items():
            u, a, opened_at = rec
            x = utts[u]
            if a < len(x) and not st.plans[s].closed and step_no > opened_at:
                if modality == "audio":
                    room = st.max_samples - st.n_held[s]
                    n = min(rng.choice([0, 1, 300, 1000, 2500, 5003]), len(x) - a, room)
                else:
                    room = st.max_frames - st.f_held[s]
                    n = min(rng.choice([0, 0, 1, 3, 7, 12]), len(x) - a, room)
                blk = torch.from_numpy(x[a:a + n])
                blk = blk.cuda() if rng.random() < 0.5 else blk
                if n:
                    st.push(s, **({"wave": blk} if modality == "audio" else {"video_u8": blk}))
                rec[1] = a + n
            if rec[1] == len(x) and not st.plans[s].closed:
                st.close(s)
        lg, post, dec, count, frame0 = st.step()
        if any(count[s] == 0 for s in live) and any(count[s] > 0 for s in live):
            mixed_steps += 1
        for s in list(live):
            u = live[s][0]
            c = count[s]
            assert frame0[s] == sum(x[0].shape[0] for x in got[u]), (s, u)
            assert c <= max_step
            if c:
                got[u].append((lg[s, :c].clone(), post[s, :c].clone(), dec[s, :c].clone()))
            if st.plans[s] is None:             # flushed: the slot is free again
                del live[s]
        step_no += 1
        assert step_no < 3000
    assert mixed_steps > 0, "no step had slots with and without ready frames"
    assert opened > slots, "no slot was reused"
    for u, (rl, rp, rd) in enumerate(ref):
        cl = torch.cat([x[0] for x in got[u]])
        cp = torch.cat([x[1] for x in got[u]])
        cd = torch.cat([x[2] for x in got[u]])
        assert cl.shape[0] == T[u], (u, cl.shape[0], T[u])
        assert torch.equal(cl, rl), f"utterance {u}: streamed logits differ at {int((cl != rl).sum())} frames"
        assert torch.equal(cp, rp) and torch.equal(cd, rd), u
    print(f"{modality}, {max_step} frames per step: {len(utts)} utterances, {step_no} steps, {mixed_steps} steps with "
          f"idle slots; bit-identical")


def test_single_modality_stream_errors():
    sa = AVVADStream(_pipeline("audio"), 2)
    with pytest.raises(ValueError, match="peak"):
        sa.open(0)                                 # the audio model needs the utterance's peak
    sa.open(0, 0.5)
    with pytest.raises(ValueError, match="no video"):
        sa.push(0, video_u8=torch.zeros(2, 67, 67, dtype=torch.uint8))
    sv = AVVADStream(_pipeline("video"), 2)
    with pytest.raises(ValueError, match="no audio"):
        sv.open(0, 0.5)
    sv.open(0)
    with pytest.raises(ValueError, match="no audio"):
        sv.push(0, wave=torch.zeros(100))
    sd = synth.seeded_state_dict(synth.model_spec("video"), 1)
    up = AVVADPipeline(sd, video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD, modality="video",
                       upsampled_video=True)
    with pytest.raises(ValueError, match="upsampled"):
        AVVADStream(up, 2)
