"""GPU: AVVADStream against one offline call.  Ragged synthetic utterances ("strong" weights) are streamed through a
few slots in irregular, unaligned blocks of samples and source frames -- slots opened at different times, closed,
reopened with the next utterance, steps in which some slots have no ready frame -- with the peak max|x| and the MCB norm
of the offline call as the per-utterance constants.  Concatenated per utterance, the streamed logits, posteriors and
decisions must be bit-identical to AVVADPipeline.infer_device(per_utterance=True) on the whole utterances, and each
utterance must emit exactly frame_counts frames."""
import random

import numpy as np
import pytest
import torch

from avvad import synth
from avvad.pipeline import AVVADPipeline
from avvad.stream import AVVADStream

pytestmark = pytest.mark.gpu


def _pipeline(use_mcb):
    mean, std = synth.synth_audio_stats(0)
    sd = synth.seeded_state_dict(synth.model_spec("av", use_mcb=use_mcb), 51, "strong")
    if use_mcb:
        sd = synth.calibrate_mcb_bn_(sd, 90)
    return AVVADPipeline(sd, mean, std, synth.VIDEO_MEAN, synth.VIDEO_STD, use_mcb=use_mcb)


def _offline(pipe, utts):
    ns = [len(w) for w, _ in utts]
    nf = [v.shape[0] for _, v in utts]
    B = len(utts)
    wave = torch.zeros(B, max(ns))
    vid = torch.zeros(B, max(nf), 67, 67, dtype=torch.uint8)
    for i, (w, v) in enumerate(utts):
        wave[i, :len(w)] = torch.from_numpy(w)
        vid[i, :v.shape[0]] = torch.from_numpy(v)
    norms = torch.zeros(B, device="cuda") if pipe.use_mcb else None
    lg, post, dec = pipe.infer_device(wave.cuda(), ns, vid.cuda(), nf, per_utterance=True, mcb_norms_out=norms)
    T = AVVADPipeline.frame_counts(ns, nf)
    return [(lg[i, :t], post[i, :t], dec[i, :t]) for i, t in enumerate(T)], T, norms


@pytest.mark.parametrize("use_mcb,slots,max_step", [(True, 3, 64), (False, 4, 16)], ids=["mcb", "concat"])
def test_stream_equals_offline(use_mcb, slots, max_step):
    rng = random.Random(5)
    utts = [(synth.synth_wave(rng.randint(9000, 40000), 70 + i), synth.synth_video_u8(rng.randint(18, 80), 70 + i))
            for i in range(7)]
    pipe = _pipeline(use_mcb)
    ref, T, norms = _offline(pipe, utts)
    norms = norms.tolist() if norms is not None else [None] * len(utts)

    st = AVVADStream(pipe, slots, max_step=max_step)
    queue = list(range(len(utts)))
    live = {}                                        # slot -> [utterance, samples pushed, frames pushed]
    got = {u: [] for u in range(len(utts))}
    mixed_steps = 0
    step_no = 0
    while queue or live:
        # slot s first opens at step 2 s; a freed slot takes the next utterance at once
        for s in range(slots):
            if s not in live and queue and step_no >= 2 * s:
                u = queue.pop(0)
                w, _ = utts[u]
                st.open(s, float(np.abs(w).max()), norms[u])
                live[s] = [u, 0, 0]
        for s, rec in live.items():
            u, a, f = rec
            w, v = utts[u]
            if a < len(w) or f < v.shape[0]:
                na = min(rng.choice([1, 300, 1000, 2500, 5003, 9000]), len(w) - a)
                nv = min(rng.choice([0, 0, 1, 3, 7, 12]), v.shape[0] - f)
                on_dev = rng.random() < 0.5
                wb = torch.from_numpy(w[a:a + na])
                vb = torch.from_numpy(v[f:f + nv])
                st.push(s, wave=wb.cuda() if on_dev else wb, video_u8=(vb.cuda() if on_dev else vb) if nv else None)
                rec[1], rec[2] = a + na, f + nv
                if rec[1] == len(w) and rec[2] == v.shape[0]:
                    st.close(s)
        lg, post, dec, count, frame0 = st.step()
        if any(count[s] == 0 for s in live) and any(count[s] > 0 for s in live):
            mixed_steps += 1
        for s in list(live):
            u = live[s][0]
            c = count[s]
            assert frame0[s] == sum(x[0].shape[0] for x in got[u]), (s, u)
            if c:
                got[u].append((lg[s, :c].clone(), post[s, :c].clone(), dec[s, :c].clone()))
            if st.plans[s] is None:              # flushed: the slot is free again
                del live[s]
        step_no += 1
        assert step_no < 500
    assert mixed_steps > 0, "no step had slots with and without ready frames"
    for u, (rl, rp, rd) in enumerate(ref):
        cl = torch.cat([x[0] for x in got[u]]) if got[u] else rl[:0]
        cp = torch.cat([x[1] for x in got[u]]) if got[u] else rp[:0]
        cd = torch.cat([x[2] for x in got[u]]) if got[u] else rd[:0]
        assert cl.shape[0] == T[u], (u, cl.shape[0], T[u])
        assert torch.equal(cl, rl), f"utterance {u}: streamed logits differ at {int((cl != rl).sum())} frames"
        assert torch.equal(cp, rp) and torch.equal(cd, rd), u
    print(f"use_mcb={use_mcb}: {len(utts)} utterances, {step_no} steps, {mixed_steps} steps with idle slots; "
          f"bit-identical")


def test_stream_errors():
    pipe = _pipeline(True)
    st = AVVADStream(pipe, 2, max_samples=4096, max_frames=8)
    with pytest.raises(ValueError):
        st.push(0, wave=torch.zeros(10))          # not open
    with pytest.raises(ValueError):
        st.open(0, 1.0)                           # MCB needs its norm
    st.open(0, 1.0, 2.0)
    with pytest.raises(ValueError):
        st.push(0, wave=torch.zeros(5000))        # over capacity
    with pytest.raises(ValueError):
        st.push(0, video_u8=torch.zeros(9, 67, 67, dtype=torch.uint8))
    st.close(0)
    with pytest.raises(ValueError):
        st.push(0, wave=torch.zeros(10))          # after close
    lg, post, dec, count, frame0 = st.step()      # nothing ready: no work, and the empty slot is free again
    assert lg.shape[1] == 0 and count == [0, 0]
    assert st.plans[0] is None
    with pytest.raises(ValueError):
        st.close(0)
