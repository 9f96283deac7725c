"""Frame accounting of the streaming front end (avvad.stream.FramePlan), on the host: over random block splits of the
samples and source frames, a streamed utterance emits exactly the offline frames, never one before its inputs are
final, and stages exactly the source frames of the offline 30 -> 62.5 fps index map."""
import random

import pytest

from avvad import engine as E
from avvad.stream import FramePlan, audio_full_frames, source_index
from oracle import video as OV


def test_unclamped_source_index_stays_inside_the_source():
    """For every k < upsampled_length(F) the unclamped source index is at most F - 1, so a frame emitted as soon as
    k < upsampled_length(F) never uses the clamp a later frame could change."""
    for F in range(1, 3000):
        n = E.upsampled_length(F)
        assert n == OV.upsampled_length(F)
        assert source_index(n - 1) <= F - 1, F


def _split(total, rng, small):
    out = []
    while total > 0:
        n = min(total, 1 if small and rng.random() < 0.3 else rng.randint(1, max(1, total // 3)))
        out.append(n)
        total -= n
    return out


@pytest.mark.parametrize("seed", range(40))
def test_random_block_splits(seed):
    rng = random.Random(seed)
    N = rng.randint(1000, 110000)
    F = rng.randint(1, 200)
    T = min(E.stft_num_frames(N), E.upsampled_length(F))
    index = OV.upsample_index(F, T).tolist() if T else []
    a = _split(N, rng, seed % 2 == 0)
    v = _split(F, rng, seed % 3 == 0)
    # interleave: video ahead of audio for some seeds, behind for others
    ahead = seed % 4
    events = []
    ia = iv = 0
    while ia < len(a) or iv < len(v):
        pick_video = iv < len(v) and (ia >= len(a) or (rng.random() < (0.8 if ahead == 0 else 0.2 if ahead == 1 else 0.5)))
        if pick_video:
            events.append((0, v[iv]))
            iv += 1
        else:
            events.append((a[ia], 0))
            ia += 1
    plan = FramePlan()
    staged = []
    for ns, nf in events:
        plan.push(ns, nf)
        k0 = plan.emitted
        c = plan.take(rng.choice([1, 3, 16, 64, 10 ** 6]))
        for k in range(k0, k0 + c):
            # inputs final: the whole 1024-sample window has arrived, and the source frame exists
            assert k * 256 + 1024 <= plan.n_samples, (seed, k)
            assert source_index(k) <= plan.n_src - 1, (seed, k)
            staged.append(source_index(k))
    plan.close()
    with pytest.raises(ValueError):
        plan.push(1, 0)
    while not plan.finished():
        k0 = plan.emitted
        c = plan.take(rng.choice([1, 7, 64]))
        assert c > 0
        staged += [source_index(k) for k in range(k0, k0 + c)]
    assert plan.emitted == T
    assert staged == index


def test_audio_full_frames():
    assert audio_full_frames(1023) == 0
    assert audio_full_frames(1024) == 1
    assert audio_full_frames(1279) == 1
    assert audio_full_frames(1280) == 2
    for N in range(1024, 20000, 97):   # full frames never exceed the offline count
        assert audio_full_frames(N) <= E.stft_num_frames(N)
