"""Sharded batch evaluation of a list of utterances (BASELINE config 4): the host side of
``scripts/evaluate_AV_net.py`` (main: 310-340, process_sublist / process_utt: 120-260) on top of the device pipeline.

The reference splits the file list over its devices with ``np.array_split`` and then calls the model ONCE PER
UTTERANCE (``x[None]``, ``v[None]``, ``lengths = [T]``), so the whole-tensor L2 norm of the MCB branch
(``AV_Net.py:117``) is a per-utterance norm there and nothing is ever zero-padded.  Here a rank's shard is processed in
calls of ``batch_size`` utterances with ``per_utterance=True`` (every utterance normalised by its own norm over its
valid frames): the posteriors of an utterance do not depend on which utterances share its call, so the shard may be
sorted by length to keep the collate padding small, and the result of a call is what ``batch_size`` reference calls
return.  No collective: ranks never exchange anything (SURVEY 8e).

The same loop evaluates the audio-only and video-only models (``process_sublist`` of scripts/evaluate_audio_net.py and
evaluate_video_net.py): an item holds the input its pipeline's model reads and None for the other.  Length sorting is
valid there too: those models have no MCB, and their front end or trunk, recurrence and head are all per row, so an
utterance's posteriors never depend on the others in its call."""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .pipeline import AVVADPipeline, modality_lengths
from .sharding import shard_bounds


def plan_calls(frame_counts: Sequence[int], batch_size: int, sort_by_length: bool = True) -> List[List[int]]:
    """Group the positions 0..n-1 of one shard into calls of at most ``batch_size`` utterances.  With
    ``sort_by_length`` the shard is ordered by descending frame count first (stable), so a call pads every utterance
    to a length close to its own; without it the calls are consecutive blocks in list order."""
    if batch_size <= 0:
        raise ValueError("batch_size must be positive")
    n = len(frame_counts)
    order = list(range(n))
    if sort_by_length:
        order.sort(key=lambda i: -int(frame_counts[i]))  # list.sort is stable
    return [order[i:i + batch_size] for i in range(0, n, batch_size)]


def padding_overhead(frame_counts: Sequence[int], calls: Sequence[Sequence[int]]) -> float:
    """padded frames / valid frames - 1 of a call plan (what the trunk computes beyond the valid frames)."""
    valid = sum(int(frame_counts[i]) for c in calls for i in c)
    padded = sum(len(c) * max(int(frame_counts[i]) for i in c) for c in calls if c)
    return padded / valid - 1.0 if valid else 0.0


def evaluate_shard(pipe: AVVADPipeline, utterances: Sequence[Tuple[Optional[np.ndarray], Optional[np.ndarray]]],
                   batch_size: int = 256, sort_by_length: bool = True,
                   sink: Optional[Callable[[int, torch.Tensor, torch.Tensor], None]] = None):
    """utterances: (waveform f32 (N,), ROI frames u8 (F,67,67) at the source rate) per item, host arrays; for the
    audio-only model (waveform, None), for the video-only model (None, frames) -- at the output rate with
    ``pipe.upsampled_video``.  Returns [(y_hat_soft (T,) f32, y_hat_hard (T,) i32)] in list order (the two tensors the
    reference saves per utterance, scripts/evaluate_AV_net.py:238-250) unless ``sink(position, soft, hard)`` is
    given."""
    n = len(utterances)
    modality = getattr(pipe, "modality", "av")
    hears, sees = modality != "video", modality != "audio"
    for i, (w, v) in enumerate(utterances):
        if (w is not None) != hears or (v is not None) != sees:
            raise ValueError(f"evaluate_shard: item {i} must be ({'waveform' if hears else 'None'}, "
                             f"{'frames' if sees else 'None'}) for the {modality!r} model")
    ns = [int(np.asarray(w).shape[-1]) for w, _ in utterances] if hears else None
    nf = [int(np.asarray(v).shape[0]) for _, v in utterances] if sees else None
    T = modality_lengths(modality, ns, nf, getattr(pipe, "video_rate", None) or (25, 12))
    out: List = [None] * n
    wave_p = vid_p = None  # flat pinned staging buffers, grow-only; a call views them as (B, n_max) / (B, f_max, 67, 67)
    pin = torch.cuda.is_available()  # (the host-logic tests drive this loop with a stub pipeline on a CPU box)
    for call in plan_calls(T, batch_size, sort_by_length):
        B = len(call)
        w_call = v_call = None
        if hears:
            n_max = max(ns[i] for i in call)
            if wave_p is None or wave_p.numel() < B * n_max:
                wave_p = torch.empty(B * n_max, dtype=torch.float32, pin_memory=pin)
            w_call = wave_p[: B * n_max].view(B, n_max)
            w_call.zero_()  # not required (the kernels bound every read by n_samples); keeps stale samples out of the upload
        if sees:
            f_max = max(nf[i] for i in call)
            if vid_p is None or vid_p.numel() < B * f_max * 4489:
                vid_p = torch.empty(B * f_max * 4489, dtype=torch.uint8, pin_memory=pin)
            v_call = vid_p[: B * f_max * 4489].view(B, f_max, 67, 67)
        for k, i in enumerate(call):
            w, v = utterances[i]
            if hears:
                w_call[k, : ns[i]] = torch.as_tensor(np.asarray(w, dtype=np.float32).reshape(-1))
            if sees:
                v_call[k, : nf[i]] = torch.as_tensor(np.asarray(v, dtype=np.uint8).reshape(nf[i], 67, 67))
        lens = [T[i] for i in call]
        post, dec = pipe.infer_host(w_call, [ns[i] for i in call] if hears else None, v_call,
                                    [nf[i] for i in call] if sees else None, lengths=lens,
                                    per_utterance=True if modality == "av" else None)
        for k, i in enumerate(call):
            soft = post[k, : T[i], 0].clone() if post.shape[-1] == 1 else post[k, : T[i]].clone()
            hard = dec[k, : T[i], 0].clone() if dec.shape[-1] == 1 else dec[k, : T[i]].clone()
            if sink is not None:
                sink(i, soft, hard)
            else:
                out[i] = (soft, hard)
    return None if sink is not None else out


def evaluate_sharded(pipe: AVVADPipeline, utterances: Sequence[Tuple[Optional[np.ndarray], Optional[np.ndarray]]],
                     world_size: int,
                     rank: int, batch_size: int = 256, sort_by_length: bool = True):
    """This rank's contiguous block of the list (``np.array_split`` partition, scripts/evaluate_AV_net.py:329-332).
    Returns (start, stop, results of utterances[start:stop])."""
    a, b = shard_bounds(len(utterances), world_size, rank)
    return a, b, evaluate_shard(pipe, utterances[a:b], batch_size, sort_by_length)
