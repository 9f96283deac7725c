"""Streaming inference: audio and mouth-ROI frames arrive in blocks, decisions come out for the new frames.

:class:`AVVADStream` keeps a fixed number of slots, one live utterance each, and runs every :meth:`AVVADStream.step`
as one batched call over the slots with ready frames, through the same kernels and weights as
:meth:`avvad.pipeline.AVVADPipeline.infer_device`.  The recurrence carries its state across steps
(:class:`avvad.engine.LstmState`), and every other stage is per frame, so the streamed logits, posteriors and
decisions are bit-identical to one offline ``infer_device(per_utterance=True)`` call on the whole utterances.

Two quantities of the reference look at the whole utterance: the peak normalisation of the waveform
(packages/data_handling.py:441) and the L2 norm of the MCB output (AV_Net.py:117).  A stream cannot know them in
advance, so the caller supplies both when it opens a slot.

:class:`FramePlan` is the frame accounting of one slot: which 62.5 fps output frames are final given the samples and
30 fps source frames seen so far.  It is pure host code.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import engine as E

HOP, NFFT = 256, 1024


def source_index(k: int) -> int:
    """30 fps source frame of 62.5 fps output frame k, unclamped (include/avvad.h, avvad_upsample_index)."""
    return (E.FPS_DEN * (2 * k + 1) - 1) // (2 * E.FPS_NUM)


def audio_full_frames(n_samples: int) -> int:
    """STFT frames whose 1024 samples have all arrived: they never touch the end padding."""
    return (n_samples - NFFT) // HOP + 1 if n_samples >= NFFT else 0


class FramePlan:
    """Frame accounting of one utterance streamed in blocks.

    Before :meth:`close`, frame k is ready when its audio window is complete and k < upsampled_length(F): for
    those k the unclamped source index is at most F - 1, so the frame is exactly the offline one.  After
    :meth:`close`, the frames up to T = min(stft_num_frames(N), upsampled_length(F)) follow, the reference's
    pad-at-end frame included."""

    def __init__(self):
        self.n_samples = 0   # N: samples seen
        self.n_src = 0       # F: source frames seen
        self.emitted = 0     # k: output frames emitted
        self.closed = False

    def push(self, n_samples: int = 0, n_src: int = 0):
        if self.closed:
            raise ValueError("push after close")
        self.n_samples += int(n_samples)
        self.n_src += int(n_src)

    def close(self):
        self.closed = True

    def total(self) -> int:
        """Frames this utterance emits in all (the offline frame count once closed)."""
        return min(E.stft_num_frames(self.n_samples), E.upsampled_length(self.n_src))

    def ready(self) -> int:
        """Frames that may be emitted now, counted from frame 0."""
        if self.closed:
            return self.total()
        return min(audio_full_frames(self.n_samples), E.upsampled_length(self.n_src))

    def take(self, limit: int) -> int:
        """Emit up to `limit` ready frames; returns how many (they start at the previous `emitted`)."""
        n = max(min(self.ready() - self.emitted, limit), 0)
        self.emitted += n
        return n

    def finished(self) -> bool:
        return self.closed and self.emitted >= self.total()


class AVVADStream:
    """Streaming front end of an :class:`~avvad.pipeline.AVVADPipeline` (same weights, same engines).

    ``slots`` utterances live at a time.  Per slot the stream buffers at most ``max_samples`` samples (from the first
    frame not yet emitted on) and ``max_frames`` source frames; a push beyond that raises ``ValueError``.  A step emits
    at most ``max_step`` frames per slot."""

    def __init__(self, pipeline, slots: int, max_samples: int = 16000 * 4, max_frames: int = 128, max_step: int = 64):
        if slots <= 0 or max_step <= 0 or max_samples < NFFT or max_frames <= 0:
            raise ValueError("AVVADStream: bad sizes")
        self.p = pipeline
        self.S, self.max_samples, self.max_frames, self.max_step = slots, max_samples, max_frames, max_step
        dev = pipeline.device
        self.wave = torch.zeros(slots, max_samples, dtype=torch.float32, device=dev)   # samples from k * 256 on
        self.video = torch.zeros(slots, max_frames, 67, 67, dtype=torch.uint8, device=dev)  # frames from src(k) on
        self.n_held = [0] * slots      # samples in `wave`
        self.f_held = [0] * slots      # frames in `video`
        self.f_base = [0] * slots      # source index of video[slot, 0]
        self.plans: List[Optional[FramePlan]] = [None] * slots
        self.peak = torch.ones(slots, dtype=torch.float32, device=dev)
        self.norm = torch.ones(slots, dtype=torch.float32, device=dev)
        self.state = E.LstmState(pipeline.lstm, slots, dev)

    # ---- slot life cycle -----------------------------------------------------------------------------------------
    def open(self, slot: int, peak: float, mcb_norm: Optional[float] = None):
        """Start a new utterance in `slot`.  `peak` = max|x| of the utterance's waveform; `mcb_norm` = L2 norm of its
        MCB output (required with use_mcb), e.g. from ``infer_device(..., per_utterance=True, mcb_norms_out=)``."""
        self._slot(slot)
        if self.p.use_mcb and mcb_norm is None:
            raise ValueError("open: mcb_norm is required when the pipeline fuses with MCB")
        self.plans[slot] = FramePlan()
        self.n_held[slot] = self.f_held[slot] = self.f_base[slot] = 0
        self.peak[slot] = float(peak)
        self.norm[slot] = float(mcb_norm) if mcb_norm is not None else 1.0
        self.state.reset([slot])

    def push(self, slot: int, wave: Optional[torch.Tensor] = None, video_u8: Optional[torch.Tensor] = None):
        """Append samples (1-D f32) and / or source frames ((n, 67, 67) u8), on the host or the device, any sizes."""
        plan = self._live(slot)
        if plan.closed:
            raise ValueError(f"push: slot {slot} is closed")
        n = 0 if wave is None else int(wave.numel())
        f = 0 if video_u8 is None else int(video_u8.shape[0])
        if self.n_held[slot] + n > self.max_samples or self.f_held[slot] + f > self.max_frames:
            raise ValueError(f"push: slot {slot} would buffer more than {self.max_samples} samples or "
                             f"{self.max_frames} frames")
        if n:
            self.wave[slot, self.n_held[slot]:self.n_held[slot] + n].copy_(wave.reshape(-1), non_blocking=True)
        if f:
            assert video_u8.dtype == torch.uint8 and tuple(video_u8.shape[1:]) == (67, 67)
            self.video[slot, self.f_held[slot]:self.f_held[slot] + f].copy_(video_u8, non_blocking=True)
        self.n_held[slot] += n
        self.f_held[slot] += f
        plan.push(n, f)

    def close(self, slot: int):
        """No more input for `slot`: the following steps flush its last frames, then the slot is free."""
        self._live(slot).close()

    # ---- one batched call --------------------------------------------------------------------------------------
    def step(self):
        """Run every slot's ready frames (at most ``max_step`` each) as one batched call.

        Returns (logits, post, dec, count, frame0): device tensors (S, t_step, y_dim), where row s holds
        ``count[s]`` new frames starting at the utterance's frame ``frame0[s]`` (lists of S ints).  Slots without
        ready frames get count 0 and keep their state.  t_step = 0 when no slot has a frame."""
        p, S, dev = self.p, self.S, self.p.device
        frame0 = [pl.emitted if pl is not None else 0 for pl in self.plans]
        count = [pl.take(self.max_step) if pl is not None else 0 for pl in self.plans]
        t = max(count)
        y = p.y_dim
        if t == 0:   # a slot closed after its last frame went out is freed here
            self._consume(count)
            z = torch.zeros(S, 0, y, dtype=torch.float32, device=dev)
            return z, z.clone(), torch.zeros(S, 0, y, dtype=torch.int32, device=dev), count, frame0
        M = S * t
        audio = p._buf("s_audio", (S, t, 513), torch.float32)
        x = p._buf("s_x", (S, t, p.lstm.ld), torch.bfloat16)
        xv = x.view(M, p.lstm.ld)
        # audio: frame j of this step reads wave[s, j * 256:], zero padded past the samples held
        E.frontend_logpower(self.wave, self.n_held, count, t, p.audio_mean, p.audio_std, p.eps, True, out=audio,
                            peaks=self.peak)
        # video: staging frame j = source frame src(k + j), then the stem's identity map (num = den = 1)
        idx = [[(source_index(frame0[s] + j) - self.f_base[s]) if j < count[s] else 0 for j in range(t)]
               for s in range(S)]
        idx_t = torch.tensor(idx, dtype=torch.int64).to(dev, non_blocking=True)
        staged = self.video[torch.arange(S, device=dev).view(S, 1), idx_t]
        if p.use_mcb:
            feat = p._buf("s_feat", (M, 512), torch.float32)
            p.trunk.forward_u8(staged, count, count, t, p.video_mean, p.video_std, p.eps, True, feat=feat, num=1, den=1)
            p.mcb.forward_grouped(audio.view(M, 513), feat, count, t, out_bf16=xv, norms_in=self.norm)
        else:
            x.zero_()
            E.pack_rows_bf16(audio.view(M, 513), xv, 0, False)
            p.trunk.forward_u8(staged, count, count, t, p.video_mean, p.video_std, p.eps, True, feat_bf16=xv,
                               col_off=513, want_f32=False, num=1, den=1)
        logits, post, dec, _ = p.lstm.forward(x, count, want_post=True, want_dec=True, state=self.state)
        self._consume(count)
        return logits, post, dec, count, frame0

    # ---- internals -----------------------------------------------------------------------------------------------
    def _consume(self, count):
        for s, c in enumerate(count):
            plan = self.plans[s]
            if plan is None:
                continue
            if c:
                drop = min(c * HOP, self.n_held[s])
                rest = self.n_held[s] - drop
                if rest:
                    self.wave[s, :rest] = self.wave[s, drop:drop + rest].clone()
                self.n_held[s] = rest
                keep_from = min(source_index(plan.emitted), self.f_base[s] + self.f_held[s]) - self.f_base[s]
                rest = self.f_held[s] - keep_from
                if keep_from and rest:
                    self.video[s, :rest] = self.video[s, keep_from:keep_from + rest].clone()
                self.f_held[s] = rest
                self.f_base[s] += keep_from
            if plan.finished():
                self.plans[s] = None

    def _slot(self, slot: int):
        if not 0 <= slot < self.S:
            raise ValueError(f"slot {slot} out of range [0, {self.S})")

    def _live(self, slot: int) -> FramePlan:
        self._slot(slot)
        plan = self.plans[slot]
        if plan is None:
            raise ValueError(f"slot {slot} is not open")
        return plan
