"""End-to-end AV-VAD inference pipeline: raw 16 kHz waveforms + 30 fps mouth-ROI frames in, frame
posteriors / decisions out, everything between on the GPU (SURVEY §8a rows A1-A4, U, V1-V2, F1-F3,
R1, H1-H2; §8f row 2 "on-device batching front end").

This is the public call a user makes for batched inference (the reference has only a B=1,
CPU-STFT evaluation loop: scripts/evaluate_AV_net.py:141-250); the reference-compatible modules in
``packages.models`` share the same engines.
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Sequence

import torch

from . import engine as E
from . import lib as L


class AVVADPipeline:
    def __init__(self, state_dict: Dict[str, torch.Tensor], audio_mean, audio_std, video_mean: float,
                 video_std: float, use_mcb=True, y_dim=1, hidden=1024, layers=2, eps=1e-8, device="cuda"):
        L.require_cuda()
        self.device = torch.device(device)
        self.use_mcb, self.eps, self.y_dim = use_mcb, float(eps), y_dim
        self.audio_mean = torch.as_tensor(audio_mean, dtype=torch.float32).reshape(-1).to(self.device)
        self.audio_std = torch.as_tensor(audio_std, dtype=torch.float32).reshape(-1).to(self.device)
        self.video_mean, self.video_std = float(video_mean), float(video_std)
        with torch.cuda.device(self.device):
            self.trunk = E.ResNet18Trunk()
            self.trunk.load(state_dict, self.device)
            in_size = 1024 if use_mcb else 1025
            self.lstm = E.Lstm(layers, in_size, hidden, y_dim)
            self.lstm.load(state_dict, self.device, "lstm_merged", "vad_merged")
            self.mcb = None
            if use_mcb:
                self.mcb = E.Mcb()
                self.mcb.load(state_dict, self.device, eps)
        self._bufs = {}
        self.piece = int(os.environ.get("AVVAD_PIECE", "64"))  # utterances per video piece (upload / trunk granularity)
        self.fuse_gather = True    # u8 video: gather + standardise inside the stem (False: separate fp32 gather)
        # Optional: run the trunk on the 30 fps SOURCE frames and gather the 512-d features to 62.5 fps.  The eval-mode
        # trunk is a pure per-frame function and the upsampled sequence only duplicates frames, so the result is
        # bit-identical with 2.09x less convolution work.  Off by default: the headline benchmark keeps the
        # reference's order (every 62.5 fps frame through the ResNet).
        self.dedup_video = False
        # MCB L2 norm per utterance instead of per call: a batched call == one reference call per utterance
        # (scripts/evaluate_AV_net.py); see infer_device
        self.per_utterance = False
        self._feat_pad = None
        self._copy_stream = None
        self._events = []

    def _buf(self, name, shape, dtype):
        """Grow-only device scratch: a call with a smaller shape (another t_max / batch) gets a view of the same storage."""
        n = 1
        for d in shape:
            n *= int(d)
        t = self._bufs.get(name)
        if t is None or t.numel() < n or t.dtype != dtype:
            t = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            self._bufs[name] = t
        return t[:n].view(shape)

    @staticmethod
    def frame_counts(n_samples: Sequence[int], n_src: Sequence[int]):
        """T_b = min(STFT frames, upsampled video frames) (packages/data_handling.py:483-486)."""
        return [min(E.stft_num_frames(n), E.upsampled_length(f)) for n, f in zip(n_samples, n_src)]

    def infer_device(self, wave: torch.Tensor, n_samples, video_u8: torch.Tensor, n_src, lengths=None,
                     t_max: Optional[int] = None, _video_ready=None, _wave_ready=None,
                     per_utterance: Optional[bool] = None, mcb_norms_out: Optional[torch.Tensor] = None):
        """wave (B,N) f32 and video (B,F,67,67) u8/f32 already on the device.
        Returns (logits, posteriors, decisions), each (B,t_max,y_dim) on the device.

        ``per_utterance`` (default: ``self.per_utterance``): normalise every utterance's MCB output by its own L2 norm
        over its valid frames, so the batched call returns what B separate forward calls of the reference return --
        the semantics of scripts/evaluate_AV_net.py:186-236, which calls the model once per utterance.  Off: one norm
        over the whole padded (B,T,1024) tensor of the call (AV_Net.py:117 for a batched call, the training scripts).
        ``mcb_norms_out`` (f32 (B,) on the device, with ``per_utterance`` and ``use_mcb``): receives the norms used --
        the constants :class:`avvad.stream.AVVADStream` needs to stream these utterances.

        The video branch runs in pieces of ``self.piece`` utterances (frames of an utterance are independent for
        the trunk); ``_video_ready[k]`` / ``_wave_ready`` are optional CUDA events the current stream waits on
        before touching piece k / the waveforms (used by :meth:`infer_host` to overlap the uploads)."""
        B = wave.shape[0]
        if lengths is None:
            lengths = self.frame_counts(n_samples, n_src)
        if t_max is None:
            t_max = max(lengths)
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        lens = E._i32(lengths, dev)
        ns, nsrc = E._i32(n_samples, dev), E._i32(n_src, dev)
        M = B * t_max
        audio = self._buf("audio", (B, t_max, 513), torch.float32)
        x = self._buf("x", (B, t_max, self.lstm.ld), torch.bfloat16)
        xv = x.view(M, self.lstm.ld)
        feat = self._buf("feat", (M, 512), torch.float32) if self.use_mcb else None
        if not self.use_mcb:
            x.zero_()
        P = max(1, min(self.piece, B))
        fused = self.fuse_gather and video_u8.dtype == torch.uint8
        frames = None if fused else self._buf("frames", (P, t_max, 67, 67), torch.float32)

        def front_end():
            if _wave_ready is not None:
                cur.wait_event(_wave_ready)
            E.frontend_logpower(wave, ns, lens, t_max, self.audio_mean, self.audio_std, self.eps, True, out=audio)
            if not self.use_mcb:
                E.pack_rows_bf16(audio.view(M, 513), xv, 0, False)

        if _wave_ready is None:
            front_end()
        for k, b0 in enumerate(range(0, B, P)):
            b1 = min(B, b0 + P)
            if _video_ready is not None:
                cur.wait_event(_video_ready[k])
            m0, m1 = b0 * t_max, b1 * t_max
            if fused and self.dedup_video:
                Fm = video_u8.shape[1]
                if self._feat_pad is None:  # trunk feature of the collate zero frame (input independent)
                    z = torch.zeros(1, 1, 67, 67, dtype=torch.uint8, device=dev)
                    self._feat_pad = self.trunk.forward_u8(z, [0], [0], 1, self.video_mean, self.video_std, self.eps,
                                                           True, num=1, den=1).clone()
                fs = self._buf("feat_src", (P * Fm, 512), torch.float32)[: (b1 - b0) * Fm]
                self.trunk.forward_u8(video_u8[b0:b1], nsrc[b0:b1], nsrc[b0:b1], Fm, self.video_mean, self.video_std,
                                      self.eps, True, feat=fs, num=1, den=1)
                E.feature_gather(fs.view(b1 - b0, Fm, 512), self._feat_pad, nsrc[b0:b1], lens[b0:b1], t_max,
                                 out_f32=feat[m0:m1] if self.use_mcb else None,
                                 out_bf16=None if self.use_mcb else xv[m0:m1], col_off=513)
            elif fused:  # gather + standardise + collate padding inside the stem kernel
                kw = dict(feat=feat[m0:m1]) if self.use_mcb else dict(feat_bf16=xv[m0:m1], col_off=513, want_f32=False)
                self.trunk.forward_u8(video_u8[b0:b1], nsrc[b0:b1], lens[b0:b1], t_max, self.video_mean,
                                      self.video_std, self.eps, True, **kw)
            else:
                fr = frames[: b1 - b0]
                E.upsample_gather(video_u8[b0:b1], nsrc[b0:b1], lens[b0:b1], t_max, self.video_mean, self.video_std,
                                  self.eps, True, out=fr)
                if self.use_mcb:
                    self.trunk.forward(fr.view(m1 - m0, 67, 67), feat=feat[m0:m1])
                else:
                    self.trunk.forward(fr.view(m1 - m0, 67, 67), feat_bf16=xv[m0:m1], col_off=513, want_f32=False)
            if k == 0 and _wave_ready is not None:
                front_end()  # the waveforms arrive behind the first video piece
        if self.use_mcb:
            if self.per_utterance if per_utterance is None else per_utterance:
                self.mcb.forward_grouped(audio.view(M, 513), feat, lens, t_max, out_bf16=xv, norms_out=mcb_norms_out)
            else:
                if mcb_norms_out is not None:
                    raise ValueError("mcb_norms_out needs per_utterance=True")
                self.mcb.forward(audio.view(M, 513), feat, out_bf16=xv)
        logits, post, dec, _ = self.lstm.forward(x, lens, want_post=True, want_dec=True)
        return logits, post, dec

    def infer_host(self, wave_pinned: torch.Tensor, n_samples, video_pinned: torch.Tensor, n_src, lengths=None,
                   t_max: Optional[int] = None, per_utterance: Optional[bool] = None):
        """Host (pinned) buffers in, host posteriors/decisions out.  The uploads run on a copy stream -- first video
        piece, waveforms, remaining video pieces -- while the current stream computes piece by piece, so only the
        first piece's upload is exposed; the D2H read-back is inside the call (this is what bench.py's `e2e` times)."""
        dev = self.device
        B = wave_pinned.shape[0]
        w = self._buf("wave_dev", tuple(wave_pinned.shape), wave_pinned.dtype)
        v = self._buf("video_dev", tuple(video_pinned.shape), video_pinned.dtype)
        cur = torch.cuda.current_stream(dev)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        cs = self._copy_stream
        P = max(1, min(self.piece, B))
        n_pieces = (B + P - 1) // P
        while len(self._events) < n_pieces + 1:
            self._events.append(torch.cuda.Event())
        ew, ev = self._events[0], self._events[1:n_pieces + 1]
        cs.wait_stream(cur)  # earlier consumers of the staging buffers
        with torch.cuda.stream(cs):
            for k, b0 in enumerate(range(0, B, P)):
                b1 = min(B, b0 + P)
                v[b0:b1].copy_(video_pinned[b0:b1], non_blocking=True)
                ev[k].record(cs)
                if k == 0:
                    w.copy_(wave_pinned, non_blocking=True)
                    ew.record(cs)
        _, post, dec = self.infer_device(w, n_samples, v, n_src, lengths=lengths, t_max=t_max, _video_ready=ev,
                                         _wave_ready=ew, per_utterance=per_utterance)
        n_out = post.numel()
        hp = self._bufs.get("post_host")
        if hp is None or hp.numel() < n_out:  # pinned read-back buffers, grow-only
            self._bufs["post_host"] = torch.empty(n_out, dtype=post.dtype, pin_memory=True)
            self._bufs["dec_host"] = torch.empty(n_out, dtype=dec.dtype, pin_memory=True)
        hp = self._bufs["post_host"][:n_out].view(post.shape)
        hd = self._bufs["dec_host"][:n_out].view(dec.shape)
        hp.copy_(post, non_blocking=True)
        hd.copy_(dec, non_blocking=True)
        cur.synchronize()
        return hp, hd
