"""End-to-end VAD inference pipeline: raw 16 kHz waveforms and / or 30 fps mouth-ROI frames in, frame posteriors /
decisions out, everything between on the GPU (SURVEY §8a rows A1-A4, U, V1-V2, F1-F3, R1, H1-H2; §8f row 2 "on-device
batching front end").

This is the public call a user makes for batched inference (the reference has only a B=1, CPU-STFT evaluation loop per
model: scripts/evaluate_AV_net.py:141-250, evaluate_audio_net.py, evaluate_video_net.py); the reference-compatible
modules in ``packages.models`` share the same engines.  One pipeline serves one of the three models (``modality``):

- ``"av"``    DeepVAD_AV: front end + trunk, fused by MCB or concatenation -> LSTM -> head;
- ``"audio"`` DeepVAD_audio: front end written straight into the LSTM's bf16 operand -> LSTM -> head;
- ``"video"`` DeepVAD_video: trunk written straight into the LSTM's bf16 operand -> LSTM -> head.
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Sequence

import torch

from . import engine as E
from . import lib as L

MODALITIES = ("av", "audio", "video")
# modality -> (LSTM key, head key, trunk needed)
_KEYS = {"av": ("lstm_merged", "vad_merged", True), "audio": ("lstm_audio", "vad_audio", False),
         "video": ("lstm_video", "vad_video", True)}


def lstm_input_size(modality: str, use_mcb: bool) -> int:
    if modality == "av":
        return 1024 if use_mcb else 1025
    return {"audio": 513, "video": 512}[modality]


def check_state_dict(sd, modality: str, use_mcb: bool, layers: int, hidden: int, y_dim: int):
    """The keys and shapes one modality's engines load (a checkpoint of another model fails here, not in a kernel)."""
    lstm, head, trunk = _KEYS[modality]
    need = {f"{lstm}.{k}_l{l}": None for l in range(layers) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")}
    need[f"{lstm}.weight_ih_l0"] = (4 * hidden, lstm_input_size(modality, use_mcb))
    need[f"{lstm}.weight_hh_l0"] = (4 * hidden, hidden)
    need[f"{head}.weight"] = (y_dim, hidden)
    need[f"{head}.bias"] = None
    if trunk:
        need.update({f"features.{c}.weight": None for c, _ in E.RESNET_LAYER_KEYS})
    if modality == "av" and use_mcb:
        need.update({k: None for k in ("mcb.sketch1.h", "mcb.sketch2.h", "mcb_bn.weight", "mcb_bn.running_var")})
    missing = [k for k in need if k not in sd]
    if missing:
        raise KeyError(f"state_dict of a {modality!r} model (use_mcb={use_mcb}) lacks {len(missing)} keys, "
                       f"e.g. {missing[:3]}; keys present start with {sorted({k.split('.')[0] for k in sd})}")
    for k, shape in need.items():
        if shape is not None and tuple(sd[k].shape) != shape:
            raise ValueError(f"state_dict[{k!r}] has shape {tuple(sd[k].shape)}, a {modality!r} model with hidden="
                             f"{hidden}, y_dim={y_dim}, use_mcb={use_mcb} needs {shape}")


def modality_of(module) -> str:
    """'av', 'audio' or 'video' for a DeepVAD_AV / DeepVAD_audio / DeepVAD_video module (or a subclass)."""
    from packages.models.AV_Net import DeepVAD_AV
    from packages.models.Audio_Net import DeepVAD_audio
    from packages.models.Video_Net import DeepVAD_video

    for cls, m in ((DeepVAD_AV, "av"), (DeepVAD_audio, "audio"), (DeepVAD_video, "video")):
        if isinstance(module, cls):
            return m
    raise TypeError(f"modality_of: {type(module).__name__} is none of DeepVAD_AV, DeepVAD_audio, DeepVAD_video")


def check_inputs(modality: str, use_mcb: bool, wave, video, per_utterance=None, mcb_norms_out=None):
    """Argument rules of infer_device / infer_host: the inputs a modality reads are given, the others are None, and the
    MCB options need an MCB."""
    hears, sees = modality in ("av", "audio"), modality in ("av", "video")
    for name, x, used in (("wave", wave, hears), ("video", video, sees)):
        if used and x is None:
            raise ValueError(f"{name} is required: the {modality!r} model reads it")
        if not used and x is not None:
            raise ValueError(f"{name} must be None: the {modality!r} model does not read it")
    if modality != "av":   # (the AV model without MCB ignores both, as it always has)
        if per_utterance:
            raise ValueError(f"per_utterance applies to the MCB norm; the {modality!r} model has no MCB, and its "
                             "utterances never share anything within a call")
        if mcb_norms_out is not None:
            raise ValueError(f"mcb_norms_out: the {modality!r} model has no MCB")


class AVVADPipeline:
    def __init__(self, state_dict: Dict[str, torch.Tensor], audio_mean=None, audio_std=None,
                 video_mean: Optional[float] = None, video_std: Optional[float] = None, use_mcb=True, y_dim=1,
                 hidden=1024, layers=2, eps=1e-8, device="cuda", modality="av", upsampled_video=False):
        """``modality`` "av" (DeepVAD_AV, keys ``lstm_merged`` / ``vad_merged``), "audio" (DeepVAD_audio, keys
        ``lstm_audio`` / ``vad_audio``; the video statistics are not used) or "video" (DeepVAD_video, keys
        ``features``, ``lstm_video`` / ``vad_video``; the audio statistics are not used).  ``use_mcb`` only applies to
        "av".  ``upsampled_video`` ("video" only): the frames are already at the 62.5 fps output rate, as
        scripts/evaluate_video_net.py reads them from *_upsampled.h5 (identity frame map, T = F)."""
        if modality not in MODALITIES:
            raise ValueError(f"modality must be one of {MODALITIES}, got {modality!r}")
        if upsampled_video and modality != "video":
            raise ValueError("upsampled_video applies to the 'video' model only")
        use_mcb = bool(use_mcb) and modality == "av"
        if modality != "video" and (audio_mean is None or audio_std is None):
            raise ValueError(f"audio_mean and audio_std are required by the {modality!r} model")
        if modality != "audio" and (video_mean is None or video_std is None):
            raise ValueError(f"video_mean and video_std are required by the {modality!r} model")
        check_state_dict(state_dict, modality, use_mcb, layers, hidden, y_dim)
        L.require_cuda()
        self.modality, self.upsampled_video = modality, bool(upsampled_video)
        self.device = torch.device(device)
        self.use_mcb, self.eps, self.y_dim = use_mcb, float(eps), y_dim
        self.audio_mean = self.audio_std = None
        if modality != "video":
            self.audio_mean = torch.as_tensor(audio_mean, dtype=torch.float32).reshape(-1).to(self.device)
            self.audio_std = torch.as_tensor(audio_std, dtype=torch.float32).reshape(-1).to(self.device)
        self.video_mean = float(video_mean) if video_mean is not None else None
        self.video_std = float(video_std) if video_std is not None else None
        lstm_key, head_key, has_trunk = _KEYS[modality]
        with torch.cuda.device(self.device):
            self.trunk = None
            if has_trunk:
                self.trunk = E.ResNet18Trunk()
                self.trunk.load(state_dict, self.device)
            self.lstm = E.Lstm(layers, lstm_input_size(modality, use_mcb), hidden, y_dim)
            self.lstm.load(state_dict, self.device, lstm_key, head_key)
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

    @classmethod
    def from_module(cls, model, audio_mean=None, audio_std=None, video_mean=None, video_std=None, device=None,
                    **kw):
        """Pipeline of a DeepVAD_AV / DeepVAD_audio / DeepVAD_video module: the modality from its class, sizes, MCB and
        eps from its attributes, the weights from its (nn.DataParallel replica aware) state dict.  ``device``: the
        module's device if it is on a GPU, else cuda.  Other keywords go to the constructor."""
        from packages.models._engine import full_state_dict

        modality = modality_of(model)
        sd = {k: v.detach() for k, v in full_state_dict(model).items()}
        if device is None:
            devs = {v.device for v in sd.values() if v.is_cuda}
            device = devs.pop() if len(devs) == 1 else "cuda"
        return cls(sd, audio_mean, audio_std, video_mean, video_std, use_mcb=getattr(model, "use_mcb", False),
                   y_dim=model.y_dim, hidden=model.lstm_hidden_size, layers=model.lstm_layers,
                   eps=getattr(model, "eps", 1e-8), device=device, modality=modality, **kw)

    @property
    def hears(self) -> bool:
        """The model reads the waveform."""
        return self.modality != "video"

    @property
    def sees(self) -> bool:
        """The model reads the mouth-ROI frames."""
        return self.modality != "audio"

    @property
    def video_rate(self):
        """(num, den) of the video frame map: 62.5 / 30 fps, or the identity for already upsampled frames."""
        return (1, 1) if self.upsampled_video else (E.FPS_NUM, E.FPS_DEN)

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

    def lengths_of(self, n_samples: Optional[Sequence[int]], n_src: Optional[Sequence[int]]):
        """Frame count of every utterance for this pipeline's model: :meth:`frame_counts` for "av",
        stft_num_frames(N) for "audio", upsampled_length(F) (F for ``upsampled_video``) for "video"."""
        return modality_lengths(self.modality, n_samples, n_src, self.video_rate)

    def infer_device(self, wave: Optional[torch.Tensor], n_samples, video_u8: Optional[torch.Tensor], n_src,
                     lengths=None, t_max: Optional[int] = None, _video_ready=None, _wave_ready=None,
                     per_utterance: Optional[bool] = None, mcb_norms_out: Optional[torch.Tensor] = None):
        """wave (B,N) f32 and video (B,F,67,67) u8/f32 already on the device; the input the model does not read (and
        its n_samples / n_src) is None.  Returns (logits, posteriors, decisions), each (B,t_max,y_dim) on the device.
        ``lengths`` default: :meth:`lengths_of`; a caller may trim further (evaluate_audio_net.py trims to the labels).

        ``per_utterance`` (default: ``self.per_utterance``; "av" only): normalise every utterance's MCB output by its
        own L2 norm over its valid frames, so the batched call returns what B separate forward calls of the reference
        return -- the semantics of scripts/evaluate_AV_net.py:186-236, which calls the model once per utterance.  Off:
        one norm over the whole padded (B,T,1024) tensor of the call (AV_Net.py:117 for a batched call, the training
        scripts).  ``mcb_norms_out`` (f32 (B,) on the device, with ``per_utterance`` and ``use_mcb``): receives the norms
        used -- the constants :class:`avvad.stream.AVVADStream` needs to stream these utterances.  The audio-only and
        video-only models have no MCB and reject both: nothing couples the utterances of a call there.

        The video branch runs in pieces of ``self.piece`` utterances (frames of an utterance are independent for
        the trunk); ``_video_ready[k]`` / ``_wave_ready`` are optional CUDA events the current stream waits on
        before touching piece k / the waveforms (used by :meth:`infer_host` to overlap the uploads)."""
        if per_utterance is None:
            per_utterance = self.per_utterance
        check_inputs(self.modality, self.use_mcb, wave, video_u8, per_utterance, mcb_norms_out)
        B = (wave if wave is not None else video_u8).shape[0]
        if lengths is None:
            lengths = self.lengths_of(n_samples, n_src)
        if t_max is None:
            t_max = max(lengths)
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        lens = E._i32(lengths, dev)
        M = B * t_max
        x = self._buf("x", (B, t_max, self.lstm.ld), torch.bfloat16)
        xv = x.view(M, self.lstm.ld)
        if self.modality == "audio":
            # front end -> bf16 operand rows (zero tail columns) in one kernel: nothing else feeds the LSTM
            if _wave_ready is not None:
                cur.wait_event(_wave_ready)
            E.frontend_logpower(wave, E._i32(n_samples, dev), lens, t_max, self.audio_mean, self.audio_std, self.eps,
                                True, out_bf16=x)
        elif self.modality == "video":
            # trunk -> bf16 operand rows (ld = 512 = the trunk's width: no tail columns)
            self._video_pieces(video_u8, E._i32(n_src, dev), lens, t_max, None, xv, 0, _video_ready)
        else:
            ns, nsrc = E._i32(n_samples, dev), E._i32(n_src, dev)
            audio = self._buf("audio", (B, t_max, 513), torch.float32)
            feat = self._buf("feat", (M, 512), torch.float32) if self.use_mcb else None
            if not self.use_mcb:
                x.zero_()

            def front_end():
                if _wave_ready is not None:
                    cur.wait_event(_wave_ready)
                E.frontend_logpower(wave, ns, lens, t_max, self.audio_mean, self.audio_std, self.eps, True, out=audio)
                if not self.use_mcb:
                    E.pack_rows_bf16(audio.view(M, 513), xv, 0, False)

            if _wave_ready is None:
                front_end()
            # the waveforms arrive behind the first video piece
            self._video_pieces(video_u8, nsrc, lens, t_max, feat, xv, 513, _video_ready,
                               after_first=front_end if _wave_ready is not None else None)
            if self.use_mcb:
                if per_utterance:
                    self.mcb.forward_grouped(audio.view(M, 513), feat, lens, t_max, out_bf16=xv,
                                             norms_out=mcb_norms_out)
                else:
                    if mcb_norms_out is not None:
                        raise ValueError("mcb_norms_out needs per_utterance=True")
                    self.mcb.forward(audio.view(M, 513), feat, out_bf16=xv)
        logits, post, dec, _ = self.lstm.forward(x, lens, want_post=True, want_dec=True)
        return logits, post, dec

    def _video_pieces(self, video_u8, nsrc, lens, t_max, feat, xv, col_off, _video_ready, after_first=None):
        """Trunk features of every frame in pieces of ``self.piece`` utterances: fp32 into ``feat`` (M,512), or (feat
        None) bf16 into columns col_off .. col_off + 511 of the operand rows ``xv``.  ``after_first`` runs after the
        first piece."""
        B = video_u8.shape[0]
        dev = self.device
        cur = torch.cuda.current_stream(dev)
        num, den = self.video_rate
        P = max(1, min(self.piece, B))
        fused = self.fuse_gather and video_u8.dtype == torch.uint8
        frames = None if fused else self._buf("frames", (P, t_max, 67, 67), torch.float32)
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
                                 out_f32=feat[m0:m1] if feat is not None else None,
                                 out_bf16=None if feat is not None else xv[m0:m1], col_off=col_off, num=num, den=den)
            elif fused:  # gather + standardise + collate padding inside the stem kernel
                kw = dict(feat=feat[m0:m1]) if feat is not None else dict(feat_bf16=xv[m0:m1], col_off=col_off,
                                                                         want_f32=False)
                self.trunk.forward_u8(video_u8[b0:b1], nsrc[b0:b1], lens[b0:b1], t_max, self.video_mean,
                                      self.video_std, self.eps, True, num=num, den=den, **kw)
            else:
                fr = frames[: b1 - b0]
                E.upsample_gather(video_u8[b0:b1], nsrc[b0:b1], lens[b0:b1], t_max, self.video_mean, self.video_std,
                                  self.eps, True, num=num, den=den, out=fr)
                if feat is not None:
                    self.trunk.forward(fr.view(m1 - m0, 67, 67), feat=feat[m0:m1])
                else:
                    self.trunk.forward(fr.view(m1 - m0, 67, 67), feat_bf16=xv[m0:m1], col_off=col_off, want_f32=False)
            if k == 0 and after_first is not None:
                after_first()

    def infer_host(self, wave_pinned: Optional[torch.Tensor], n_samples, video_pinned: Optional[torch.Tensor], n_src,
                   lengths=None, t_max: Optional[int] = None, per_utterance: Optional[bool] = None):
        """Host (pinned) buffers in, host posteriors/decisions out; the input the model does not read is None.  The
        uploads run on a copy stream -- first video piece, waveforms, remaining video pieces -- while the current
        stream computes piece by piece, so only the first piece's upload is exposed; the D2H read-back is inside the
        call (this is what bench.py's `e2e` times)."""
        check_inputs(self.modality, self.use_mcb, wave_pinned, video_pinned, per_utterance)
        dev = self.device
        B = (wave_pinned if wave_pinned is not None else video_pinned).shape[0]
        w = v = None
        if wave_pinned is not None:
            w = self._buf("wave_dev", tuple(wave_pinned.shape), wave_pinned.dtype)
        if video_pinned is not None:
            v = self._buf("video_dev", tuple(video_pinned.shape), video_pinned.dtype)
        cur = torch.cuda.current_stream(dev)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        cs = self._copy_stream
        P = max(1, min(self.piece, B))
        n_pieces = (B + P - 1) // P if v is not None else 0
        while len(self._events) < n_pieces + 1:
            self._events.append(torch.cuda.Event())
        ew, ev = self._events[0], self._events[1:n_pieces + 1]
        cs.wait_stream(cur)  # earlier consumers of the staging buffers
        with torch.cuda.stream(cs):
            if v is None:
                w.copy_(wave_pinned, non_blocking=True)
                ew.record(cs)
            for k, b0 in enumerate(range(0, B, P) if v is not None else ()):
                b1 = min(B, b0 + P)
                v[b0:b1].copy_(video_pinned[b0:b1], non_blocking=True)
                ev[k].record(cs)
                if k == 0 and w is not None:
                    w.copy_(wave_pinned, non_blocking=True)
                    ew.record(cs)
        _, post, dec = self.infer_device(w, n_samples, v, n_src, lengths=lengths, t_max=t_max,
                                         _video_ready=ev if v is not None else None,
                                         _wave_ready=ew if w is not None else None, per_utterance=per_utterance)
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


def modality_lengths(modality: str, n_samples, n_src, video_rate=(E.FPS_NUM, E.FPS_DEN)):
    """Frame counts of a list of utterances for one model (host only): min(STFT frames, upsampled video frames) for
    "av", stft_num_frames(N) for "audio" (scripts/evaluate_audio_net.py), upsampled_length(F) for "video"."""
    if modality == "av":
        return AVVADPipeline.frame_counts(n_samples, n_src)
    if modality == "audio":
        return [E.stft_num_frames(n) for n in n_samples]
    if modality == "video":
        return [E.upsampled_length(f, *video_rate) for f in n_src]
    raise ValueError(f"modality must be one of {MODALITIES}, got {modality!r}")
