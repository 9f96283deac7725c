"""Host-side drivers of the libavvad C ABI.

PyTorch is used only as plumbing here: device memory (tensors as buffers), the current CUDA stream and
parameter storage.  All arithmetic of the hot path happens inside libavvad.so.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import lib as L

FPS_NUM, FPS_DEN = 25, 12  # 62.5 / 30 (scripts/create_video_train_files_upsampled.py:58-59)

# conv layer index (include/avvad.h) -> (conv key, bn key) under the `features.` prefix
RESNET_LAYER_KEYS = [("0", "1")]
for _stage in (4, 5, 6, 7):
    RESNET_LAYER_KEYS += [(f"{_stage}.0.conv1", f"{_stage}.0.bn1"), (f"{_stage}.0.conv2", f"{_stage}.0.bn2")]
    if _stage != 4:
        RESNET_LAYER_KEYS += [(f"{_stage}.0.downsample.0", f"{_stage}.0.downsample.1")]
    RESNET_LAYER_KEYS += [(f"{_stage}.1.conv1", f"{_stage}.1.bn1"), (f"{_stage}.1.conv2", f"{_stage}.1.bn2")]
assert len(RESNET_LAYER_KEYS) == 20


def _f32(t: torch.Tensor, device) -> torch.Tensor:
    return t.detach().to(device=device, dtype=torch.float32).contiguous()


def _i32(x, device) -> torch.Tensor:
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.int32).contiguous()
    return torch.tensor(list(x), dtype=torch.int32, device=device)


class _Workspace:
    """Grow-only byte buffer reused across calls (caller-owned scratch of the C ABI)."""

    def __init__(self):
        self.buf: Optional[torch.Tensor] = None

    def get(self, nbytes: int, device) -> torch.Tensor:
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != torch.device(device):
            self.buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        return self.buf


# ---------------------------------------------------------------------------------------------
# front end / upsampling
# ---------------------------------------------------------------------------------------------
def stft_num_frames(n_samples: int, fs=16000, wlen_sec=64e-3, hop_percent=0.25, pad_at_end=True) -> int:
    return int(L.lib().avvad_stft_num_frames(int(n_samples), float(fs), float(wlen_sec), float(hop_percent),
                                             1 if pad_at_end else 0))


def upsampled_length(n_src: int, num=FPS_NUM, den=FPS_DEN) -> int:
    return int(L.lib().avvad_upsampled_length(int(n_src), num, den))


def frontend_logpower(wave: torch.Tensor, n_samples, n_frames, t_max: int, mean: Optional[torch.Tensor],
                      std: Optional[torch.Tensor], eps=1e-8, normalise=True, out: Optional[torch.Tensor] = None,
                      peaks: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None,
                      ld: Optional[int] = None, col_off=0):
    """(B,N) fp32 waveforms -> (B,t_max,513) standardised log-power features (SURVEY A1-A4).

    ``peaks`` (f32 (B,)): with ``normalise``, divide by these per-utterance peaks instead of max|x| over the samples
    given -- a stream sees only part of the utterance.

    ``out_bf16`` (bf16, B * t_max rows of ``ld`` elements, default ld = its last dimension): write the features
    rounded to bf16 there instead, at columns ``col_off .. col_off + 512``, and zero the columns after them -- an LSTM
    layer-0 operand in one kernel, bit-identical to ``pack_rows_bf16(features, out_bf16, col_off, zero_tail=True)``.
    Returns ``out_bf16`` then."""
    L.require_cuda(wave)
    assert wave.dim() == 2 and wave.dtype == torch.float32
    wave = wave.contiguous()
    B = wave.shape[0]
    dev = wave.device
    ns, nf = _i32(n_samples, dev), _i32(n_frames, dev)
    if out_bf16 is not None:
        if out is not None:
            raise ValueError("frontend_logpower: give out or out_bf16, not both")
        ld = int(out_bf16.shape[-1]) if ld is None else int(ld)
        if (out_bf16.dtype != torch.bfloat16 or not out_bf16.is_contiguous() or out_bf16.device != dev
                or out_bf16.numel() < B * t_max * ld):
            raise ValueError(f"frontend_logpower: out_bf16 must be a contiguous bf16 tensor of B * t_max = {B * t_max} "
                             f"rows of ld = {ld} on {dev}")
    elif out is None:
        out = torch.empty(B, t_max, 513, dtype=torch.float32, device=dev)
    mode = 0
    if normalise:
        mode = 2 if peaks is not None else 1
    if peaks is not None:
        peak = _f32(peaks.reshape(-1), dev)
        if peak.numel() != B:
            raise ValueError("frontend_logpower: one peak per utterance required")
    else:
        peak = torch.empty(B, dtype=torch.float32, device=dev)
    m = _f32(mean.reshape(-1), dev) if mean is not None else None
    s = _f32(std.reshape(-1), dev) if std is not None else None
    if out_bf16 is not None:
        L.check(L.lib().avvad_frontend_logpower_bf16(L.ptr(wave), wave.stride(0), L.ptr(ns), L.ptr(nf), B, t_max, mode,
                                                     L.ptr(m), L.ptr(s), eps, L.ptr(out_bf16), ld, int(col_off),
                                                     L.ptr(peak), L.stream_ptr()))
        return out_bf16
    L.check(L.lib().avvad_frontend_logpower(L.ptr(wave), wave.stride(0), L.ptr(ns), L.ptr(nf), B, t_max,
                                            mode, L.ptr(m), L.ptr(s), eps, L.ptr(out), L.ptr(peak),
                                            L.stream_ptr()))
    return out


def stft(wave: torch.Tensor, n_samples, n_frames, t_max: int) -> torch.Tensor:
    """(B,N) -> (B,513,t_max,2) real view, as the legacy torch.stft the reference calls."""
    L.require_cuda(wave)
    wave = wave.contiguous()
    B, dev = wave.shape[0], wave.device
    ns, nf = _i32(n_samples, dev), _i32(n_frames, dev)
    out = torch.empty(B, 513, t_max, 2, dtype=torch.float32, device=dev)
    L.check(L.lib().avvad_stft(L.ptr(wave), wave.stride(0), L.ptr(ns), L.ptr(nf), B, t_max, L.ptr(out),
                               L.stream_ptr()))
    return out


def upsample_gather(src: torch.Tensor, n_src, n_out, t_max: int, mean=0.0, std=1.0, eps=1e-8, standardise=False,
                    num=FPS_NUM, den=FPS_DEN, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B,F,H,W) u8/f32 frames at 30 fps -> (B,t_max,H,W) fp32 at 62.5 fps (SURVEY U + A4)."""
    L.require_cuda(src)
    assert src.dim() == 4 and src.dtype in (torch.uint8, torch.float32)
    src = src.contiguous()
    B, F, H, W = src.shape
    dev = src.device
    a, b = _i32(n_src, dev), _i32(n_out, dev)
    if out is None:
        out = torch.empty(B, t_max, H, W, dtype=torch.float32, device=dev)
    L.check(L.lib().avvad_upsample_gather(L.ptr(src), 1 if src.dtype == torch.float32 else 0, L.ptr(a), L.ptr(b), B,
                                          F, t_max, H * W, num, den, float(mean), float(std), float(eps),
                                          1 if standardise else 0, L.ptr(out), L.stream_ptr()))
    return out


def feature_gather(feat_src: torch.Tensor, feat_pad: torch.Tensor, n_src, n_out, t_max: int,
                   out_f32: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None, col_off=0,
                   num=FPS_NUM, den=FPS_DEN):
    """(B,F,C) fp32 source-rate features -> (B*t_max, C) at 62.5 fps (same index map as upsample_gather); rows past
    n_out[b] get `feat_pad` (the feature of the collate zero frame)."""
    L.require_cuda(feat_src, feat_pad)
    B, F, Cc = feat_src.shape
    dev = feat_src.device
    a, b = _i32(n_src, dev), _i32(n_out, dev)
    ld = out_bf16.stride(-2) if out_bf16 is not None else 0
    L.check(L.lib().avvad_feature_gather(L.ptr(feat_src.contiguous()), L.ptr(feat_pad.contiguous()), L.ptr(a), L.ptr(b),
                                         B, F, t_max, Cc, num, den, L.ptr(out_f32), L.ptr(out_bf16), ld, col_off,
                                         L.stream_ptr()))


def upsample_index(n_src: int, n_out: int, device="cuda", num=FPS_NUM, den=FPS_DEN) -> torch.Tensor:
    out = torch.empty(n_out, dtype=torch.int32, device=device)
    L.check(L.lib().avvad_upsample_index(n_src, n_out, num, den, L.ptr(out), L.stream_ptr()))
    return out


# ---------------------------------------------------------------------------------------------
# data preparation on the device (SURVEY 8f rows 1, 3)
# ---------------------------------------------------------------------------------------------
def dct_roi_decode(dct: torch.Tensor, mode="per_frame", want_raw=False):
    """(F, 4489) fp32 DCT rows of an NTCD-TIMIT .mat file -> mouth-ROI frames.
    mode "per_frame": u8 (F,67,67), per-frame min-max + rot90(.,3) (the variant behind the shipped *_upsampled.h5);
    mode "global": fp32 (F,67,67), the script as shipped (global min, largest per-row range)."""
    L.require_cuda(dct)
    dct = dct.to(torch.float32).contiguous()
    F = dct.shape[0]
    dev = dct.device
    if mode == "per_frame":
        out = torch.empty(F, 67, 67, dtype=torch.uint8, device=dev)
        raw = torch.empty(F, 67, 67, dtype=torch.float32, device=dev) if want_raw else None
        L.check(L.lib().avvad_dct_roi_decode(L.ptr(dct), F, 0, L.ptr(out), L.ptr(raw), None, 0, L.stream_ptr()))
        return (out, raw) if want_raw else out
    ws = torch.empty(L.lib().avvad_dct_roi_workspace_bytes(F), dtype=torch.uint8, device=dev)
    out = torch.empty(F, 67, 67, dtype=torch.float32, device=dev)
    L.check(L.lib().avvad_dct_roi_decode(L.ptr(dct), F, 1, None, L.ptr(out), L.ptr(ws), ws.numel(), L.stream_ptr()))
    return out


def vad_labels(wave: torch.Tensor, n_samples, n_frames, t_max: int, nfft=1024, hop=256, vad_threshold=1.70):
    """clean_speech_VAD (center=False) for a batch of (B,N) fp32 waveforms -> (B,t_max) fp32 0/1."""
    L.require_cuda(wave)
    wave = wave.contiguous()
    B, dev = wave.shape[0], wave.device
    ns, nf = _i32(n_samples, dev), _i32(n_frames, dev)
    energy = torch.empty(B, t_max, dtype=torch.float32, device=dev)
    labels = torch.empty(B, t_max, dtype=torch.float32, device=dev)
    L.check(L.lib().avvad_vad_labels(L.ptr(wave), wave.stride(0), L.ptr(ns), L.ptr(nf), B, t_max, nfft, hop,
                                     float(vad_threshold), L.ptr(energy), L.ptr(labels), L.stream_ptr()))
    return labels


def ibm_labels(stft_ft2: torch.Tensor, n_frames, eps=1e-8, ibm_threshold=50.0):
    """clean_speech_IBM on (B,513,T,2) STFTs (layout of `stft`) -> (B,513,T) fp32 0/1."""
    L.require_cuda(stft_ft2)
    stft_ft2 = stft_ft2.contiguous()
    B, bins, T, _ = stft_ft2.shape
    dev = stft_ft2.device
    nf = _i32(n_frames, dev)
    db = torch.empty(B, bins, T, dtype=torch.float32, device=dev)
    mx = torch.empty(B, dtype=torch.float32, device=dev)
    mask = torch.empty(B, bins, T, dtype=torch.float32, device=dev)
    L.check(L.lib().avvad_ibm_labels(L.ptr(stft_ft2), L.ptr(nf), B, T, bins, float(eps), float(ibm_threshold), L.ptr(db),
                                     L.ptr(mx), L.ptr(mask), L.stream_ptr()))
    return mask


class RunningStats:
    """Per-bin mean / empirical std over a dataset (create_audio_train_files.py:273-280,365-368), accumulated on the
    device in fp64 batch by batch."""

    def __init__(self, bins: int, device="cuda"):
        self.bins = bins
        self.sum = torch.zeros(bins, dtype=torch.float64, device=device)
        self.sumsq = torch.zeros(bins, dtype=torch.float64, device=device)
        self.n = 0

    def update(self, x: torch.Tensor, n_frames):
        """x (B,T,bins) fp32; only frames t < n_frames[b] count."""
        L.require_cuda(x)
        x = x.contiguous()
        B, T, bins = x.shape
        assert bins == self.bins
        nf = _i32(n_frames, x.device)
        L.check(L.lib().avvad_stats_accumulate(L.ptr(x), L.ptr(nf), B, T, bins, L.ptr(self.sum), L.ptr(self.sumsq),
                                               L.stream_ptr()))
        self.n += int(torch.clamp(nf, max=T).sum().item())

    def finalize(self):
        mean = torch.empty(self.bins, dtype=torch.float32, device=self.sum.device)
        std = torch.empty(self.bins, dtype=torch.float32, device=self.sum.device)
        L.check(L.lib().avvad_stats_finalize(L.ptr(self.sum), L.ptr(self.sumsq), float(self.n), self.bins, L.ptr(mean),
                                             L.ptr(std), L.stream_ptr()))
        return mean, std


# ---------------------------------------------------------------------------------------------
# generic tensor-core ops (exposed for tests)
# ---------------------------------------------------------------------------------------------
def gemm_bf16(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, out_bf16=False, relu=False):
    """C = A @ W^T (+bias); A (M,K) bf16, W (N,K) bf16."""
    L.require_cuda(a, w)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16
    a, w = a.contiguous(), w.contiguous()
    M, K = a.shape
    N = w.shape[0]
    c = torch.empty(M, N, dtype=torch.bfloat16 if out_bf16 else torch.float32, device=a.device)
    b = _f32(bias, a.device) if bias is not None else None
    L.check(L.lib().avvad_gemm_bf16(L.ptr(a), K, L.ptr(w), K, L.ptr(b), L.ptr(c), N, 1 if out_bf16 else 0,
                                    1 if relu else 0, M, N, K, L.stream_ptr()))
    return c


def conv2d_nhwc_bf16(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], stride: int, pad: int,
                     residual: Optional[torch.Tensor] = None, relu=False) -> torch.Tensor:
    """x (n,H,W,Cin) bf16, w (Cout,R,S,Cin) bf16 -> (n,OH,OW,Cout) bf16."""
    L.require_cuda(x, w)
    x, w = x.contiguous(), w.contiguous()
    n, H, W, Cin = x.shape
    Cout, R, S, _ = w.shape
    OH = (H + 2 * pad - R) // stride + 1
    OW = (W + 2 * pad - S) // stride + 1
    out = torch.empty(n, OH, OW, Cout, dtype=torch.bfloat16, device=x.device)
    b = _f32(bias, x.device) if bias is not None else None
    r = residual.contiguous() if residual is not None else None
    L.check(L.lib().avvad_conv2d_nhwc_bf16(L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(r), L.ptr(out), n, H, W, Cin, Cout, R,
                                           S, stride, pad, 1 if relu else 0, L.stream_ptr()))
    return out


def conv2d_nhwc_bf16_dual(x: torch.Tensor, x2: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor],
                          stride: int, pad: int, k: int, stride2: int, relu=False) -> torch.Tensor:
    """out = act(conv_kxk(x; w[:, :k*k*Cin]) + conv_1x1_stride2(x2; w[:, k*k*Cin:]) + bias) in one implicit GEMM."""
    L.require_cuda(x, x2, w)
    x, x2, w = x.contiguous(), x2.contiguous(), w.contiguous()
    n, H, W, Cin = x.shape
    _, H2, W2, Cin2 = x2.shape
    Cout = w.shape[0]
    assert w.shape[1] == k * k * Cin + Cin2
    OH = (H + 2 * pad - k) // stride + 1
    OW = (W + 2 * pad - k) // stride + 1
    out = torch.empty(n, OH, OW, Cout, dtype=torch.bfloat16, device=x.device)
    b = _f32(bias, x.device) if bias is not None else None
    L.check(L.lib().avvad_conv2d_nhwc_bf16_dual(L.ptr(x), L.ptr(x2), L.ptr(w), L.ptr(b), L.ptr(out), n, H, W, Cin, H2, W2,
                                                Cin2, stride2, Cout, k, k, stride, pad, 1 if relu else 0,
                                                L.stream_ptr()))
    return out


def pack_rows_bf16(src: torch.Tensor, dst: torch.Tensor, col_off: int, zero_tail: bool):
    """dst[m, col_off:col_off+cols] = bf16(src[m, :]) (dst is a (rows, ld) bf16 operand buffer)."""
    rows, cols = src.shape
    L.check(L.lib().avvad_pack_rows_bf16(L.ptr(src), src.stride(0), L.ptr(dst), dst.stride(0), col_off, rows, cols,
                                         1 if zero_tail else 0, L.stream_ptr()))


# ---------------------------------------------------------------------------------------------
# model blocks
# ---------------------------------------------------------------------------------------------
class ResNet18Trunk:
    """Eval-mode ResNet-18 trunk (children[:-1]) on (M,67,67) fp32 ROIs -> (M,512)."""

    def __init__(self):
        h = C.c_void_p()
        L.check(L.lib().avvad_resnet18_create(C.byref(h)))
        self.h = h
        self.ws = _Workspace()
        self.chunk = int(os.environ.get("AVVAD_CHUNK", "24576"))  # frames per trunk pass (buffers: 4 x chunk x 37 KB)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                L.lib().avvad_resnet18_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def load(self, sd: Dict[str, torch.Tensor], device, prefix="features.", bn_eps=1e-5):
        keep = []
        for i, (ck, bk) in enumerate(RESNET_LAYER_KEYS):
            w = _f32(sd[prefix + ck + ".weight"], device)
            g = _f32(sd[prefix + bk + ".weight"], device)
            b = _f32(sd[prefix + bk + ".bias"], device)
            m = _f32(sd[prefix + bk + ".running_mean"], device)
            v = _f32(sd[prefix + bk + ".running_var"], device)
            keep += [w, g, b, m, v]
            L.check(L.lib().avvad_resnet18_set_conv(self.h, i, L.ptr(w), L.ptr(g), L.ptr(b), L.ptr(m), L.ptr(v),
                                                    bn_eps, L.stream_ptr()))
        torch.cuda.current_stream().synchronize()  # sources may be temporaries
        del keep

    def forward(self, frames: torch.Tensor, feat: Optional[torch.Tensor] = None,
                feat_bf16: Optional[torch.Tensor] = None, col_off=0, want_f32=True):
        L.require_cuda(frames)
        assert frames.dtype == torch.float32 and frames.shape[-2:] == (67, 67)
        frames = frames.contiguous()
        n = frames.numel() // (67 * 67)
        nbytes = L.lib().avvad_resnet18_workspace_bytes(n, self.chunk)
        ws = self.ws.get(nbytes, frames.device)
        if feat is None and want_f32:
            feat = torch.empty(n, 512, dtype=torch.float32, device=frames.device)
        ld = feat_bf16.stride(-2) if feat_bf16 is not None else 0
        L.check(L.lib().avvad_resnet18_forward(self.h, L.ptr(frames), n, self.chunk, L.ptr(ws), ws.numel(),
                                               L.ptr(feat), L.ptr(feat_bf16), ld, col_off, L.stream_ptr()))
        return feat

    def forward_u8(self, src: torch.Tensor, n_src, n_out, t_max: int, mean=0.0, std=1.0, eps=1e-8, standardise=True,
                   feat: Optional[torch.Tensor] = None, feat_bf16: Optional[torch.Tensor] = None, col_off=0,
                   want_f32=True, num=FPS_NUM, den=FPS_DEN):
        """Trunk fed from the 30 fps u8 source frames (B,F,67,67): the 30->62.5 fps gather, standardisation and
        collate padding happen while a frame is staged in shared memory (== upsample_gather + forward, bit for bit)."""
        L.require_cuda(src)
        assert src.dtype == torch.uint8 and src.dim() == 4 and src.shape[-2:] == (67, 67)
        src = src.contiguous()
        B, F = src.shape[:2]
        dev = src.device
        a, b = _i32(n_src, dev), _i32(n_out, dev)
        n = B * t_max
        nbytes = L.lib().avvad_resnet18_workspace_bytes(n, self.chunk)
        ws = self.ws.get(nbytes, dev)
        if feat is None and want_f32:
            feat = torch.empty(n, 512, dtype=torch.float32, device=dev)
        ld = feat_bf16.stride(-2) if feat_bf16 is not None else 0
        L.check(L.lib().avvad_resnet18_forward_u8(self.h, L.ptr(src), L.ptr(a), L.ptr(b), B, F, t_max, num, den,
                                                  float(mean), float(std), float(eps), 1 if standardise else 0,
                                                  self.chunk, L.ptr(ws), ws.numel(), L.ptr(feat), L.ptr(feat_bf16), ld,
                                                  col_off, L.stream_ptr()))
        return feat

    def load_train(self, sd: Dict[str, torch.Tensor], device, prefix="features."):
        """Un-folded weights + BN affine parameters for the batch-statistics (training-mode) forward."""
        keep = []
        for i, (ck, bk) in enumerate(RESNET_LAYER_KEYS):
            w = _f32(sd[prefix + ck + ".weight"], device)
            g = _f32(sd[prefix + bk + ".weight"], device)
            b = _f32(sd[prefix + bk + ".bias"], device)
            keep += [w, g, b]
            L.check(L.lib().avvad_resnet18_set_conv_train(self.h, i, L.ptr(w), L.ptr(g), L.ptr(b), L.stream_ptr()))
        torch.cuda.current_stream().synchronize()

    def forward_train(self, frames: torch.Tensor, running: Optional[Sequence[Tuple[torch.Tensor, torch.Tensor]]] = None,
                      feat_bf16: Optional[torch.Tensor] = None, col_off=0, want_f32=True, bn_eps=1e-5, momentum=0.1):
        """Training-mode forward: batch statistics over all frames of the call; `running` = 20 (running_mean,
        running_var) fp32 CUDA tensor pairs updated in place (the module's BatchNorm buffers)."""
        L.require_cuda(frames)
        frames = frames.contiguous()
        n = frames.numel() // (67 * 67)
        nbytes = L.lib().avvad_resnet18_train_workspace_bytes(n)
        if not hasattr(self, "tws"):
            self.tws = _Workspace()
        ws = self.tws.get(nbytes, frames.device)
        feat = torch.empty(n, 512, dtype=torch.float32, device=frames.device) if want_f32 else None
        rm = _ptr_array([r[0] for r in running]) if running is not None else None
        rv = _ptr_array([r[1] for r in running]) if running is not None else None
        ld = feat_bf16.stride(-2) if feat_bf16 is not None else 0
        L.check(L.lib().avvad_resnet18_forward_train(self.h, L.ptr(frames), n, L.ptr(ws), ws.numel(), bn_eps, momentum,
                                                     rm, rv, L.ptr(feat), L.ptr(feat_bf16), ld, col_off,
                                                     L.stream_ptr()))
        return feat

    def forward_tape(self, frames: torch.Tensor, running: Optional[Sequence[Tuple[torch.Tensor, torch.Tensor]]] = None,
                     bn_eps=1e-5, momentum=0.1):
        """Training-mode forward of a TRAINABLE trunk: returns (feat f32 (n,512), tape) -- the tape (a caller-owned
        byte tensor) carries every activation `backward` needs."""
        L.require_cuda(frames)
        frames = frames.contiguous()
        n = frames.numel() // (67 * 67)
        if not hasattr(self, "tws"):
            self.tws = _Workspace()
        ws = self.tws.get(L.lib().avvad_resnet18_tape_workspace_bytes(n), frames.device)
        tape = torch.empty(L.lib().avvad_resnet18_tape_bytes(n), dtype=torch.uint8, device=frames.device)
        feat = torch.empty(n, 512, dtype=torch.float32, device=frames.device)
        rm = _ptr_array([r[0] for r in running]) if running is not None else None
        rv = _ptr_array([r[1] for r in running]) if running is not None else None
        L.check(L.lib().avvad_resnet18_forward_tape(self.h, L.ptr(frames), n, L.ptr(ws), ws.numel(), L.ptr(tape),
                                                    tape.numel(), bn_eps, momentum, rm, rv, L.ptr(feat), None, 0, 0,
                                                    L.stream_ptr()))
        return feat, tape

    @staticmethod
    def tape_tensors(tape: torch.Tensor, n: int):
        """Views into a tape (inspection hook for the parity tests): dict with 'raw' (20 NHWC bf16 tensors), 'act0',
        'pool', 'y1' / 'out' (8 each) and 'stats' (float (20, 1024): per layer mean[:C] | invstd[C:2C])."""
        off = (C.c_int64 * 39)()
        L.check(L.lib().avvad_resnet18_tape_layout(n, off, 39))
        shapes = [(34, 34, 64), (34, 34, 64), (17, 17, 64)]
        specs = [(64, 17), (64, 17), (64, 17), (64, 17), (128, 9), (128, 9), (128, 9), (128, 9), (128, 9), (256, 5),
                 (256, 5), (256, 5), (256, 5), (256, 5), (512, 3), (512, 3), (512, 3), (512, 3), (512, 3)]
        shapes += [(h, h, c) for c, h in specs]
        for c, h in ((64, 17), (64, 17), (128, 9), (128, 9), (256, 5), (256, 5), (512, 3), (512, 3)):
            shapes += [(h, h, c), (h, h, c)]

        def view(i):
            numel = n * shapes[i][0] * shapes[i][1] * shapes[i][2]
            return tape[off[i]:off[i] + 2 * numel].view(torch.bfloat16).view((n,) + shapes[i])
        stats = tape[off[38]:off[38] + 20 * 1024 * 4].view(torch.float32).view(20, 1024)
        return {"raw": [view(0)] + [view(3 + l - 1) for l in range(1, 20)], "act0": view(1), "pool": view(2),
                "y1": [view(22 + 2 * b) for b in range(8)], "out": [view(23 + 2 * b) for b in range(8)], "stats": stats}

    def backward(self, frames: torch.Tensor, tape: torch.Tensor, dfeat: torch.Tensor, bn_eps=1e-5):
        """Gradients of the 20 conv weights (PyTorch layout) and BatchNorm (weight, bias) pairs from dfeat (n,512)."""
        frames = frames.contiguous()
        n = frames.numel() // (67 * 67)
        dev = frames.device
        dfeat = dfeat.detach().to(torch.float32).reshape(n, 512).contiguous()
        if not hasattr(self, "bws"):
            self.bws = _Workspace()
        ws = self.bws.get(L.lib().avvad_resnet18_backward_workspace_bytes(n), dev)
        shapes = [(64, 3, 7, 7)]
        for stage, cin, cout in ((4, 64, 64), (5, 64, 128), (6, 128, 256), (7, 256, 512)):
            shapes += [(cout, cin, 3, 3), (cout, cout, 3, 3)]
            if stage != 4:
                shapes += [(cout, cin, 1, 1)]
            shapes += [(cout, cout, 3, 3), (cout, cout, 3, 3)]
        dw = [torch.empty(s, dtype=torch.float32, device=dev) for s in shapes]
        dg = [torch.empty(s[0], dtype=torch.float32, device=dev) for s in shapes]
        db = [torch.empty(s[0], dtype=torch.float32, device=dev) for s in shapes]
        L.check(L.lib().avvad_resnet18_backward(self.h, L.ptr(frames), n, L.ptr(tape), L.ptr(dfeat), L.ptr(ws), ws.numel(),
                                                bn_eps, _ptr_array(dw), _ptr_array(dg), _ptr_array(db), L.stream_ptr()))
        return dw, dg, db

    def forward_upto(self, frames: torch.Tensor, upto: int, shape: Tuple[int, int, int]) -> torch.Tensor:
        """Test hook: NHWC bf16 activation after conv layer `upto` (shape = (h, w, c))."""
        frames = frames.contiguous()
        n = frames.numel() // (67 * 67)
        nbytes = L.lib().avvad_resnet18_workspace_bytes(n, n)
        ws = self.ws.get(nbytes, frames.device)
        out = torch.empty((n,) + tuple(shape), dtype=torch.bfloat16, device=frames.device)
        L.check(L.lib().avvad_resnet18_forward_upto(self.h, L.ptr(frames), n, upto, L.ptr(ws), ws.numel(), L.ptr(out),
                                                    L.stream_ptr()))
        return out


class Mcb:
    """MCB + signed sqrt + whole-tensor L2 + BatchNorm1d(eval) (SURVEY F2-F3)."""

    def __init__(self):
        h = C.c_void_p()
        L.check(L.lib().avvad_mcb_create(C.byref(h)))
        self.h = h
        self.ws = _Workspace()

    def __del__(self):
        try:
            if getattr(self, "h", None):
                L.lib().avvad_mcb_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def load(self, sd: Dict[str, torch.Tensor], device, eps=1e-8):
        h1 = sd["mcb.sketch1.h"].to(device=device, dtype=torch.int64).contiguous()
        h2 = sd["mcb.sketch2.h"].to(device=device, dtype=torch.int64).contiguous()
        s1, s2 = _f32(sd["mcb.sketch1.s"], device), _f32(sd["mcb.sketch2.s"], device)
        g, b = _f32(sd["mcb_bn.weight"], device), _f32(sd["mcb_bn.bias"], device)
        m, v = _f32(sd["mcb_bn.running_mean"], device), _f32(sd["mcb_bn.running_var"], device)
        L.check(L.lib().avvad_mcb_load(self.h, L.ptr(h1), L.ptr(s1), L.ptr(h2), L.ptr(s2), L.ptr(g), L.ptr(b),
                                       L.ptr(m), L.ptr(v), eps, L.stream_ptr()))
        torch.cuda.current_stream().synchronize()

    def forward(self, audio: torch.Tensor, video: torch.Tensor, out_bf16: Optional[torch.Tensor] = None,
                out_f32: Optional[torch.Tensor] = None):
        L.require_cuda(audio, video)
        audio = audio.reshape(-1, 513).contiguous()
        video = video.reshape(-1, 512).contiguous()
        rows = audio.shape[0]
        nbytes = L.lib().avvad_mcb_workspace_bytes(rows)
        ws = self.ws.get(nbytes, audio.device)
        ld = out_bf16.stride(-2) if out_bf16 is not None else 0
        L.check(L.lib().avvad_mcb_forward(self.h, L.ptr(audio), L.ptr(video), rows, L.ptr(ws), ws.numel(),
                                          L.ptr(out_bf16), ld, L.ptr(out_f32), L.stream_ptr()))

    def forward_grouped(self, audio: torch.Tensor, video: torch.Tensor, lengths, t_max: int,
                        out_bf16: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None,
                        norms_in: Optional[torch.Tensor] = None, norms_out: Optional[torch.Tensor] = None):
        """audio (B,t_max,513), video (B,t_max,512): every utterance normalised by its own L2 norm over its
        ``lengths[b]`` valid rows -- B stand-alone forward calls of the reference module in one launch
        (scripts/evaluate_AV_net.py:186-236 calls the model once per utterance).  ``norms_in`` (f32 (B,)): use these
        norms instead (a stream normalises every block of an utterance by one constant); ``norms_out`` (f32 (B,),
        contiguous): receives the norms used."""
        L.require_cuda(audio, video)
        audio = audio.reshape(-1, 513).contiguous()
        video = video.reshape(-1, 512).contiguous()
        t_max = int(t_max)
        if t_max <= 0 or audio.shape[0] % t_max or video.shape[0] != audio.shape[0]:
            raise ValueError("forward_grouped: rows must be n_groups * t_max for both inputs")
        B = audio.shape[0] // t_max
        lens = _i32(lengths, audio.device)
        if lens.numel() != B:
            raise ValueError("forward_grouped: one length per utterance required")
        nbytes = L.lib().avvad_mcb_grouped_workspace_bytes(B, t_max)
        ws = self.ws.get(nbytes, audio.device)
        ld = out_bf16.stride(-2) if out_bf16 is not None else 0
        nin = None
        if norms_in is not None:
            nin = _f32(norms_in.reshape(-1), audio.device)
            if nin.numel() != B:
                raise ValueError("forward_grouped: one norm per utterance required")
        if norms_out is not None:
            assert norms_out.dtype == torch.float32 and norms_out.is_contiguous() and norms_out.numel() == B
        L.check(L.lib().avvad_mcb_forward_grouped_norms(self.h, L.ptr(audio), L.ptr(video), B, t_max, L.ptr(lens),
                                                        L.ptr(nin), L.ptr(norms_out), L.ptr(ws), ws.numel(),
                                                        L.ptr(out_bf16), ld, L.ptr(out_f32), L.stream_ptr()))


def mcb_forward_train(mcb: "Mcb", audio, video, gamma, beta, running_mean, running_var, out_bf16, momentum=0.1):
    """Training-mode MCB fusion; returns the workspace (kept alive for mcb_backward_bn)."""
    audio = audio.reshape(-1, 513).contiguous()
    video = video.reshape(-1, 512).contiguous()
    rows = audio.shape[0]
    nbytes = L.lib().avvad_mcb_workspace_bytes(rows)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=audio.device)
    ld = out_bf16.stride(-2)
    L.check(L.lib().avvad_mcb_forward_train(mcb.h, L.ptr(audio), L.ptr(video), rows, L.ptr(ws), ws.numel(), L.ptr(gamma),
                                            L.ptr(beta), momentum, L.ptr(running_mean), L.ptr(running_var),
                                            L.ptr(out_bf16), ld, None, L.stream_ptr()))
    return ws, rows


def mcb_backward_bn(mcb: "Mcb", ws, rows, dx: torch.Tensor):
    dx = dx.reshape(rows, -1).contiguous()
    dg = torch.empty(1024, dtype=torch.float32, device=dx.device)
    db = torch.empty(1024, dtype=torch.float32, device=dx.device)
    L.check(L.lib().avvad_mcb_backward_bn(mcb.h, L.ptr(ws), L.ptr(dx), dx.stride(0), rows, L.ptr(dg), L.ptr(db),
                                          L.stream_ptr()))
    return dg, db


class Lstm:
    """L-layer LSTM + Linear head over padded batches (SURVEY R1, R2, H1, H2)."""

    def __init__(self, layers: int, input_size: int, hidden: int, y_dim: int):
        h = C.c_void_p()
        L.check(L.lib().avvad_lstm_create(C.byref(h), layers, input_size, hidden, y_dim))
        self.h = h
        self.layers, self.input_size, self.hidden, self.y_dim = layers, input_size, hidden, y_dim
        self.ld = int(L.lib().avvad_lstm_input_ld(self.h))
        self.ws = _Workspace()

    def __del__(self):
        try:
            if getattr(self, "h", None):
                L.lib().avvad_lstm_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def load(self, sd: Dict[str, torch.Tensor], device, lstm_prefix: str, head_prefix: str):
        keep = []
        for l in range(self.layers):
            t = [_f32(sd[f"{lstm_prefix}.{k}_l{l}"], device) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            keep += t
            L.check(L.lib().avvad_lstm_set_layer(self.h, l, *[L.ptr(x) for x in t], L.stream_ptr()))
        w, b = _f32(sd[head_prefix + ".weight"], device), _f32(sd[head_prefix + ".bias"], device)
        L.check(L.lib().avvad_lstm_set_head(self.h, L.ptr(w), L.ptr(b), L.stream_ptr()))
        torch.cuda.current_stream().synchronize()

    def new_input(self, B: int, T: int, device) -> torch.Tensor:
        """bf16 operand buffer (B,T,ld); columns >= input_size must stay zero."""
        return torch.zeros(B, T, self.ld, dtype=torch.bfloat16, device=device)

    def forward(self, x_bf16: torch.Tensor, lengths, want_post=False, want_dec=False, want_last=False,
                state: Optional["LstmState"] = None):
        """With `state`, the recurrence continues from it and the call leaves each row's state after its
        ``lengths[b]`` new steps there (rows with length 0 keep theirs)."""
        L.require_cuda(x_bf16)
        B, T, ld = x_bf16.shape
        assert ld == self.ld and x_bf16.is_contiguous() and x_bf16.dtype == torch.bfloat16
        dev = x_bf16.device
        lens = _i32(lengths, dev)
        if state is not None:
            state.check(self, B, dev)
            nbytes = L.lib().avvad_lstm_state_workspace_bytes(self.h, B, T)
        else:
            nbytes = L.lib().avvad_lstm_workspace_bytes(self.h, B, T)
        ws = self.ws.get(nbytes, dev)
        logits = torch.empty(B, T, self.y_dim, dtype=torch.float32, device=dev)
        post = torch.empty_like(logits) if want_post else None
        dec = torch.empty(B, T, self.y_dim, dtype=torch.int32, device=dev) if want_dec else None
        last = torch.empty(B, self.y_dim, dtype=torch.float32, device=dev) if want_last else None
        if state is not None:
            L.check(L.lib().avvad_lstm_forward_state(self.h, L.ptr(x_bf16), L.ptr(lens), B, T, L.ptr(state.h),
                                                     L.ptr(state.c), L.ptr(state.h), L.ptr(state.c), L.ptr(ws),
                                                     ws.numel(), L.ptr(logits), L.ptr(post), L.ptr(dec), L.ptr(last),
                                                     L.stream_ptr()))
        else:
            L.check(L.lib().avvad_lstm_forward(self.h, L.ptr(x_bf16), L.ptr(lens), B, T, L.ptr(ws), ws.numel(),
                                               L.ptr(logits), L.ptr(post), L.ptr(dec), L.ptr(last), L.stream_ptr()))
        return logits, post, dec, last


class LstmState:
    """Recurrent state of an :class:`Lstm` over ``B`` rows, updated in place by ``Lstm.forward(..., state=)``:
    ``h`` bf16 (layers, B, H) -- the h the recurrence feeds its MMA -- and ``c`` f32 (layers, B, H).  Zero when
    created, as at the start of a sequence."""

    def __init__(self, lstm: Lstm, B: int, device="cuda"):
        self.h = torch.zeros(lstm.layers, B, lstm.hidden, dtype=torch.bfloat16, device=device)
        self.c = torch.zeros(lstm.layers, B, lstm.hidden, dtype=torch.float32, device=device)

    def reset(self, rows=None):
        """Start new sequences in ``rows`` (an index, a list of indices or a bool mask; None = every row)."""
        if rows is None:
            self.h.zero_()
            self.c.zero_()
        else:
            self.h[:, rows] = 0
            self.c[:, rows] = 0

    def check(self, lstm: Lstm, B: int, device):
        shape = (lstm.layers, B, lstm.hidden)
        if tuple(self.h.shape) != shape or tuple(self.c.shape) != shape:
            raise ValueError(f"LstmState: expected h, c of shape {shape}, got {tuple(self.h.shape)}, "
                             f"{tuple(self.c.shape)}")
        if self.h.device != torch.device(device) or self.c.device != torch.device(device):
            raise ValueError("LstmState: state and input on different devices")
        assert self.h.dtype == torch.bfloat16 and self.c.dtype == torch.float32
        assert self.h.is_contiguous() and self.c.is_contiguous()


def _ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


def _state_pair(lstm: "Lstm", state, B: int, dev):
    """(h bf16, c f32), both (layers, B, H) contiguous, from an LstmState or an (h, c) pair (h of any float dtype is
    rounded to bf16, the h the recurrence feeds its MMA; None = a zero state)."""
    if isinstance(state, LstmState):
        state.check(lstm, B, dev)
        return state.h, state.c
    shape = (lstm.layers, B, lstm.hidden)

    def take(t, dtype):
        if t is None:
            return None
        if tuple(t.shape) != shape:
            raise ValueError(f"state: expected h, c of shape {shape}, got {tuple(t.shape)}")
        if t.device != torch.device(dev):
            raise ValueError("state and input on different devices")
        return t.detach().to(dtype).contiguous()
    return take(state[0], torch.bfloat16), take(state[1], torch.float32)


def lstm_train_forward(lstm: "Lstm", x_bf16: torch.Tensor, lengths, state=None):
    """Forward that keeps the activations BPTT needs.  Returns (logits (B,T,y_dim), tape).

    With `state` (an LstmState or an (h, c) pair of shape (layers, B, H)) the recurrence continues from it, the tape
    holds T + 1 positions per row (position 0 = the state; its pack carries a fourth entry that marks it stateful) and
    the call returns (logits, tape, (h_out, c_out)): h_out bf16 and c_out f32 (layers, B, H) at each row's last step
    (the input state for rows of length 0)."""
    L.require_cuda(x_bf16)
    B, T, ld = x_bf16.shape
    assert ld == lstm.ld and x_bf16.is_contiguous()
    dev = x_bf16.device
    lens = _i32(lengths, dev)
    if state is not None:
        h_in, c_in = _state_pair(lstm, state, B, dev)
        nbytes = L.lib().avvad_lstm_train_state_workspace_bytes(lstm.h, B, T)
    else:
        nbytes = L.lib().avvad_lstm_workspace_bytes(lstm.h, B, T)
    ws = lstm.ws.get(nbytes, dev)
    tb = L.lib().avvad_lstm_tape_bytes(lstm.layers, lstm.hidden, B, T + (state is not None))
    # The tape lives with the engine and is reused step after step: its address is baked into the cached CUDA graph of
    # the backward recurrence (csrc/lstm_train.cu), so a stable buffer means graph replays instead of re-captures.  A
    # second forward before the first one's backward (gradient accumulation over micro-batches) gets its own tape.
    tape = getattr(lstm, "_tape", None)
    if tape is None or tape.numel() != tb or tape.device != dev or getattr(lstm, "_tape_busy", False):
        tape = torch.empty(tb, dtype=torch.uint8, device=dev)
        if not getattr(lstm, "_tape_busy", False):
            lstm._tape = tape
    if tape is getattr(lstm, "_tape", None):
        lstm._tape_busy = True
    logits = torch.empty(B, T, lstm.y_dim, dtype=torch.float32, device=dev)
    if state is None:
        L.check(L.lib().avvad_lstm_forward_train(lstm.h, L.ptr(x_bf16), L.ptr(lens), B, T, L.ptr(ws), ws.numel(),
                                                 L.ptr(tape), tape.numel(), L.ptr(logits), L.stream_ptr()))
        return logits, (tape, lens, x_bf16)
    shape = (lstm.layers, B, lstm.hidden)
    h_out = torch.empty(shape, dtype=torch.bfloat16, device=dev)
    c_out = torch.empty(shape, dtype=torch.float32, device=dev)
    L.check(L.lib().avvad_lstm_forward_train_state(lstm.h, L.ptr(x_bf16), L.ptr(lens), B, T, L.ptr(h_in), L.ptr(c_in),
                                                   L.ptr(h_out), L.ptr(c_out), L.ptr(ws), ws.numel(), L.ptr(tape),
                                                   tape.numel(), L.ptr(logits), L.stream_ptr()))
    return logits, (tape, lens, x_bf16, "state"), (h_out, c_out)


def lstm_tape_views(lstm: "Lstm", tape, B: int, T: int):
    """Views into a training tape (inspection hook for the state tests): one (gates, c, h) triple per layer with
    gates bf16 (B, T, 4H) gate-interleaved (element 4u+g, g = i, f, g, o), c f32 (B, T, H) and h bf16 (B, T, H).
    `tape` is the byte tensor or the pack lstm_train_forward returns."""
    if isinstance(tape, tuple):
        tape = tape[0]
    H, Lyr = lstm.hidden, lstm.layers
    off = (C.c_int64 * (3 * Lyr))()
    L.check(L.lib().avvad_lstm_tape_layout(Lyr, H, B, T, off, 3 * Lyr))
    assert tape.dtype == torch.uint8 and tape.numel() >= L.lib().avvad_lstm_tape_bytes(Lyr, H, B, T)

    def view(o, numel, dtype, shape):
        nbytes = numel * torch.empty((), dtype=dtype).element_size()
        return tape[o:o + nbytes].view(dtype).view(shape)
    n = B * T * H
    return [(view(off[3 * l], 4 * n, torch.bfloat16, (B, T, 4 * H)), view(off[3 * l + 1], n, torch.float32, (B, T, H)),
             view(off[3 * l + 2], n, torch.bfloat16, (B, T, H))) for l in range(Lyr)]


def lstm_train_backward(lstm: "Lstm", tape_pack, dlogits: torch.Tensor, want_dx=False, d_state=None,
                        want_state_grad=False):
    """BPTT.  Returns dict(weight_ih=[...], weight_hh=[...], bias=[...], head_w, head_b, dx).

    For a stateful tape (lstm_train_forward with `state`): `d_state` = (dh_out, dc_out), the gradients w.r.t. the
    returned (h_out, c_out) (either may be None = zero), and with `want_state_grad` the dict also holds dh_in and
    dc_in, f32 (layers, B, H), the gradients w.r.t. the input state."""
    tape, lens, x_bf16 = tape_pack[:3]
    stateful = len(tape_pack) > 3
    if not stateful and (d_state is not None or want_state_grad):
        raise ValueError("state gradients need a tape from lstm_train_forward(..., state=)")
    B, T, _ = x_bf16.shape
    dev = x_bf16.device
    H, Lyr = lstm.hidden, lstm.layers
    dl = dlogits.detach().to(torch.float32).contiguous()
    if stateful:
        nbytes = L.lib().avvad_lstm_backward_state_workspace_bytes(lstm.h, B, T)
    else:
        nbytes = L.lib().avvad_lstm_backward_workspace_bytes(lstm.h, B, T)
    if not hasattr(lstm, "bws"):
        lstm.bws = _Workspace()
    ws = lstm.bws.get(nbytes, dev)
    dwi = [torch.empty(4 * H, lstm.input_size if l == 0 else H, dtype=torch.float32, device=dev) for l in range(Lyr)]
    dwh = [torch.empty(4 * H, H, dtype=torch.float32, device=dev) for _ in range(Lyr)]
    dbs = [torch.empty(4 * H, dtype=torch.float32, device=dev) for _ in range(Lyr)]
    dhw = torch.empty(lstm.y_dim, H, dtype=torch.float32, device=dev)
    dhb = torch.empty(lstm.y_dim, dtype=torch.float32, device=dev)
    dx = torch.empty(B, T, lstm.input_size, dtype=torch.float32, device=dev) if want_dx else None
    out = {}
    if stateful:
        shape = (Lyr, B, H)

        def grad_in(g):
            if g is None:
                return None
            assert tuple(g.shape) == shape, f"state gradient: expected shape {shape}, got {tuple(g.shape)}"
            return g.detach().to(device=dev, dtype=torch.float32).contiguous()
        dh_out, dc_out = (grad_in(g) for g in (d_state if d_state is not None else (None, None)))
        dh_in = torch.empty(shape, dtype=torch.float32, device=dev) if want_state_grad else None
        dc_in = torch.empty(shape, dtype=torch.float32, device=dev) if want_state_grad else None
        L.check(L.lib().avvad_lstm_backward_state(lstm.h, L.ptr(x_bf16), L.ptr(lens), B, T, L.ptr(tape), L.ptr(dl),
                                                  L.ptr(dh_out), L.ptr(dc_out), L.ptr(dh_in), L.ptr(dc_in), L.ptr(ws),
                                                  ws.numel(), _ptr_array(dwi), _ptr_array(dwh), _ptr_array(dbs),
                                                  L.ptr(dhw), L.ptr(dhb), L.ptr(dx), L.stream_ptr()))
        if want_state_grad:
            out = {"dh_in": dh_in, "dc_in": dc_in}
    else:
        L.check(L.lib().avvad_lstm_backward(lstm.h, L.ptr(x_bf16), L.ptr(lens), B, T, L.ptr(tape), L.ptr(dl),
                                            L.ptr(ws), ws.numel(), _ptr_array(dwi), _ptr_array(dwh), _ptr_array(dbs),
                                            L.ptr(dhw), L.ptr(dhb), L.ptr(dx), L.stream_ptr()))
    if tape is getattr(lstm, "_tape", None):
        lstm._tape_busy = False
    return {"weight_ih": dwi, "weight_hh": dwh, "bias": dbs, "head_w": dhw, "head_b": dhb, "dx": dx, **out}


def adam_step(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, step: int,
              lr=1e-4, betas=(0.9, 0.999), eps=1e-8):
    """In-place torch.optim.Adam update of one contiguous fp32 tensor."""
    assert param.is_contiguous() and grad.is_contiguous() and param.dtype == torch.float32
    L.check(L.lib().avvad_adam_step(L.ptr(param), L.ptr(grad), L.ptr(exp_avg), L.ptr(exp_avg_sq), param.numel(), lr,
                                    betas[0], betas[1], eps, step, L.stream_ptr()))


def launch_count() -> int:
    return int(L.lib().avvad_launch_count())


def profile_enable(on: bool):
    L.check(L.lib().avvad_profile_enable(1 if on else 0))


def profile_read(cat: int):
    """(ms, flops, launches) of the recorded tensor-core launches of one category."""
    ms, fl, n = C.c_double(), C.c_double(), C.c_uint64()
    L.check(L.lib().avvad_profile_read(cat, C.byref(ms), C.byref(fl), C.byref(n)))
    return ms.value, fl.value, n.value


def profile_clear():
    L.check(L.lib().avvad_profile_clear())


def profile_dump(cat: int, max_n=200000):
    """Per-launch (ms, flops) arrays of one category, in launch order."""
    import numpy as np

    ms = (C.c_double * max_n)()
    fl = (C.c_double * max_n)()
    n = int(L.lib().avvad_profile_dump(cat, ms, fl, max_n))
    return np.frombuffer(ms, dtype=np.float64, count=n).copy(), np.frombuffer(fl, dtype=np.float64, count=n).copy()


def batch_bce(logits: torch.Tensor, target: torch.Tensor, lengths, eps=1e-8, want_grad=False):
    """Sum over utterances of the per-utterance mean BCE (scripts/train_AV_net.py:298-301).
    Returns (loss 0-dim, per_utterance (B,), dlogits or None)."""
    L.require_cuda(logits, target)
    B, T, Y = logits.shape
    lg = logits.detach().to(torch.float32).contiguous()
    tg = target.detach().to(torch.float32).contiguous()
    lens = _i32(lengths, lg.device)
    loss = torch.empty(1, dtype=torch.float32, device=lg.device)
    per = torch.empty(B, dtype=torch.float32, device=lg.device)
    grad = torch.empty_like(lg) if want_grad else None
    L.check(L.lib().avvad_bce_loss(L.ptr(lg), L.ptr(tg), L.ptr(lens), B, T, Y, eps, L.ptr(loss), L.ptr(per),
                                   L.ptr(grad), L.stream_ptr()))
    return loss[0], per, grad


def batch_f1(logits: torch.Tensor, target: torch.Tensor, lengths, epsilon=1e-8):
    """Per-utterance (accuracy, precision, recall, f1) of sigmoid(logit) > 0.5 (packages/models/utils.py:164-203).
    logits/target (B,T) or (B,T,1).  Returns (metrics (B,4), decisions (B,T) int32)."""
    L.require_cuda(logits, target)
    lg = logits.detach().to(torch.float32).reshape(logits.shape[0], -1).contiguous()
    tg = target.detach().to(torch.float32).reshape(target.shape[0], -1).contiguous()
    B, T = lg.shape
    lens = _i32(lengths, lg.device)
    met = torch.empty(B, 4, dtype=torch.float32, device=lg.device)
    dec = torch.empty(B, T, dtype=torch.int32, device=lg.device)
    L.check(L.lib().avvad_f1_metrics(L.ptr(lg), L.ptr(tg), L.ptr(lens), B, T, epsilon, L.ptr(met), L.ptr(dec),
                                     L.stream_ptr()))
    return met, dec


class WaveNetEncoder:
    """Dilated valid Conv1d encoder (SURVEY W1) on the tcgen05 GEMM engine."""

    def __init__(self, filter_width, quantization_channel, dilations, residual_channel, dilation_channel,
                 bottleneck_width, pool_size):
        dil = (C.c_int32 * len(dilations))(*[int(d) for d in dilations])
        h = C.c_void_p()
        L.check(L.lib().avvad_wavenet_create(C.byref(h), filter_width, quantization_channel, dil, len(dilations),
                                             residual_channel, dilation_channel, bottleneck_width, pool_size))
        self.h = h
        self.n_dil = len(dilations)
        self.bottleneck, self.pool = bottleneck_width, pool_size
        self.ws = _Workspace()

    def __del__(self):
        try:
            if getattr(self, "h", None):
                L.lib().avvad_wavenet_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def load(self, sd: Dict[str, torch.Tensor], device):
        def put(kind, index, name):
            w = _f32(sd[name + ".weight"], device)
            b = _f32(sd[name + ".bias"], device) if (name + ".bias") in sd else None
            L.check(L.lib().avvad_wavenet_set_layer(self.h, kind, index, L.ptr(w), L.ptr(b), L.stream_ptr()))
            return w, b
        keep = [put(0, 0, "en_causal_layer"), put(3, 0, "bottleneck_layer")]
        for i in range(self.n_dil):
            keep.append(put(1, i, f"en_dilation_layer_stack.{i}"))
            keep.append(put(2, i, f"en_dense_layer_stack.{i}"))
        # weight shapes and bias presence in the backward's gradient order (WAVENET_LAYER_NAMES)
        self.grad_layout = [(tuple(sd[n + ".weight"].shape), (n + ".bias") in sd)
                            for n in wavenet_layer_names(self.n_dil)]
        torch.cuda.current_stream().synchronize()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        L.require_cuda(x)
        x = x.detach().to(torch.float32).contiguous()
        B, _, N = x.shape
        nbytes = L.lib().avvad_wavenet_workspace_bytes(self.h, B, N)
        ws = self.ws.get(nbytes, x.device)
        out = torch.empty(B, self.bottleneck, self.pool, dtype=torch.float32, device=x.device)
        L.check(L.lib().avvad_wavenet_encode(self.h, L.ptr(x), B, N, L.ptr(ws), ws.numel(), L.ptr(out), L.stream_ptr()))
        return out

    def forward_train(self, x: torch.Tensor):
        """(out, tape): ``forward``'s output, bit for bit, and the tape ``backward`` reads (its own buffer per call, so
        several forwards may precede their backwards)."""
        L.require_cuda(x)
        x = x.detach().to(torch.float32).contiguous()
        B, _, N = x.shape
        ws = self.ws.get(L.lib().avvad_wavenet_workspace_bytes(self.h, B, N), x.device)
        tape = torch.empty(max(int(L.lib().avvad_wavenet_tape_bytes(self.h, B, N)), 1), dtype=torch.uint8,
                           device=x.device)
        out = torch.empty(B, self.bottleneck, self.pool, dtype=torch.float32, device=x.device)
        L.check(L.lib().avvad_wavenet_encode_train(self.h, L.ptr(x), B, N, L.ptr(ws), ws.numel(), L.ptr(tape),
                                                   tape.numel(), L.ptr(out), L.stream_ptr()))
        return out, (x, tape)

    def backward(self, tape, dout: torch.Tensor, want_dx: bool = False):
        """Gradients from a ``forward_train`` tape and d loss / d out (any strides).  Returns (dx or None, grads), grads
        in ``wavenet_params`` order: weight (and bias, when the module has them) of en_causal_layer, then per layer
        en_dilation_layer_stack.i / en_dense_layer_stack.i, then bottleneck_layer, in PyTorch's layout."""
        x, tp = tape
        B, _, N = x.shape
        dout = dout.detach().to(device=x.device, dtype=torch.float32).contiguous()
        dws = [torch.empty(shape, dtype=torch.float32, device=x.device) for shape, _ in self.grad_layout]
        dbs = [torch.empty(shape[0], dtype=torch.float32, device=x.device) if has_b else None
               for shape, has_b in self.grad_layout]
        dx = torch.empty_like(x) if want_dx else None
        n = len(dws)
        pw = (C.c_void_p * n)(*[t.data_ptr() for t in dws])
        pb = (C.c_void_p * n)(*[t.data_ptr() if t is not None else None for t in dbs])
        ws = self.ws.get(L.lib().avvad_wavenet_backward_workspace_bytes(self.h, B, N), x.device)
        L.check(L.lib().avvad_wavenet_backward(self.h, L.ptr(x), B, N, L.ptr(tp), tp.numel(), L.ptr(dout), L.ptr(dx),
                                               pw, pb, L.ptr(ws), ws.numel(), L.stream_ptr()))
        grads = []
        for w, b in zip(dws, dbs):
            grads += [w] if b is None else [w, b]
        return dx, grads


def wavenet_layer_names(n_dilations: int):
    """Conv1d layers of the WaveNet encoder in the C ABI's gradient order."""
    names = ["en_causal_layer"]
    for i in range(n_dilations):
        names += [f"en_dilation_layer_stack.{i}", f"en_dense_layer_stack.{i}"]
    return names + ["bottleneck_layer"]
