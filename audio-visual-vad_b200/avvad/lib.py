"""ctypes binding of libavvad.so (the C-ABI boundary declared in include/avvad.h).

The product path has no CPU fallback: importing this module is cheap, but the first call to
:func:`lib` raises if the shared library has not been built (``python -c 'import
__graft_entry__ as g; g.build()'`` or ``make -C audio-visual-vad_b200/csrc``), and every compute
entry point raises :class:`AvvadError` on a box without a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libavvad.so")

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_f32p = C.POINTER(C.c_float)
VP = C.c_void_p

# name -> (restype, argtypes); every symbol include/avvad.h declares
PROTOTYPES = {
    "avvad_last_error": (C.c_char_p, []),
    "avvad_version": (C.c_int, []),
    "avvad_launch_count": (C.c_uint64, []),
    "avvad_profile_enable": (C.c_int, [C.c_int]),
    "avvad_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "avvad_profile_clear": (C.c_int, []),
    "avvad_profile_dump": (C.c_int64, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int64]),
    "avvad_debug_lstm_trace": (None, [VP]),
    "avvad_stft_num_frames": (C.c_int64, [C.c_int64, C.c_double, C.c_double, C.c_double, C.c_int]),
    "avvad_frontend_logpower": (C.c_int, [VP, C.c_int64, VP, VP, C.c_int32, C.c_int32, C.c_int, VP, VP, C.c_float,
                                          VP, VP, VP]),
    "avvad_stft": (C.c_int, [VP, C.c_int64, VP, VP, C.c_int32, C.c_int32, VP, VP]),
    "avvad_upsampled_length": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "avvad_upsample_gather": (C.c_int, [VP, C.c_int, VP, VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_float, C.c_float, C.c_float, C.c_int, VP, VP]),
    "avvad_upsample_index": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, VP, VP]),
    "avvad_resnet18_create": (C.c_int, [C.POINTER(VP)]),
    "avvad_resnet18_destroy": (None, [VP]),
    "avvad_resnet18_set_conv": (C.c_int, [VP, C.c_int, VP, VP, VP, VP, VP, C.c_float, VP]),
    "avvad_resnet18_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "avvad_resnet18_forward": (C.c_int, [VP, VP, C.c_int64, C.c_int64, VP, C.c_size_t, VP, VP, C.c_int64, C.c_int64,
                                         VP]),
    "avvad_resnet18_forward_u8": (C.c_int, [VP, VP, VP, VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                            C.c_float, C.c_float, C.c_float, C.c_int, C.c_int64, VP, C.c_size_t, VP, VP,
                                            C.c_int64, C.c_int64, VP]),
    "avvad_resnet18_forward_upto": (C.c_int, [VP, VP, C.c_int64, C.c_int, VP, C.c_size_t, VP, VP]),
    "avvad_resnet18_set_conv_train": (C.c_int, [VP, C.c_int, VP, VP, VP, VP]),
    "avvad_resnet18_train_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "avvad_resnet18_forward_train": (C.c_int, [VP, VP, C.c_int64, VP, C.c_size_t, C.c_float, C.c_float, VP, VP, VP, VP,
                                               C.c_int64, C.c_int64, VP]),
    "avvad_resnet18_tape_bytes": (C.c_size_t, [C.c_int64]),
    "avvad_resnet18_tape_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "avvad_resnet18_tape_layout": (C.c_int, [C.c_int64, c_i64p, C.c_int]),
    "avvad_resnet18_forward_tape": (C.c_int, [VP, VP, C.c_int64, VP, C.c_size_t, VP, C.c_size_t, C.c_float, C.c_float, VP,
                                              VP, VP, VP, C.c_int64, C.c_int64, VP]),
    "avvad_resnet18_backward_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "avvad_resnet18_backward": (C.c_int, [VP, VP, C.c_int64, VP, VP, VP, C.c_size_t, C.c_float, VP, VP, VP, VP]),
    "avvad_gemm_bf16": (C.c_int, [VP, C.c_int64, VP, C.c_int64, VP, VP, C.c_int64, C.c_int, C.c_int, C.c_int64,
                                  C.c_int64, C.c_int64, VP]),
    "avvad_conv2d_nhwc_bf16": (C.c_int, [VP, VP, VP, VP, VP, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_int, VP]),
    "avvad_dct_roi_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "avvad_dct_roi_decode": (C.c_int, [VP, C.c_int64, C.c_int, VP, VP, VP, C.c_size_t, VP]),
    "avvad_vad_labels": (C.c_int, [VP, C.c_int64, VP, VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, VP, VP,
                                   VP]),
    "avvad_ibm_labels": (C.c_int, [VP, VP, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, VP, VP, VP, VP]),
    "avvad_stats_accumulate": (C.c_int, [VP, VP, C.c_int32, C.c_int32, C.c_int32, VP, VP, VP]),
    "avvad_stats_finalize": (C.c_int, [VP, VP, C.c_double, C.c_int32, VP, VP, VP]),
    "avvad_feature_gather": (C.c_int, [VP, VP, VP, VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       VP, VP, C.c_int64, C.c_int64, VP]),
    "avvad_conv2d_nhwc_bf16_dual": (C.c_int, [VP, VP, VP, VP, VP, C.c_int64] + [C.c_int] * 13 + [VP]),
    "avvad_pack_rows_bf16": (C.c_int, [VP, C.c_int64, VP, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, VP]),
    "avvad_mcb_create": (C.c_int, [C.POINTER(VP)]),
    "avvad_mcb_destroy": (None, [VP]),
    "avvad_mcb_load": (C.c_int, [VP, VP, VP, VP, VP, VP, VP, VP, VP, C.c_float, VP]),
    "avvad_mcb_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "avvad_mcb_forward": (C.c_int, [VP, VP, VP, C.c_int64, VP, C.c_size_t, VP, C.c_int64, VP, VP]),
    "avvad_mcb_grouped_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "avvad_mcb_forward_grouped": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, VP, C.c_size_t, VP, C.c_int64, VP, VP]),
    "avvad_mcb_forward_grouped_norms": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, VP, VP, VP, C.c_size_t, VP,
                                                  C.c_int64, VP, VP]),
    "avvad_count_sketch_forward": (C.c_int, [VP, C.c_int64, C.c_int, C.c_int, VP, VP, VP, VP, VP]),
    "avvad_count_sketch_backward": (C.c_int, [VP, C.c_int64, C.c_int, C.c_int, VP, VP, VP, VP]),
    "avvad_mcb_raw_forward": (C.c_int, [VP] * 8 + [C.c_int64, VP, VP]),
    "avvad_mcb_raw_backward": (C.c_int, [VP] * 11 + [C.c_int64, VP, VP, VP]),
    "avvad_lzf_compress": (C.c_int64, [VP, C.c_int64, VP, C.c_int64, C.c_int, VP]),
    "avvad_lzf_decompress": (C.c_int64, [VP, C.c_int64, VP, C.c_int64]),
    "avvad_lstm_tape_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64, C.c_int64]),
    "avvad_lstm_tape_layout": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_int64, c_i64p, C.c_int]),
    "avvad_lstm_forward_train": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, C.c_size_t, VP, C.c_size_t, VP, VP]),
    "avvad_lstm_backward_workspace_bytes": (C.c_size_t, [VP, C.c_int64, C.c_int64]),
    "avvad_lstm_backward": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, VP, VP, C.c_size_t, VP, VP, VP, VP, VP, VP,
                                      VP]),
    "avvad_adam_step": (C.c_int, [VP, VP, VP, VP, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int64, VP]),
    "avvad_bce_loss": (C.c_int, [VP, VP, VP, C.c_int32, C.c_int32, C.c_int32, C.c_float, VP, VP, VP, VP]),
    "avvad_f1_metrics": (C.c_int, [VP, VP, VP, C.c_int32, C.c_int32, C.c_float, VP, VP, VP]),
    "avvad_wavenet_create": (C.c_int, [C.POINTER(VP), C.c_int, C.c_int, VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "avvad_wavenet_destroy": (None, [VP]),
    "avvad_wavenet_set_layer": (C.c_int, [VP, C.c_int, C.c_int, VP, VP, VP]),
    "avvad_wavenet_encoded_length": (C.c_int64, [VP, C.c_int64]),
    "avvad_wavenet_workspace_bytes": (C.c_size_t, [VP, C.c_int64, C.c_int64]),
    "avvad_wavenet_encode": (C.c_int, [VP, VP, C.c_int64, C.c_int64, VP, C.c_size_t, VP, VP]),
    "avvad_mcb_forward_train": (C.c_int, [VP, VP, VP, C.c_int64, VP, C.c_size_t, VP, VP, C.c_float, VP, VP, VP, C.c_int64,
                                          VP, VP]),
    "avvad_mcb_backward_bn": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, VP, VP]),
    "avvad_lstm_create": (C.c_int, [C.POINTER(VP), C.c_int, C.c_int, C.c_int, C.c_int]),
    "avvad_lstm_destroy": (None, [VP]),
    "avvad_lstm_set_layer": (C.c_int, [VP, C.c_int, VP, VP, VP, VP, VP]),
    "avvad_lstm_set_head": (C.c_int, [VP, VP, VP, VP]),
    "avvad_lstm_input_ld": (C.c_int64, [VP]),
    "avvad_lstm_workspace_bytes": (C.c_size_t, [VP, C.c_int64, C.c_int64]),
    "avvad_lstm_forward": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, C.c_size_t, VP, VP, VP, VP, VP]),
    "avvad_lstm_state_workspace_bytes": (C.c_size_t, [VP, C.c_int64, C.c_int64]),
    "avvad_lstm_forward_state": (C.c_int, [VP, VP, VP, C.c_int64, C.c_int64, VP, VP, VP, VP, VP, C.c_size_t, VP, VP,
                                           VP, VP, VP]),
}


class AvvadError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load libavvad.so once; fail loudly when it is missing (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AvvadError(
                f"{LIB_PATH} not found: build it with `make -C audio-visual-vad_b200/csrc` "
                "(or __graft_entry__.build()).  There is no CPU / PyTorch fallback for this path.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(l, name)  # AttributeError = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status: int):
    if status != 0:
        msg = lib().avvad_last_error()
        raise AvvadError(f"libavvad status {status}: {msg.decode() if msg else '?'}")


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    import torch

    if not torch.cuda.is_available():
        raise AvvadError("CUDA device required: the AV-VAD hot path has no CPU fallback")
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise AvvadError("expected CUDA tensors (the AV-VAD hot path has no CPU fallback)")
