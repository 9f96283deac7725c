"""WaveNet-style encoder with the reference's constructor and parameters
(packages/models/wavenet_autoencoder.py:7-108); `_encode` / `forward` run on libavvad (csrc/wavenet.cu)."""
import warnings

import torch
import torch.nn as nn

from ._engine import E, EngineCache, WaveNetFunction, device_of, full_state_dict, on_input_device, wavenet_params


class wavenet_autoencoder(nn.Module):
    def __init__(self, filter_width, quantization_channel, dilations, en_residual_channel, en_dilation_channel,
                 en_bottleneck_width, en_pool_kernel_size, use_bias):
        super().__init__()
        self.filter_width = filter_width
        self.quantization_channel = quantization_channel
        self.dilations = dilations
        self.en_residual_channel = en_residual_channel
        self.en_dilation_channel = en_dilation_channel
        self.en_bottleneck_width = en_bottleneck_width
        self.en_pool_kernel_size = en_pool_kernel_size
        self.use_bias = use_bias
        self.receptive_field = (filter_width - 1) * (sum(dilations) + 1) + 1
        # same registration order / names as the reference (_init_encoding, then _init_causal_layer)
        self.en_dilation_layer_stack = nn.ModuleList()
        self.en_dense_layer_stack = nn.ModuleList()
        for d in dilations:
            self.en_dilation_layer_stack.append(nn.Conv1d(en_residual_channel, en_dilation_channel, filter_width,
                                                          dilation=d, bias=use_bias))
            self.en_dense_layer_stack.append(nn.Conv1d(en_dilation_channel, en_residual_channel, 1, bias=use_bias))
        self.en_causal_layer = nn.Conv1d(quantization_channel, en_residual_channel, filter_width, bias=use_bias)
        self.bottleneck_layer = nn.Conv1d(en_residual_channel, en_bottleneck_width, 1, bias=use_bias)
        object.__setattr__(self, "_engines", EngineCache())

    def __getstate__(self):
        d = self.__dict__.copy()
        d.pop("_engines", None)
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        object.__setattr__(self, "_engines", EngineCache())

    def _build(self, device):
        sd = full_state_dict(self)
        return self._engines.get(device, "encoder", list(sd.values()),
                                 lambda: E.WaveNetEncoder(self.filter_width, self.quantization_channel,
                                                          list(self.dilations), self.en_residual_channel,
                                                          self.en_dilation_channel, self.en_bottleneck_width,
                                                          self.en_pool_kernel_size),
                                 lambda e: e.load(sd, device))

    def _encode(self, sample):
        device = device_of(sample)
        eng = self._build(device)
        if torch.is_grad_enabled():
            params = wavenet_params(self)
            want_params = any(p.requires_grad for p in params)
            # Differentiable when x requires grad, or when a parameter does in train() mode.  In eval() the parameters'
            # requires_grad alone keeps the inference output (no grad_fn, so `.numpy()` works on it as it always
            # has); the values are the same either way, the encoder has no mode-dependent layer.
            if sample.requires_grad or (want_params and self.training):
                # the forward keeps a tape (its output is the inference output, bit for bit) and loss.backward() runs
                # the device backward (csrc/wavenet_bwd.cuh)
                return WaveNetFunction.apply(eng, sample, *params)
            if want_params:
                warnings.warn("wavenet_autoencoder in eval() returns an output without a graph to its parameters; "
                              "call train() to train them (the values are identical in both modes) or run under "
                              "torch.no_grad()", stacklevel=3)
        return eng.forward(sample)

    @on_input_device
    def forward(self, wave_sample):
        return self._encode(wave_sample)
