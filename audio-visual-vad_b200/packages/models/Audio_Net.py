"""Audio-only VAD network (reference: packages/models/Audio_Net.py:11-68); forward on libavvad."""
import torch
import torch.nn as nn

from .utils import weights_init_normal
from ._engine import (E, EngineCache, LstmHeadFunction, all_parameters, device_of, full_state_dict, lstm_params,
                      lstm_with_hx, on_input_device, select_state)


class DeepVAD_audio(nn.Module):
    def __init__(self, lstm_layers, lstm_hidden_size, y_dim):
        super().__init__()
        self.lstm_input_size = 513
        self.lstm_layers = lstm_layers
        self.lstm_hidden_size = lstm_hidden_size
        self.y_dim = y_dim
        self.lstm_audio = nn.LSTM(input_size=self.lstm_input_size, hidden_size=self.lstm_hidden_size,
                                  num_layers=self.lstm_layers, bidirectional=False)
        self.vad_audio = nn.Linear(self.lstm_hidden_size, y_dim)
        self.dropout = nn.Dropout(p=0.5)
        object.__setattr__(self, "_engines", EngineCache())

    def __getstate__(self):
        d = self.__dict__.copy()
        d.pop("_engines", None)
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)
        object.__setattr__(self, "_engines", EngineCache())

    def weight_init(self, mean=0.0, std=0.02):
        for m in self.named_parameters():
            weights_init_normal(m, mean=mean, std=std)

    def _build(self, device):
        sd = full_state_dict(self)
        return {"lstm": self._engines.get(device, "lstm", select_state(sd, ("lstm_audio.", "vad_audio.")),
                                          lambda: E.Lstm(self.lstm_layers, self.lstm_input_size, self.lstm_hidden_size,
                                                         self.y_dim),
                                          lambda e: e.load(sd, device, "lstm_audio", "vad_audio"))}

    @on_input_device
    def forward(self, x, lengths, return_posteriors=False, hx=None):
        """x (B,T,513) standardised log-power, lengths -> logits (B,T,y_dim).

        ``hx = (h0, c0)``, each (lstm_layers, B, H) as for nn.LSTM: the LSTM continues from that state and the call
        returns ``(logits, (h_n, c_n))`` with the state at each row's last valid step; in a training step gradients
        flow to h0 / c0 and from h_n / c_n.  Feeding h_n / c_n (detached) into the next block of the same utterances
        trains it in blocks (truncated BPTT)."""
        if hx is not None and return_posteriors:
            raise ValueError("hx: posteriors are not returned with a state; apply a sigmoid to the logits")
        device = device_of(x)
        eng = self._build(device)
        B, T, F = x.shape
        xb = eng["lstm"].new_input(B, T, device)
        E.pack_rows_bf16(x.detach().to(torch.float32).reshape(B * T, F).contiguous(), xb.view(B * T, -1), 0, False)
        train = torch.is_grad_enabled() and any(p.requires_grad for p in all_parameters(self))
        if hx is not None:
            return lstm_with_hx(eng["lstm"], xb, lengths, x if x.requires_grad else None, hx,
                                lstm_params(self.lstm_audio, self.vad_audio), train)
        if train:
            # training step: forward keeps a tape, loss.backward() runs BPTT on the device (SURVEY O1)
            return LstmHeadFunction.apply(eng["lstm"], xb, lengths, x if x.requires_grad else None,
                                          *lstm_params(self.lstm_audio, self.vad_audio))
        logits, post, dec, _ = eng["lstm"].forward(xb, lengths, want_post=return_posteriors,
                                                   want_dec=return_posteriors)
        if return_posteriors:
            return logits, post, dec
        return logits
