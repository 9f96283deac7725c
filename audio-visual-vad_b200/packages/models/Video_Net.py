"""Video-only VAD network (reference: packages/models/Video_Net.py:12-125); forward on libavvad."""
import torch
import torch.nn as nn
import torchvision.models as models

from .utils import weights_init_normal, method1, method3  # noqa: F401  (re-exported like the reference)
from ._engine import (E, EngineCache, LstmHeadFunction, TrunkFunction, all_parameters, bump_generation, device_of,
                      full_state_dict, lstm_params, lstm_with_hx, on_input_device, select_state, trunk_bn_modules,
                      trunk_engine, trunk_params)


class DeepVAD_video(nn.Module):
    def __init__(self, lstm_layers, lstm_hidden_size, y_dim):
        super().__init__()
        resnet = models.resnet18(weights=None)
        self.lstm_input_size = 512
        self.lstm_layers = lstm_layers
        self.lstm_hidden_size = lstm_hidden_size
        self.y_dim = y_dim
        self.features = nn.Sequential(*list(resnet.children())[:-1])
        self.mean = torch.as_tensor([0.485, 0.456, 0.406])
        self.std = torch.as_tensor([0.229, 0.224, 0.225])
        self.lstm_video = nn.LSTM(input_size=self.lstm_input_size, hidden_size=self.lstm_hidden_size,
                                  num_layers=self.lstm_layers, bidirectional=False)
        self.vad_video = nn.Linear(self.lstm_hidden_size, y_dim)
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
        c = self._engines
        return {"trunk": trunk_engine(c, sd, device, self.training),
                "lstm": c.get(device, "lstm", select_state(sd, ("lstm_video.", "vad_video.")),
                              lambda: E.Lstm(self.lstm_layers, self.lstm_input_size, self.lstm_hidden_size, self.y_dim),
                              lambda e: e.load(sd, device, "lstm_video", "vad_video"))}

    @on_input_device
    def forward(self, x, lengths, return_last=False, hx=None):
        """x (B,T,67,67), lengths -> logits (B,T,y_dim), or (B,y_dim) at the last valid step.

        ``hx = (h0, c0)``, each (lstm_layers, B, H) as for nn.LSTM: the LSTM continues from that state and the call
        returns ``(logits, (h_n, c_n))`` with the state at each row's last valid step; in a training step gradients
        flow to h0 / c0 and from h_n / c_n.  Feeding h_n / c_n (detached) into the next block of the same utterances
        trains it in blocks (truncated BPTT).  Blocks of one utterance are separate calls, so the quantities a call
        computes over all its frames -- train()-mode BatchNorm statistics -- are per block: the caller decides
        whether that is what it wants."""
        if hx is not None and return_last:
            raise ValueError("hx and return_last=True cannot be combined: with hx the call returns (logits, (h_n, c_n))")
        device = device_of(x)
        eng = self._build(device)
        batch, frames, height, width = x.size()
        M = batch * frames
        xb = eng["lstm"].new_input(batch, frames, device)
        vid = x.detach().to(torch.float32).reshape(M, height, width)
        # eval() forward is inference only (detached logits, folded BN).  train(): batch-statistics BatchNorm; the LSTM +
        # head train through the device BPTT, and a trainable trunk -- scripts/train_video_net.py:145-173 hands every
        # parameter to Adam -- through the device dgrad / wgrad / BatchNorm backward (TrunkFunction); a frozen trunk
        # (scripts/train_AV_net.py:241-245 style) takes the cheaper forward without a tape.
        need_grad = self.training and torch.is_grad_enabled() and any(p.requires_grad for p in all_parameters(self))
        trunk_trainable = need_grad and any(p.requires_grad for p in all_parameters(self.features))
        if need_grad and return_last:
            raise NotImplementedError("return_last=True has no training path (unused by the scripts)")
        x_src = None
        if self.training:
            bns = trunk_bn_modules(self.features)
            running = [(b.running_mean, b.running_var) for b in bns]
            if trunk_trainable:
                feat = TrunkFunction.apply(eng["trunk"], vid, running, *trunk_params(self.features))
                E.pack_rows_bf16(feat.detach(), xb.view(M, -1), 0, False)
                x_src = feat.view(batch, frames, self.lstm_input_size)
            else:
                eng["trunk"].forward_train(vid, running, feat_bf16=xb.view(M, -1), col_off=0, want_f32=False)
            for b in bns:
                b.num_batches_tracked += 1
                bump_generation(b.running_mean, b.running_var)
        else:
            eng["trunk"].forward(vid, feat_bf16=xb.view(M, -1), col_off=0, want_f32=False)
        if hx is not None:
            return lstm_with_hx(eng["lstm"], xb, lengths, x_src, hx, lstm_params(self.lstm_video, self.vad_video),
                                need_grad)
        if need_grad:
            return LstmHeadFunction.apply(eng["lstm"], xb, lengths, x_src, *lstm_params(self.lstm_video, self.vad_video))
        logits, _, _, last = eng["lstm"].forward(xb, lengths, want_last=return_last)
        return last if return_last else logits
