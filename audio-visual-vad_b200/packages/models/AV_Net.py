"""Audio-visual VAD network -- same class, constructor, parameters and state_dict as the reference
(packages/models/AV_Net.py:12-141); ``forward`` runs on libavvad (sm_100a) instead of cuDNN/ATen."""
import torch
import torch.nn as nn
import torchvision.models as models

from .compact_bilinear_pooling import CompactBilinearPooling
from .utils import weights_init_normal
from ._engine import (E, EngineCache, LstmHeadFunction, McbBnFunction, TrunkFunction, all_parameters, bump_generation,
                      device_of, full_state_dict, lstm_params, lstm_with_hx, on_input_device, select_state,
                      trunk_bn_modules, trunk_engine, trunk_params)


class DeepVAD_AV(nn.Module):
    def __init__(self, lstm_layers, lstm_hidden_size, y_dim, use_mcb=False, eps=1e-8):
        super().__init__()
        self.lstm_layers = lstm_layers
        self.lstm_hidden_size = lstm_hidden_size
        self.y_dim = y_dim
        self.dropout = nn.Dropout(p=0.05)
        self.use_mcb = use_mcb
        self.eps = eps
        # Extension (default off = the reference's semantics): in eval(), normalise every utterance's MCB output by its
        # OWN L2 norm over its `lengths[b]` valid frames, so ONE batched forward returns what the reference returns
        # when it is called once per utterance, as scripts/evaluate_AV_net.py:186-236 does (x[None], v[None],
        # lengths = [T]); rows behind an utterance's length are ignored (they do not exist in those calls).
        self.norm_per_utterance = False

        # parameter containers only: the child named 'features' must exist (train_AV_net.py:242-245)
        resnet = models.resnet18(weights=None)
        self.num_video_ftrs = 512
        self.features = nn.Sequential(*list(resnet.children())[:-1])
        self.bn = nn.BatchNorm1d(self.num_video_ftrs, eps=self.eps, momentum=0.1, affine=True)  # unused, kept for keys
        self.num_audio_ftrs = 513
        if self.use_mcb:
            self.mcb_output_size = 1024
            self.lstm_input_size = self.mcb_output_size
            self.mcb = CompactBilinearPooling(self.num_audio_ftrs, self.num_video_ftrs, self.mcb_output_size)
            self.mcb_bn = nn.BatchNorm1d(self.mcb_output_size, eps=self.eps, momentum=0.1, affine=True)
        else:
            self.lstm_input_size = self.num_audio_ftrs + self.num_video_ftrs
        self.lstm_merged = nn.LSTM(input_size=self.lstm_input_size, hidden_size=self.lstm_hidden_size,
                                   num_layers=self.lstm_layers, bidirectional=False)
        self.vad_merged = nn.Linear(self.lstm_hidden_size, y_dim)
        object.__setattr__(self, "_engines", EngineCache())

    def __getstate__(self):  # ctypes handles are per-process: drop them when pickled (mp spawn)
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
        """Sub-engines for `device`, each re-packed only when one of ITS tensors changed (see EngineCache)."""
        sd = full_state_dict(self)
        c = self._engines
        eng = {"trunk": trunk_engine(c, sd, device, self.training)}
        eng["lstm"] = c.get(device, "lstm", select_state(sd, ("lstm_merged.", "vad_merged.")),
                            lambda: E.Lstm(self.lstm_layers, self.lstm_input_size, self.lstm_hidden_size, self.y_dim),
                            lambda e: e.load(sd, device, "lstm_merged", "vad_merged"))
        eng["mcb"] = None
        if self.use_mcb:
            # train(): gamma / beta / running statistics are passed per call, only the sketches are packed
            keys = ("mcb.",) if self.training else ("mcb.", "mcb_bn.")
            eng["mcb"] = c.get(device, "mcb_train" if self.training else "mcb_eval", select_state(sd, keys),
                               lambda: c.shared(device, "_mcb_handle", E.Mcb), lambda e: e.load(sd, device, self.eps))
        return eng

    @on_input_device
    def forward(self, audio, video, lengths, return_posteriors=False, hx=None):
        """audio (B,T,513), video (B,T,67,67), lengths list / CPU / CUDA tensor -> logits (B,T,y_dim).

        ``hx = (h0, c0)``, each (lstm_layers, B, H) as for nn.LSTM: the LSTM continues from that state and the call
        returns ``(logits, (h_n, c_n))`` with the state at each row's last valid step; in a training step gradients
        flow to h0 / c0 and from h_n / c_n.  Feeding h_n / c_n (detached) into the next block of the same utterances
        trains it in blocks (truncated BPTT).  Blocks of one utterance are separate calls, so the quantities a call
        computes over all its frames -- train()-mode BatchNorm statistics and, with MCB, the L2 norm of the fused features -- are per block: the caller decides
        whether that is what it wants."""
        if hx is not None and return_posteriors:
            raise ValueError("hx: posteriors are not returned with a state; apply a sigmoid to the logits")
        device = device_of(audio, video)
        eng = self._build(device)
        batch, frames, height, width = video.size()
        M = batch * frames
        x = eng["lstm"].new_input(batch, frames, device)
        xv = x.view(M, x.shape[-1])
        vid = video.detach().to(torch.float32).reshape(M, height, width)
        aud = audio.detach().to(torch.float32).reshape(M, self.num_audio_ftrs).contiguous()
        # eval() forward is inference only (detached logits, folded BN); the autograd path is the train() step
        need_grad = self.training and torch.is_grad_enabled() and any(p.requires_grad for p in all_parameters(self))
        trunk_trainable = need_grad and any(p.requires_grad for p in all_parameters(self.features))

        # ---- video branch: batch-statistics BN while the module is in train() (train_AV_net.py:253), folded BN in eval()
        def trunk(feat_bf16=None, col_off=0, want_f32=True):
            if self.training:
                bns = trunk_bn_modules(self.features)
                running = [(b.running_mean, b.running_var) for b in bns]
                if trunk_trainable:   # features with a tape (differentiable), packed into the operand below
                    out = TrunkFunction.apply(eng["trunk"], vid, running, *trunk_params(self.features))
                else:
                    out = eng["trunk"].forward_train(vid, running, feat_bf16=feat_bf16, col_off=col_off,
                                                     want_f32=want_f32)
                for b in bns:
                    b.num_batches_tracked += 1
                    bump_generation(b.running_mean, b.running_var)
                return out
            return eng["trunk"].forward(vid, feat_bf16=feat_bf16, col_off=col_off, want_f32=want_f32)

        proxy = None
        if self.use_mcb:
            feat = trunk()
            if trunk_trainable:
                # Trainable trunk under MCB (train_AV_net.py with 'features' left trainable): the fusion of AV_Net.py:111-121
                # as differentiable pieces -- the stand-alone CompactBilinearPooling module (device sketch + FFT kernels
                # forward and backward, avvad_mcb_raw_*), signed sqrt, whole-tensor L2 norm (detached, as in the
                # reference) and the module's BatchNorm1d as PyTorch device ops -- so that the LSTM's input gradient
                # reaches the device ResNet backward.  The frozen-trunk case below stays on the fused MCB kernels.
                m_raw = self.mcb(aud.view(batch, frames, -1), feat.view(batch, frames, -1))
                y = torch.sign(m_raw) * torch.sqrt(torch.abs(m_raw) + self.eps)
                y = y / torch.norm(y, p=2).detach()
                y = self.mcb_bn(y.view(M, 1024)).view(batch, frames, 1024)
                bump_generation(self.mcb_bn.running_mean, self.mcb_bn.running_var)
                E.pack_rows_bf16(y.detach().reshape(M, 1024).contiguous(), xv, 0, False)
                proxy = y
            elif self.training:
                proxy = McbBnFunction.apply(eng["mcb"], aud, feat, x, self.mcb_bn, self.mcb_bn.weight, self.mcb_bn.bias)
                self.mcb_bn.num_batches_tracked += 1
                bump_generation(self.mcb_bn.running_mean, self.mcb_bn.running_var)
            elif self.norm_per_utterance:
                eng["mcb"].forward_grouped(aud, feat, lengths, frames, out_bf16=xv)
            else:
                eng["mcb"].forward(aud, feat, out_bf16=xv)
        else:
            E.pack_rows_bf16(aud, xv, 0, False)
            feat = trunk(feat_bf16=xv, col_off=self.num_audio_ftrs, want_f32=False)
            if trunk_trainable:
                E.pack_rows_bf16(feat.detach(), xv, self.num_audio_ftrs, False)
                # the LSTM's input gradient (B,T,1025) reaches the trunk through this concatenation (AV_Net.py:124)
                proxy = torch.cat([aud.view(batch, frames, -1), feat.view(batch, frames, -1)], dim=2)
        if hx is not None:
            return lstm_with_hx(eng["lstm"], x, lengths, proxy, hx, lstm_params(self.lstm_merged, self.vad_merged),
                                need_grad)
        if need_grad:
            return LstmHeadFunction.apply(eng["lstm"], x, lengths, proxy,
                                          *lstm_params(self.lstm_merged, self.vad_merged))
        logits, post, dec, _ = eng["lstm"].forward(x, lengths, want_post=return_posteriors,
                                                   want_dec=return_posteriors)
        if return_posteriors:
            return logits, post, dec
        return logits
