"""Per-device CUDA engines behind the reference-compatible nn.Modules.

The modules in this package keep the reference's parameters/buffers (so ``state_dict`` keys,
``.to()``, ``DataParallel`` replication and checkpoint loading behave as in
sp-uhh/audio-visual-vad) but their ``forward`` bodies call libavvad through ``avvad.engine``.
Packed (BN-folded, bf16, gate-interleaved) weights are cached per device and re-packed whenever a
parameter's storage or version counter changes.
"""
from __future__ import annotations

import os
import sys

import torch

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _PKG_ROOT not in sys.path:  # make `import avvad` work when only `packages` is on sys.path
    sys.path.insert(0, _PKG_ROOT)

from avvad import engine as E  # noqa: E402
from avvad import lib as L  # noqa: E402


def _replica_parameters(module: torch.nn.Module):
    """(qualified name, tensor) of the parameter copies of an nn.DataParallel replica.  torch.nn.parallel.replicate
    empties ``_parameters`` of every replica module and re-attaches the broadcast copies as plain tensor attributes
    (listed in ``_former_parameters``), so ``parameters()`` / ``state_dict()`` of a replica see buffers only."""
    for prefix, mod in module.named_modules():
        former = getattr(mod, "_former_parameters", None)
        if former:
            for k, v in former.items():
                if v is not None:
                    yield (prefix + "." if prefix else "") + k, v


def all_parameters(module: torch.nn.Module):
    """``module.parameters()`` plus, inside an nn.DataParallel replica, the broadcast parameter copies."""
    return list(module.parameters()) + [v for _, v in _replica_parameters(module)]


def full_state_dict(module: torch.nn.Module):
    """name -> LIVE tensor object (Parameter / buffer, not the detached copies ``state_dict()`` hands out) for every
    entry of ``module.state_dict()``; also complete inside an nn.DataParallel replica (reference:
    scripts/train_AV_net.py:193 wraps the model in nn.parallel.DataParallel).  The engine caches key on these objects'
    (data_ptr, version, generation): the generation tag that marks raw-pointer updates (fused Adam, in-kernel running
    statistics) lives on the tensor OBJECT, so detached copies would never see it."""
    sd = dict(module.named_parameters(remove_duplicate=False))
    sd.update(dict(module.named_buffers(remove_duplicate=False)))
    for k, v in _replica_parameters(module):
        if k not in sd:
            sd[k] = v
    return sd


def bump_generation(*tensors):
    """Mark tensors whose storage was updated in place by a libavvad kernel (autograd's version counter does not see
    raw-pointer writes): BatchNorm running statistics after a training-mode forward, parameters after the fused Adam."""
    for t in tensors:
        t._avvad_gen = getattr(t, "_avvad_gen", 0) + 1


class EngineCache:
    """Per-device, per-sub-engine cache of the packed device weights (trunk folded for eval, trunk un-folded for
    train(), LSTM + head, MCB).  Every sub-engine has its OWN signature -- (data_ptr, version, generation) of exactly the
    tensors it packs -- so an optimiser step that changes the LSTM does not re-pack the frozen trunk (40 conv uploads and
    two stream synchronisations per step before), and `num_batches_tracked` (bumped every training forward) is in no
    signature at all."""

    def __init__(self):
        self.by_device = {}

    @staticmethod
    def signature(tensors):
        return tuple((t.data_ptr(), t._version, getattr(t, "_avvad_gen", 0)) for t in tensors)

    def get(self, device: torch.device, name: str, tensors, build, load):
        slot = self.by_device.setdefault((device.type, device.index), {})
        sig = self.signature(tensors)
        hit = slot.get(name)
        if hit is not None and hit[0] == sig:
            return hit[1]
        eng = hit[1] if hit is not None else build()
        load(eng)
        slot[name] = (sig, eng)
        return eng

    def shared(self, device: torch.device, name: str, build):
        """An object several sub-engines share (one ResNet18Trunk handle holds the eval AND the train weights)."""
        slot = self.by_device.setdefault((device.type, device.index), {})
        if name not in slot:
            slot[name] = build()
        return slot[name]


def select_state(sd, prefixes, running=True):
    """Tensors of a (full) state_dict under the given key prefixes, without num_batches_tracked (and without the
    BatchNorm running statistics when running=False: the train()-mode engines do not read them)."""
    out = []
    for k, v in sd.items():
        if not k.startswith(prefixes) or k.endswith("num_batches_tracked"):
            continue
        if not running and (k.endswith("running_mean") or k.endswith("running_var")):
            continue
        out.append(v)
    return out


def trunk_engine(cache: EngineCache, sd, device, training: bool):
    """The ResNet-18 engine with the weights the current mode needs: BN folded from the running statistics in eval(),
    raw convolution weights + BN affine parameters in train() (batch statistics)."""
    obj = cache.shared(device, "_trunk_handle", E.ResNet18Trunk)
    if training:
        return cache.get(device, "trunk_train", select_state(sd, ("features.",), running=False), lambda: obj,
                         lambda e: e.load_train(sd, device))
    return cache.get(device, "trunk_eval", select_state(sd, ("features.",)), lambda: obj, lambda e: e.load(sd, device))


class LstmHeadFunction(torch.autograd.Function):
    """Differentiable LSTM + Linear head on libavvad: forward keeps a tape, backward runs BPTT on the device and
    returns the gradients of the nn.LSTM / nn.Linear parameters in PyTorch's layout (and of the input when asked)."""

    @staticmethod
    def forward(ctx, lstm_engine, x_bf16, lengths, x_src, *params):
        logits, tape = E.lstm_train_forward(lstm_engine, x_bf16, lengths)
        ctx.lstm_engine = lstm_engine
        ctx.tape = tape
        ctx.n_params = len(params)
        ctx.want_dx = x_src is not None and x_src.requires_grad
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        eng = ctx.lstm_engine
        g = E.lstm_train_backward(eng, ctx.tape, dlogits, want_dx=ctx.want_dx)
        ctx.tape = None
        grads = []
        for l in range(eng.layers):  # parameter order: weight_ih, weight_hh, bias_ih, bias_hh per layer, then head
            grads += [g["weight_ih"][l], g["weight_hh"][l], g["bias"][l], g["bias"][l]]
        grads += [g["head_w"], g["head_b"]]
        return (None, None, None, g["dx"]) + tuple(grads)


class LstmHeadStateFunction(torch.autograd.Function):
    """LstmHeadFunction with nn.LSTM's ``hx``: ``h0`` (f32, rounded to bf16 for the kernel; its gradient is passed
    straight through the rounding) and ``c0`` (f32), both (layers, B, H), are differentiable inputs, and the final
    state ``h_n`` / ``c_n`` at each row's last valid step (f32) is a differentiable output next to the logits."""

    @staticmethod
    def forward(ctx, lstm_engine, x_bf16, lengths, x_src, h0, c0, *params):
        logits, tape, (h_n, c_n) = E.lstm_train_forward(lstm_engine, x_bf16, lengths, state=(h0, c0))
        ctx.lstm_engine = lstm_engine
        ctx.tape = tape
        ctx.want_dx = x_src is not None and x_src.requires_grad
        ctx.want_state = h0.requires_grad or c0.requires_grad
        return logits, h_n.float(), c_n

    @staticmethod
    def backward(ctx, dlogits, dh_n, dc_n):
        eng = ctx.lstm_engine
        g = E.lstm_train_backward(eng, ctx.tape, dlogits, want_dx=ctx.want_dx, d_state=(dh_n, dc_n),
                                  want_state_grad=ctx.want_state)
        ctx.tape = None
        grads = []
        for l in range(eng.layers):
            grads += [g["weight_ih"][l], g["weight_hh"][l], g["bias"][l], g["bias"][l]]
        grads += [g["head_w"], g["head_b"]]
        return (None, None, None, g["dx"], g.get("dh_in"), g.get("dc_in")) + tuple(grads)


def lstm_hx(hx, layers: int, B: int, H: int, device):
    """Checks nn.LSTM's ``hx = (h0, c0)``, each (num_layers, B, H), and returns it as f32 tensors on ``device``."""
    if not (isinstance(hx, (tuple, list)) and len(hx) == 2):
        raise ValueError("hx must be a pair (h0, c0)")
    h0, c0 = hx
    shape = (layers, B, H)
    if tuple(h0.shape) != shape or tuple(c0.shape) != shape:
        raise ValueError(f"hx: expected h0, c0 of shape {shape}, got {tuple(h0.shape)}, {tuple(c0.shape)}")
    return h0.to(device=device, dtype=torch.float32), c0.to(device=device, dtype=torch.float32)


def lstm_with_hx(lstm_engine, x_bf16, lengths, x_src, hx, params, train: bool):
    """(logits, (h_n, c_n)) of the LSTM + head continued from ``hx``: the autograd path when ``train``, else the
    inference recurrence with a state (``Lstm.forward(state=)``).  h_n / c_n are f32 (num_layers, B, H), taken at each
    row's last valid step as nn.LSTM returns them for packed input (``hx`` itself for rows of length 0)."""
    B = x_bf16.shape[0]
    h0, c0 = lstm_hx(hx, lstm_engine.layers, B, lstm_engine.hidden, x_bf16.device)
    if train:
        logits, h_n, c_n = LstmHeadStateFunction.apply(lstm_engine, x_bf16, lengths, x_src, h0, c0, *params)
        return logits, (h_n, c_n)
    state = E.LstmState(lstm_engine, B, x_bf16.device)
    state.h.copy_(h0.detach())
    state.c.copy_(c0.detach())
    logits, _, _, _ = lstm_engine.forward(x_bf16, lengths, state=state)
    return logits, (state.h.float(), state.c)


class McbBnFunction(torch.autograd.Function):
    """Training-mode MCB fusion.  Fills the bf16 LSTM operand buffer (side effect) and returns a zero-storage fp32
    proxy of its shape through which the LSTM's input gradient reaches the BatchNorm1d affine parameters (the only
    trainable tensors upstream of the LSTM: the sketches are buffers and the ResNet is frozen)."""

    @staticmethod
    def forward(ctx, mcb_engine, audio, feat, x_bf16, bn, gamma, beta):
        ws, rows = E.mcb_forward_train(mcb_engine, audio, feat, gamma.detach(), beta.detach(), bn.running_mean,
                                       bn.running_var, x_bf16.view(-1, x_bf16.shape[-1]), momentum=bn.momentum)
        ctx.mcb_engine, ctx.ws, ctx.rows = mcb_engine, ws, rows
        B, T, _ = x_bf16.shape
        return torch.zeros(1, device=x_bf16.device).expand(B, T, 1024)

    @staticmethod
    def backward(ctx, dx):
        dg, db = E.mcb_backward_bn(ctx.mcb_engine, ctx.ws, ctx.rows, dx)
        ctx.ws = None
        return None, None, None, None, None, dg, db


class TrunkFunction(torch.autograd.Function):
    """Differentiable training-mode ResNet-18 trunk on libavvad: forward keeps a tape, backward runs the device
    dgrad / wgrad / BatchNorm / pooling gradients (csrc/resnet_bwd.cuh) and returns the gradients of the 20 convolution
    weights and 40 BatchNorm affine parameters in the order `trunk_params` lists them.  This is what makes
    scripts/train_video_net.py -- which leaves the trunk trainable -- run unchanged."""

    @staticmethod
    def forward(ctx, trunk_engine, frames, running, *params):
        feat, tape = trunk_engine.forward_tape(frames, running)
        ctx.trunk_engine, ctx.tape, ctx.frames = trunk_engine, tape, frames
        return feat

    @staticmethod
    def backward(ctx, dfeat):
        dw, dg, db = ctx.trunk_engine.backward(ctx.frames, ctx.tape, dfeat)
        ctx.tape = None
        grads = []
        for i in range(20):  # parameter order of trunk_params: conv weight, bn weight, bn bias per layer
            grads += [dw[i], dg[i], db[i]]
        return (None, None, None) + tuple(grads)


class WaveNetFunction(torch.autograd.Function):
    """Differentiable WaveNet encoder on libavvad: forward keeps a tape (its output is the inference output, bit for
    bit), backward runs the device backward (csrc/wavenet_bwd.cuh) and returns the gradients of the Conv1d parameters
    in the order `wavenet_params` lists them, and of the input when it requires grad.  The input and the tape go
    through save_for_backward: an in-place change of x before the backward, or a second backward without
    retain_graph=True, raises autograd's own error."""

    @staticmethod
    def forward(ctx, wavenet_engine, x, *params):
        out, (xt, tape) = wavenet_engine.forward_train(x)
        ctx.wavenet_engine = wavenet_engine
        ctx.save_for_backward(x, xt, tape)
        ctx.want_dx = x.requires_grad
        return out

    @staticmethod
    def backward(ctx, dout):
        _, xt, tape = ctx.saved_tensors
        dx, grads = ctx.wavenet_engine.backward((xt, tape), dout, want_dx=ctx.want_dx)
        return (None, dx) + tuple(grads)


def wavenet_params(module: torch.nn.Module):
    """Weight (and bias, when present) of every Conv1d of a wavenet_autoencoder in the C ABI's gradient order.  Read
    through the attributes, so inside an nn.DataParallel replica these are the broadcast copies."""
    ps = []
    for name in E.wavenet_layer_names(len(module.dilations)):
        conv = module.get_submodule(name)
        ps += [conv.weight] + ([conv.bias] if conv.bias is not None else [])
    return ps


def trunk_params(features: torch.nn.Module):
    """(conv.weight, bn.weight, bn.bias) of the 20 conv layers in libavvad's layer order."""
    ps = []
    for ck, bk in E.RESNET_LAYER_KEYS:
        bn = features.get_submodule(bk)
        ps += [features.get_submodule(ck).weight, bn.weight, bn.bias]
    return ps


def trunk_bn_modules(features: torch.nn.Module):
    """The 20 BatchNorm2d modules of the trunk in libavvad's conv-layer order."""
    return [features.get_submodule(bk) for _, bk in E.RESNET_LAYER_KEYS]


def lstm_params(lstm: torch.nn.LSTM, head: torch.nn.Linear):
    ps = []
    for l in range(lstm.num_layers):
        ps += [getattr(lstm, f"weight_ih_l{l}"), getattr(lstm, f"weight_hh_l{l}"), getattr(lstm, f"bias_ih_l{l}"),
               getattr(lstm, f"bias_hh_l{l}")]
    return ps + [head.weight, head.bias]


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(lr, betas, eps) semantics (no weight decay / amsgrad) with the update done by libavvad."""

    def __init__(self, params, lr=1e-4, betas=(0.9, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))

    @torch.no_grad()
    def step(self, closure=None):
        for group in self.param_groups:
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p)
                    st["exp_avg_sq"] = torch.zeros_like(p)
                st["step"] += 1
                E.adam_step(p.data, p.grad.contiguous(), st["exp_avg"], st["exp_avg_sq"], st["step"], group["lr"],
                            group["betas"], group["eps"])
                # the in-place kernel bypasses autograd's version counter: bump a generation tag so that the packed
                # (bf16, gate-interleaved) weight caches of the engines are refreshed on the next forward
                bump_generation(p)


def on_input_device(forward):
    """Runs a module's forward with the CUDA device of its first tensor argument made current.  libavvad launches on
    the calling thread's current device and stream, whereas the reference's evaluation workers only ever call
    ``classifier.to(device)`` with an integer index (scripts/evaluate_AV_net.py:253, device = 4 + i % nb_devices) and
    never ``torch.cuda.set_device`` -- PyTorch's own ops switch devices per call, so these modules must too."""
    import functools

    @functools.wraps(forward)
    def wrapper(self, *args, **kwargs):
        for t in args:
            if isinstance(t, torch.Tensor) and t.is_cuda:
                with torch.cuda.device(t.device):
                    return forward(self, *args, **kwargs)
        return forward(self, *args, **kwargs)
    return wrapper


def device_of(*tensors) -> torch.device:
    L.require_cuda(*tensors)
    return tensors[0].device
