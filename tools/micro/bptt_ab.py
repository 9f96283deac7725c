#!/usr/bin/env python
"""BPTT A/B: device time of avvad_lstm_backward (2 x LSTM-1024 + head) and its gradients against another configuration
(AVVAD_BPTT_WAVEFRONT=0 = layers back to back instead of the merged-GEMM wavefront for 2B <= 128, AVVAD_BPTT_CHUNKS=1 =
layers back to back instead of the chunked two-stream chains for larger batches, AVVAD_BPTT_GRAPH=0 = no CUDA graphs).
--exact: fail unless every gradient tensor equals the --cmp file's bit for bit.
--state: the stateful forward and backward (avvad_lstm_backward_state) from a nonzero (h0, c0), with nonzero gradients
of the final state and lengths that include 0, 1 and T; dh_in and dc_in are saved with the other gradients.
usage: [AVVAD_BPTT_*=...] python tools/micro/bptt_ab.py [B] [T] [--state] [--save f.pt] [--cmp f.pt [--exact]]"""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (REPO, os.path.join(REPO, "audio-visual-vad_b200")):
    sys.path.insert(0, p)
import torch

from avvad import engine as E
from avvad import synth

args = [a for a in sys.argv[1:] if not a.startswith("--")]
B = int(args[0]) if len(args) > 0 else 256
T = int(args[1]) if len(args) > 1 else 317
val = lambda k: sys.argv[sys.argv.index(k) + 1] if k in sys.argv else None

sd = synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 1, "strong")
lstm = E.Lstm(2, 1024, 1024, 1)
lstm.load(sd, "cuda", "lstm_merged", "vad_merged")
g = torch.Generator().manual_seed(0)
x = lstm.new_input(B, T, "cuda")
x[:, :, :1024] = (torch.randn(B, T, 1024, generator=g) * 0.5).to(torch.bfloat16).cuda()
lens = torch.randint(max(1, T // 2), T + 1, (B,), generator=g).tolist()
lens[0] = T
state = "--state" in sys.argv
if state:
    lens[1 % B], lens[2 % B], lens[3 % B] = 0, 1, T
    shape = (2, B, 1024)
    hx = ((torch.randn(shape, generator=g) * 0.5).to(torch.bfloat16).cuda(), (torch.randn(shape, generator=g) * 0.5).cuda())
    d_state = ((torch.randn(shape, generator=g) * 0.1).cuda(), (torch.randn(shape, generator=g) * 0.1).cuda())
dl = (torch.randn(B, T, 1, generator=g) * 0.1).cuda()
for b, l in enumerate(lens):
    dl[b, l:] = 0


def forward():
    if state:
        return E.lstm_train_forward(lstm, x, lens, state=hx)[1]
    return E.lstm_train_forward(lstm, x, lens)[1]


def backward(tape):
    if state:
        return E.lstm_train_backward(lstm, tape, dl, want_dx=True, d_state=d_state, want_state_grad=True)
    return E.lstm_train_backward(lstm, tape, dl, want_dx=True)


for _ in range(3):
    gr = backward(forward())
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 5
ms = 0.0
for _ in range(n):
    tape = forward()
    e0.record()
    gr = backward(tape)
    e1.record()
    torch.cuda.synchronize()
    ms += e0.elapsed_time(e1) / n
tag = " ".join(f"{k[11:]}={v}" for k, v in sorted(os.environ.items()) if k.startswith("AVVAD_BPTT_")) or "default"
tag += " state" if state else ""
print(f"[{tag}] B={B} T={T}: backward {ms:.3f} ms", flush=True)
flat = {}
for k, v in gr.items():
    if isinstance(v, list):
        for i, t in enumerate(v):
            flat[f"{k}{i}"] = t.cpu()
    elif v is not None:
        flat[k] = v.cpu()
if val("--save"):
    torch.save(flat, val("--save"))
if val("--cmp"):
    ref = torch.load(val("--cmp"))
    assert set(flat) == set(ref), (sorted(flat), sorted(ref))
    worst = max(((flat[k] - ref[k]).norm() / (ref[k].norm() + 1e-30)).item() for k in ref)
    print(f"[{tag}] vs {val('--cmp')}: worst relative gradient difference {worst:.3e} over {len(ref)} tensors", flush=True)
    if "--exact" in sys.argv:
        differ = [k for k in ref if not torch.equal(flat[k], ref[k])]
        assert not differ, f"not bit-identical: {differ}"
        print(f"[{tag}] bit-identical: all {len(ref)} tensors", flush=True)
