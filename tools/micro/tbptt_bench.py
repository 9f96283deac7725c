"""LSTM training forward + backward with a carried state: what the state costs, and what truncated BPTT in blocks costs.

2 x LSTM-1024 (input 1024, as after MCB) + y_dim = 1 head, T = 317, per batch size B:
  (a) stateless:               lstm_train_forward + lstm_train_backward
  (b) stateful, zero state:    the same with state=(None, None), d_state=None (no state gradients)
  (c) 4 chained blocks:        the same frames as four blocks of ~79 frames, forward block by block with the state
                               carried, then backward from the last block to the first with the state gradients carried
Device time of one whole forward + backward with CUDA events, median and min of --reps after --warmup; prints the GPU's
name and power limit beside the numbers.  Fails without a GPU.

    python tools/micro/tbptt_bench.py [--batches 32,256] [--reps 12] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [REPO, os.path.join(REPO, "audio-visual-vad_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from avvad import engine as E  # noqa: E402

T, H, I, LAYERS, BLOCKS = 317, 1024, 1024, 2, 4


def gpu_label():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def make(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    k = 1.0 / H ** 0.5
    sd = {}
    for l in range(LAYERS):
        il = I if l == 0 else H
        for name, shape in (("weight_ih", (4 * H, il)), ("weight_hh", (4 * H, H)), ("bias_ih", (4 * H,)),
                            ("bias_hh", (4 * H,))):
            sd[f"lstm.{name}_l{l}"] = ((torch.rand(shape, generator=g) * 2 - 1) * k).cuda()
    sd["head.weight"] = ((torch.rand(1, H, generator=g) * 2 - 1) * k).cuda()
    sd["head.bias"] = torch.zeros(1).cuda()
    lstm = E.Lstm(LAYERS, I, H, 1)
    lstm.load(sd, "cuda", "lstm", "head")
    x = lstm.new_input(B, T, "cuda")
    x[..., :I] = (0.5 * torch.randn(B, T, I, generator=g)).to(torch.bfloat16).cuda()
    lens = torch.randint(T // 2, T + 1, (B,), generator=g)
    lens[0] = T
    dl = torch.randn(B, T, 1, generator=g).cuda()
    return lstm, x, lens.cuda(), dl


def run_stateless(lstm, x, lens, dl):
    _, pack = E.lstm_train_forward(lstm, x, lens)
    return E.lstm_train_backward(lstm, pack, dl)


def run_zero_state(lstm, x, lens, dl):
    _, pack, _ = E.lstm_train_forward(lstm, x, lens, state=(None, None))
    return E.lstm_train_backward(lstm, pack, dl)


def block_inputs(x, lens, dl):
    edges = [T * k // BLOCKS for k in range(BLOCKS + 1)]
    return [(x[:, s:e].contiguous(), (lens - s).clamp(0, e - s), dl[:, s:e].contiguous())
            for s, e in zip(edges[:-1], edges[1:])]


def run_blocks(lstm, blocks):
    state, packs = (None, None), []
    for xb, lb, _ in blocks:
        _, pack, state = E.lstm_train_forward(lstm, xb, lb, state=state)
        packs.append(pack)
    d, grads = None, None
    for k in reversed(range(len(blocks))):
        g = E.lstm_train_backward(lstm, packs[k], blocks[k][2], d_state=d, want_state_grad=k > 0)
        if k > 0:
            d = (g["dh_in"], g["dc_in"])
        grads = g
    return grads


def time_it(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(np.min(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="32,256")
    ap.add_argument("--reps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tbptt_bench needs a GPU"
    name, pl = gpu_label()
    print(f"GPU: {name}, power limit {pl}")
    out = {"gpu": name, "power_limit": pl, "T": T, "H": H, "layers": LAYERS, "blocks": BLOCKS, "rows": []}
    for B in [int(v) for v in args.batches.split(",")]:
        lstm, x, lens, dl = make(B)
        blocks = block_inputs(x, lens, dl)
        row = {"B": B}
        # (a) and (b) alternate, (c) after them; each warmed up on its own shapes
        for key, fn in (("stateless", lambda: run_stateless(lstm, x, lens, dl)),
                        ("zero_state", lambda: run_zero_state(lstm, x, lens, dl)),
                        ("stateless_again", lambda: run_stateless(lstm, x, lens, dl)),
                        ("blocks4", lambda: run_blocks(lstm, blocks))):
            med, mn = time_it(fn, args.reps, args.warmup)
            row[key] = {"median_ms": round(med, 3), "min_ms": round(mn, 3)}
            print(f"B={B:4d} {key:16s} median {med:8.3f} ms  min {mn:8.3f} ms")
        out["rows"].append(row)
        del lstm, x, blocks
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
