#!/usr/bin/env python
"""WaveNet encoder training on the device (csrc/wavenet_bwd.cuh) at wavenet_ab.py's shape: B = 64 x N = 16,000, k = 2,
q = 16, dilations [1,2,4,8] x 2, R = D = bottleneck = 64, pool 50.  Device times (CUDA events, warm-up excluded) of the
no_grad encode, the training forward with its tape, the backward, and forward + backward + torch.optim.Adam step; the
same step through PyTorch autograd of oracle.models.wavenet_encode in fp32 on the same GPU as the reference point; tape
bytes; TFLOP/s against the algorithmic work (the forward's MACs x 3); the kernels that take the backward's time
(torch.profiler, after the timed windows).  The GPU's name and power limit are read in the same run.
usage: python tools/micro/wavenet_train_bench.py [--iters 10]"""
import argparse
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (REPO, os.path.join(REPO, "audio-visual-vad_b200")):
    sys.path.insert(0, p)
import torch

from avvad import lib as L
from avvad import synth
from oracle import models as om
from packages.models.wavenet_autoencoder import wavenet_autoencoder

B, N, K, Q = 64, 16000, 2, 16
DIL = [1, 2, 4, 8, 1, 2, 4, 8]
R = D = BOTT = 64
POOL = 50


def forward_macs():
    Ls = [N - (K - 1)]
    for d in DIL:
        Ls.append(Ls[-1] - (K - 1) * d)
    m = B * Ls[0] * R * Q * K
    for i in range(len(DIL)):
        m += B * Ls[i + 1] * (D * R * K + R * D)
    return m + B * Ls[-1] * BOTT * R


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wavenet_train_bench needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    wn = synth.fill_module_(wavenet_autoencoder(K, Q, DIL, R, D, BOTT, POOL, use_bias=True), seed=1).cuda()
    x = torch.randn(B, Q, N, device="cuda")
    target = torch.randn(B, BOTT, POOL, device="cuda") * 0.1
    dout = torch.randn(B, BOTT, POOL, device="cuda")
    eng = wn._build(x.device)
    res = {"gpu": gpu[0] if gpu else "?", "shape": dict(B=B, N=N, k=K, q=Q, dilations=DIL, R=R, D=D, bottleneck=BOTT,
                                                        pool=POOL),
           "tape_bytes": int(L.lib().avvad_wavenet_tape_bytes(eng.h, B, N)),
           "backward_workspace_bytes": int(L.lib().avvad_wavenet_backward_workspace_bytes(eng.h, B, N))}

    with torch.no_grad():
        res["encode_no_grad_ms"] = timed(lambda: wn(x), args.iters)
    res["forward_train_ms"] = timed(lambda: eng.forward_train(x), args.iters)
    _, tape = eng.forward_train(x)
    res["backward_ms"] = timed(lambda: eng.backward(tape, dout), args.iters)
    del tape

    opt = torch.optim.Adam(wn.parameters(), lr=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        torch.nn.functional.mse_loss(wn(x), target).backward()
        opt.step()
    res["step_ms"] = timed(step, args.iters)

    # reference point: PyTorch autograd of the oracle (cuDNN convolutions), fp32 parameters, same optimiser
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in wn.state_dict().items()}
    ropt = torch.optim.Adam(list(sd.values()), lr=1e-4)

    def ref_step():
        ropt.zero_grad(set_to_none=True)
        torch.nn.functional.mse_loss(om.wavenet_encode(x, sd, DIL, POOL), target).backward()
        ropt.step()
    for tf32 in (True, False):
        torch.backends.cudnn.allow_tf32 = tf32
        res[f"torch_step_ms_cudnn_tf32_{int(tf32)}"] = timed(ref_step, args.iters)
    torch.backends.cudnn.allow_tf32 = True
    res["torch_matmul_allow_tf32"] = torch.backends.cuda.matmul.allow_tf32

    flops = 2.0 * forward_macs()
    res["forward_macs"] = forward_macs()
    res["encode_tflops"] = flops / res["encode_no_grad_ms"] / 1e9
    res["fwd_bwd_tflops"] = 3 * flops / (res["forward_train_ms"] + res["backward_ms"]) / 1e9
    res["step_tflops"] = 3 * flops / res["step_ms"] / 1e9

    # where the backward's time goes (a separate, profiled pass after the timed windows)
    _, tape = eng.forward_train(x)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            eng.backward(tape, dout)
        torch.cuda.synchronize()
    by_name = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            by_name[ev.key[:70]] = round(t / 3 / 1000, 4)   # ms per backward
    res["backward_kernels_ms"] = dict(sorted(by_name.items(), key=lambda kv: -kv[1])[:14])
    for k, v in res.items():
        print(f"{k}: {v}")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
