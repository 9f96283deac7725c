"""Streaming inference on one GPU: AVVADStream over 256 slots of the benchmark's synthetic utterances
(avvad.synth.batch_inputs, as bench.py), fed so that every step emits `block` new frames per slot, for block = 16, 32
and 64 output frames (256, 512 and 1024 ms).  Reports, device-timed with CUDA events: the per-step() time (median,
p99), output frames per second over all slots, and one offline infer_device(per_utterance=True) call on the same
utterances as the reference point.  Asserts that the streamed posteriors and decisions are bit-identical to the offline
call at every timed block size.  Prints the GPU's name and power limit beside the numbers; fails without a GPU.

    python tools/micro/stream_bench.py [--slots 256] [--blocks 16,32,64] [--reps 2]
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

from avvad import synth  # noqa: E402
from avvad.pipeline import AVVADPipeline  # noqa: E402
from avvad.stream import AVVADStream, source_index  # noqa: E402

N_SAMPLES, N_SRC = 81920, 152   # bench.py's utterance: 5.12 s, 317 frames


def gpu_label():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def stream_once(pipe, wave, vid, peaks, norms, block):
    """Stream every utterance in lock step; returns (post, dec) per slot and the device time of every step (ms)."""
    S = wave.shape[0]
    st = AVVADStream(pipe, S, max_samples=(block + 8) * 256 + 2048, max_frames=block + 8, max_step=block)
    for s in range(S):
        st.open(s, float(peaks[s]), float(norms[s]))
    a = [0] * S
    f = [0] * S
    k = 0
    posts, decs, times = [], [], []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while True:
        want = k + block   # feed exactly what frames k .. k + block - 1 need
        na = min(max((want - 1) * 256 + 1024, 0), N_SAMPLES)
        nf = min(source_index(want - 1) + 1, N_SRC)
        closed = na == N_SAMPLES and nf == N_SRC
        for s in range(S):
            if st.plans[s] is None:
                continue
            if na > a[s] or nf > f[s]:
                st.push(s, wave=wave[s, a[s]:na] if na > a[s] else None, video_u8=vid[s, f[s]:nf] if nf > f[s] else None)
                a[s], f[s] = na, nf
            if closed and not st.plans[s].closed:
                st.close(s)
        ev0.record()
        lg, post, dec, count, frame0 = st.step()
        ev1.record()
        ev1.synchronize()
        if max(count) == 0:
            break
        times.append(ev0.elapsed_time(ev1))
        posts.append(post[:, :max(count)].clone())
        decs.append(dec[:, :max(count)].clone())
        k += max(count)
    return torch.cat(posts, 1), torch.cat(decs, 1), times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=256)
    ap.add_argument("--blocks", default="16,32,64")
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench: no CUDA device")
    name, power = gpu_label()
    S = args.slots
    wave, vid, mean, std = synth.batch_inputs(S, 0, N_SAMPLES, N_SRC)
    sd = synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 1, "strong"), S * 317)
    pipe = AVVADPipeline(sd, mean, std, synth.VIDEO_MEAN, synth.VIDEO_STD, use_mcb=True)
    wave, vid = wave.cuda(), vid.cuda()
    ns, nf = [N_SAMPLES] * S, [N_SRC] * S
    T = AVVADPipeline.frame_counts(ns, nf)[0]
    norms = torch.zeros(S, device="cuda")
    peaks = wave.abs().amax(1).tolist()

    # offline reference point: one call on the whole utterances
    off = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(args.reps + 1):
        ev0.record()
        _, post_ref, dec_ref = pipe.infer_device(wave, ns, vid, nf, per_utterance=True, mcb_norms_out=norms)
        ev1.record()
        ev1.synchronize()
        if r:
            off.append(ev0.elapsed_time(ev1))
    post_ref, dec_ref = post_ref.clone(), dec_ref.clone()
    norms = norms.tolist()
    off_ms = float(np.median(off))
    print(json.dumps({"gpu": name, "power_limit": power, "slots": S, "frames_per_utterance": T,
                      "offline_ms": round(off_ms, 3), "offline_frames_per_s": round(S * T / off_ms * 1e3)}))
    for block in [int(b) for b in args.blocks.split(",")]:
        all_times = []
        for r in range(args.reps + 1):
            post, dec, times = stream_once(pipe, wave, vid, peaks, norms, block)
            assert post.shape[1] == T, (post.shape, T)
            assert torch.equal(post, post_ref[:, :T]) and torch.equal(dec, dec_ref[:, :T]), \
                f"block {block}: streamed posteriors differ from the offline call"
            if r:   # the first pass warms every step shape up
                all_times += times
        t = np.asarray(all_times)
        total_ms = t.sum() / args.reps
        print(json.dumps({"gpu": name, "power_limit": power, "block_frames": block, "steps": len(all_times) // args.reps,
                          "step_ms_median": round(float(np.median(t)), 3),
                          "step_ms_p99": round(float(np.percentile(t, 99)), 3),
                          "frames_per_s": round(S * T / total_ms * 1e3), "bit_identical": True}))


if __name__ == "__main__":
    main()
