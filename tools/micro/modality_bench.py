"""Audio-only and video-only inference on one GPU at the benchmark shape, B = 256 utterances x T = 317 frames of
bench.py's synthetic inputs (avvad.synth.batch_inputs), "strong" weights of DeepVAD_audio / DeepVAD_video.

Reports, device-timed with CUDA events (median over --reps timed calls after one warm-up call):
- AVVADPipeline.infer_device(modality="audio" / "video"): ms and output frames/s; for video also with dedup_video on;
- audio: the front end as two kernels (fp32 frontend_logpower + pack_rows_bf16) against the bf16 output mode;
- AVVADStream.step() on 256 slots at 16 / 32 / 64 frames per step: median and p99 per step, frames/s over all slots.
Asserts bit-identity where the paths compute the same thing: dedup against no dedup, two-kernel against fused front end,
every streamed pass against the offline call.  Prints the GPU's name and power limit beside the numbers; fails without
a GPU.

    python tools/micro/modality_bench.py [--modalities audio,video] [--blocks 16,32,64] [--reps 5] [--out FILE]
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


def timed(fn, reps):
    """Median device time (ms) of fn() over `reps` calls after one warm-up call; returns (ms, last result)."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts, out = [], None
    for r in range(reps + 1):
        ev0.record()
        out = fn()
        ev1.record()
        ev1.synchronize()
        if r:
            ts.append(ev0.elapsed_time(ev1))
    return float(np.median(ts)), out


def stream_once(pipe, wave, vid, peaks, block):
    """Stream every utterance in lock step, `block` new frames per step; returns (post, dec) and per-step ms."""
    S = (wave if wave is not None else vid).shape[0]
    st = AVVADStream(pipe, S, max_samples=(block + 8) * 256 + 2048, max_frames=block + 8, max_step=block)
    for s in range(S):
        st.open(s, float(peaks[s]) if wave is not None else None)
    a, f = [0] * S, [0] * S
    k = 0
    posts, decs, times = [], [], []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while True:
        want = k + block   # feed exactly what frames k .. k + block - 1 need
        na = min(max((want - 1) * 256 + 1024, 0), N_SAMPLES) if wave is not None else 0
        nf = min(source_index(want - 1) + 1, N_SRC) if vid is not None else 0
        closed = (wave is None or na == N_SAMPLES) and (vid is None or nf == N_SRC)
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
    ap.add_argument("--modalities", default="audio,video")
    ap.add_argument("--blocks", default="16,32,64")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--stream-reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("modality_bench: no CUDA device")
    name, power = gpu_label()
    B = args.slots
    wave, vid, mean, std = synth.batch_inputs(B, 0, N_SAMPLES, N_SRC)
    wave, vid = wave.cuda(), vid.cuda()
    ns, nf = [N_SAMPLES] * B, [N_SRC] * B
    peaks = wave.abs().amax(1).tolist()
    out = open(args.out, "a") if args.out else None

    def emit(d):
        line = json.dumps({"gpu": name, "power_limit": power, **d})
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    for modality in args.modalities.split(","):
        sd = synth.seeded_state_dict(synth.model_spec(modality), 1, "strong")
        if modality == "audio":
            pipe = AVVADPipeline(sd, mean, std, modality="audio")
            w, v = wave, None
            T = pipe.lengths_of(ns, None)[0]
        else:
            pipe = AVVADPipeline(sd, video_mean=synth.VIDEO_MEAN, video_std=synth.VIDEO_STD, modality="video")
            w, v = None, vid
            T = pipe.lengths_of(None, nf)[0]
        call = (lambda: pipe.infer_device(w, ns if w is not None else None, v, nf if v is not None else None))
        ms, (_, post_ref, dec_ref) = timed(call, args.reps)
        post_ref, dec_ref = post_ref.clone(), dec_ref.clone()
        emit({"modality": modality, "what": "infer_device", "B": B, "T": T, "ms": round(ms, 3),
              "frames_per_s": round(B * T / ms * 1e3)})
        if modality == "video":
            pipe.dedup_video = True
            ms, (_, post_d, dec_d) = timed(call, args.reps)
            assert torch.equal(post_d, post_ref) and torch.equal(dec_d, dec_ref), "dedup_video changed the posteriors"
            emit({"modality": modality, "what": "infer_device dedup_video", "B": B, "T": T, "ms": round(ms, 3),
                  "frames_per_s": round(B * T / ms * 1e3), "bit_identical": True})
            pipe.dedup_video = False
        else:
            m_d, s_d = torch.tensor(mean).cuda(), torch.tensor(std).cuda()
            lens = [T] * B
            f32 = torch.empty(B, T, 513, device="cuda")
            x2 = torch.zeros(B * T, pipe.lstm.ld, dtype=torch.bfloat16, device="cuda")
            x1 = torch.zeros_like(x2)

            def two_kernels():
                E.frontend_logpower(wave, ns, lens, T, m_d, s_d, 1e-8, True, out=f32)
                E.pack_rows_bf16(f32.view(B * T, 513), x2, 0, True)

            def fused():
                E.frontend_logpower(wave, ns, lens, T, m_d, s_d, 1e-8, True, out_bf16=x1)

            ms2, _ = timed(two_kernels, args.reps * 4)
            ms1, _ = timed(fused, args.reps * 4)
            assert torch.equal(x1.view(torch.int16), x2.view(torch.int16)), "bf16 front end differs from fp32 + pack"
            emit({"modality": modality, "what": "front end", "B": B, "T": T, "fp32_plus_pack_ms": round(ms2, 4),
                  "bf16_fused_ms": round(ms1, 4), "bit_identical": True})
        for block in [int(b) for b in args.blocks.split(",")]:
            all_times = []
            for r in range(args.stream_reps + 1):
                post, dec, times = stream_once(pipe, w, v, peaks, block)
                assert post.shape[1] == T, (post.shape, T)
                assert torch.equal(post, post_ref[:, :T]) and torch.equal(dec, dec_ref[:, :T]), \
                    f"{modality} block {block}: streamed posteriors differ from the offline call"
                if r:   # the first pass warms every step shape up
                    all_times += times
            t = np.asarray(all_times)
            total_ms = t.sum() / args.stream_reps
            emit({"modality": modality, "what": "stream", "slots": B, "block_frames": block,
                  "steps": len(all_times) // args.stream_reps, "step_ms_median": round(float(np.median(t)), 3),
                  "step_ms_p99": round(float(np.percentile(t, 99)), 3), "frames_per_s": round(B * T / total_ms * 1e3),
                  "bit_identical": True})
        del pipe
    if out:
        out.close()


if __name__ == "__main__":
    main()
