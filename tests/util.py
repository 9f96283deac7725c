"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def ref_models():
    """tests/golden/ref_models.npz as a dict.  The AV cases ran on the video-only input, so av_video (== video_x) is
    stored once."""
    g = dict(golden("ref_models.npz"))
    g["av_video"] = g["video_x"]
    return g


def err_stats(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    d = np.abs(a - b)
    return {"max": float(d.max()), "mean": float(d.mean()), "p99": float(np.quantile(d, 0.99)),
            "ref_absmax": float(np.abs(b).max()), "rel_fro": float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))}


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(torch.float32)


def lstm_test_weights(layers, input_size, hidden, seed):
    """PyTorch-layout LSTM weights [(w_ih, w_hh, b_ih, b_hh)] for the state tests: U(+-2/sqrt(H)) in layer 0, as the
    "strong" family uses, and U(+-4/sqrt(H)) above, where the input is an h sequence of std ~0.15 instead of ~0.5.  Both
    keep the pre-activation std of every layer within [0.3, 3] for inputs N(0, 0.5^2), so the gates are neither flat nor
    saturated (tests/test_lstm_step_oracle.py asserts it)."""
    g = torch.Generator().manual_seed(seed)
    ws = []
    for l in range(layers):
        k = (2.0 if l == 0 else 4.0) / hidden ** 0.5
        il = input_size if l == 0 else hidden
        shapes = ((4 * hidden, il), (4 * hidden, hidden), (4 * hidden,), (4 * hidden,))
        ws.append(tuple((torch.rand(s, generator=g) * 2 - 1) * k for s in shapes))
    return ws


def grad_digest_of(g) -> tuple:
    """(Frobenius norm, strided sample of <= 2048 elements) -- the digest tools/make_golden.py::grad_digest stores for
    the reference modules' gradients."""
    g = g.detach().reshape(-1).cpu()
    step = max(1, g.numel() // 2048)
    return float(g.double().norm().item()), g[::step][:2048].float().numpy()


POST_TOL = 1e-2      # |posterior - reference| (BASELINE.json north_star: bf16 vs the reference's fp32)
LOGIT_REL = 2e-2     # relative Frobenius error of the logits
AGREE = 0.999        # identical decisions, fraction of ALL valid frames (north_star)


def sigmoid(x):
    return 1.0 / (1.0 + np.exp(-np.asarray(x, dtype=np.float64)))


def check_logits(got, ref, lens=None, what=""):
    """The three parity gates on the valid frames of a (B,T,Y) logit tensor: relative Frobenius error of the logits,
    max |posterior difference|, fraction of identical decisions over ALL valid frames (no exclusion band)."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    if lens is not None:
        mask = np.zeros(ref.shape[:2], dtype=bool)
        for b, n in enumerate(lens):
            mask[b, : int(n)] = True
        got, ref = got[mask], ref[mask]
    rel = np.linalg.norm(got - ref) / np.linalg.norm(ref)
    post = np.abs(sigmoid(got) - sigmoid(ref)).max()
    agree = ((got > 0) == (ref > 0)).mean()
    print(f"{what}: logits rel_fro {rel:.2e}  max|dpost| {post:.2e}  decisions agree {agree:.5f}  "
          f"ref range [{ref.min():.2f}, {ref.max():.2f}] std {ref.std():.2f}  n={ref.size}")
    assert ref.std() > 0.15, "reference logits carry no signal"
    assert rel <= LOGIT_REL, (what, rel)
    assert post <= POST_TOL, (what, post)
    assert agree >= AGREE, (what, agree)
    return rel, post, agree


EVAL_SINGLE_LENS = [23, 9, 16, 31]


def eval_single_inputs():
    """Inputs of tests/golden/ref_eval_single.npz (tools/make_golden.py::eval_single_inputs, same PCG64 streams)."""
    B, T = len(EVAL_SINGLE_LENS), max(EVAL_SINGLE_LENS)
    a = np.random.default_rng(91).standard_normal((B, T, 513)).astype(np.float32)
    v = np.random.default_rng(92).standard_normal((B, T, 67, 67)).astype(np.float32)
    return a, v, list(EVAL_SINGLE_LENS)
