"""Every fast path against the plain path it replaced, on the same inputs and weights.

The kernels added in the second half of round 2 (CTA-pair convolutions / GEMMs, the fused layer1 BasicBlock, the CTA-pair
LSTM recurrence, the chunk-interleaved layers, the backward wavefront) are selected by environment variables that libavvad
reads once per process, so each configuration runs in a child process (tools/micro/*.py) and the outputs are compared
here.  The forward variants keep the rounding points and accumulation order of the paths they replace: they must be
BIT-IDENTICAL.  The backward wavefront sums the same products in a different order: gradients agree to bf16 rounding."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(tool, args, env_over, out):
    env = dict(os.environ)
    env.update(env_over)
    cmd = [sys.executable, os.path.join(REPO, "tools", "micro", tool)] + [str(a) for a in args] + ["--save", out]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return torch.load(out)


@pytest.mark.parametrize("n_frames,full", [(37, False), (1201, True)])
def test_trunk_pairs_and_fused_block_bit_identical(tmp_path, n_frames, full):
    """ResNet-18 trunk features: single-CTA engine with two slab convolutions per layer1 block vs CTA pairs + fused block."""
    plain = _run("trunk_ab.py", [n_frames], {"AVVAD_CG2": "0", "AVVAD_BLOCK17": "0"}, str(tmp_path / "plain.pt"))
    fast = _run("trunk_ab.py", [n_frames], {}, str(tmp_path / "fast.pt"))
    assert torch.isfinite(plain).all() and plain.abs().max() > 0
    assert torch.equal(fast, plain)
    if full:
        block_only = _run("trunk_ab.py", [n_frames], {"AVVAD_CG2": "0"}, str(tmp_path / "blk.pt"))
        assert torch.equal(block_only, plain)


@pytest.mark.parametrize("B,T,full", [(256, 80, True), (200, 48, False), (300, 40, False), (64, 80, False)])
def test_lstm_pair_and_chunked_layers_bit_identical(tmp_path, B, T, full):
    """2 x LSTM-1024 + head, ragged lengths: one CTA per block and the layers back to back vs CTA pairs (B > 128) and the
    chunk-interleaved layers; B = 300 spans two batch groups, B = 64 leaves the second CTA of every pair without rows."""
    plain = _run("lstm_ab.py", [B, T], {"AVVAD_LSTM_PAIR": "0", "AVVAD_LSTM_CHUNKS": "1"}, str(tmp_path / "plain.pt"))
    fast = _run("lstm_ab.py", [B, T], {}, str(tmp_path / "fast.pt"))
    assert torch.isfinite(plain).all() and plain.std() > 1e-3
    assert torch.equal(fast, plain)
    if full:
        chunks3 = _run("lstm_ab.py", [B, T], {"AVVAD_LSTM_CHUNKS": "3"}, str(tmp_path / "c3.pt"))
        np64 = _run("lstm_ab.py", [B, T], {"AVVAD_LSTM_NP": "64", "AVVAD_LSTM_EPI_WARPS": "4"}, str(tmp_path / "np64.pt"))
        assert torch.equal(chunks3, plain)
        assert torch.equal(np64, plain)


def test_lstm_training_forward_chunked_bit_identical(tmp_path):
    plain = _run("lstm_ab.py", [160, 64, "--train"], {"AVVAD_LSTM_PAIR": "0", "AVVAD_LSTM_CHUNKS": "1"},
                 str(tmp_path / "plain.pt"))
    fast = _run("lstm_ab.py", [160, 64, "--train"], {}, str(tmp_path / "fast.pt"))
    assert torch.equal(fast, plain)


@pytest.mark.parametrize("B", [24, 64])
def test_bptt_wavefront_matches_layer_by_layer(tmp_path, B):
    """Backward of 2 x LSTM-1024 + head: the two-layer wavefront (one merged cell kernel + one block-structured GEMM per
    iteration) against the layer-by-layer recurrence; every gradient tensor within 5e-3 relative (bf16 operands, another
    summation order)."""
    plain = _run("bptt_ab.py", [B, 60], {"AVVAD_BPTT_WAVEFRONT": "0"}, str(tmp_path / "plain.pt"))
    wave = _run("bptt_ab.py", [B, 60], {"AVVAD_BPTT_WAVEFRONT": "1"}, str(tmp_path / "wave.pt"))
    assert set(plain) == set(wave)
    for k in plain:
        rel = ((wave[k] - plain[k]).norm() / (plain[k].norm() + 1e-30)).item()
        assert rel < 5e-3, (k, rel)


def test_bptt_overlapped_chains_bit_identical(tmp_path):
    """Larger batches: the two layers' backward recurrences as chunked chains on two streams (layer 0 one chunk behind,
    its upstream gradient from one time-major GEMM per chunk) against the layer-by-layer loop: same kernels, same order."""
    plain = _run("bptt_ab.py", [96, 70], {"AVVAD_BPTT_CHUNKS": "1"}, str(tmp_path / "plain.pt"))
    fast = _run("bptt_ab.py", [96, 70], {}, str(tmp_path / "fast.pt"))
    assert set(plain) == set(fast)
    for k in plain:
        assert torch.isfinite(plain[k]).all() and torch.equal(fast[k], plain[k]), k


def test_register_fft_kernels_match_the_shared_memory_fft_kernels():
    """MCB row pass (whole-call and per-utterance norm) and log-power front end: register FFT (default) vs the radix-4
    shared-memory FFT kernels they replaced (AVVAD_MCB_REG=0 / AVVAD_FE_REG=0, also the fallback for degenerate hash
    tables), at the bench shape.  Different butterfly order -> different fp32 rounding: agreement to 1e-5 relative is
    asserted inside the tool (measured 5e-7 / 1e-7), which runs each mode in its own child process."""
    r = subprocess.run([sys.executable, os.path.join(REPO, "tools", "micro", "fft_reg_ab.py")], capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "mcb grouped: register FFT vs shared-memory FFT" in r.stdout
