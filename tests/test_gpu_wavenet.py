"""GPU parity: WaveNet encoder (dead code in the reference but named by north_star) vs the reference's own output."""
import numpy as np
import pytest
import torch

from avvad import synth
from oracle import models as om
from util import golden, err_stats

pytestmark = pytest.mark.gpu


def test_wavenet_encoder_matches_reference_golden():
    from packages.models.wavenet_autoencoder import wavenet_autoencoder
    g = golden("ref_models.npz")
    wn = wavenet_autoencoder(filter_width=2, quantization_channel=16, dilations=[1, 2, 4, 8, 1, 2, 4, 8],
                             en_residual_channel=32, en_dilation_channel=32, en_bottleneck_width=16,
                             en_pool_kernel_size=10, use_bias=True)
    synth.fill_module_(wn, seed=16)
    wn = wn.cuda().eval()
    out = wn(torch.tensor(g["wavenet_x"]).cuda()).cpu().numpy()
    st = err_stats(out, g["wavenet_out"])
    assert out.shape == g["wavenet_out"].shape
    assert st["rel_fro"] < 2e-2 and st["max"] < 3e-2 * max(1.0, st["ref_absmax"]), st


def test_wavenet_wider_config_vs_oracle():
    from packages.models.wavenet_autoencoder import wavenet_autoencoder
    dil = [1, 2, 4, 8, 16, 32]
    wn = wavenet_autoencoder(3, 64, dil, 128, 64, 48, 7, use_bias=False)
    synth.fill_module_(wn, seed=5)
    x = torch.randn(3, 64, 700, generator=torch.Generator().manual_seed(1))
    sd = {k: v for k, v in wn.state_dict().items()}
    ref = om.wavenet_encode(x, sd, dil, 7).numpy()
    out = wn.cuda().eval()(x.cuda()).cpu().numpy()
    st = err_stats(out, ref)
    assert st["rel_fro"] < 2e-2, st


@pytest.mark.parametrize("k,dil,N,B", [(2, [1, 2, 4, 8, 1, 2, 4, 8], 3000, 3), (3, [1, 2, 4, 8, 16], 1500, 2),
                                       (2, [1, 2, 4, 8, 16, 32, 64], 900, 1), (1, [1, 1], 300, 2)])
def test_fused_stack_many_time_tiles_vs_oracle(k, dil, N, B):
    """The fused kernel (csrc/wavenet_fused.cuh: whole stack in one launch, receptive-field history in shared memory)
    over inputs much longer than one time tile (225 outputs for the 8-layer k=2 stack): tile seams, the ragged last
    tile, k = 1..3, shifts up to 64 -- against the fp32 oracle."""
    from packages.models.wavenet_autoencoder import wavenet_autoencoder
    wn = wavenet_autoencoder(k, 16, dil, 32, 48, 16, 9, use_bias=True)
    synth.fill_module_(wn, seed=7)
    x = torch.randn(B, 16, N, generator=torch.Generator().manual_seed(2))
    ref = om.wavenet_encode(x, dict(wn.state_dict()), dil, 9).numpy()
    out = wn.cuda().eval()(x.cuda()).cpu().numpy()
    st = err_stats(out, ref)
    assert out.shape == ref.shape and st["rel_fro"] < 2e-2 and st["max"] < 3e-2 * max(1.0, st["ref_absmax"]), st


def test_fused_and_per_layer_paths_agree(tmp_path):
    """AVVAD_WAVENET_FUSED=0 selects the per-layer path (im2col copy + one GEMM per layer); both must give the
    reference's answer (run in a subprocess because the switch is read once per process)."""
    import os
    import subprocess
    import sys
    code = (
        "import sys; sys.path[:0] = [%r, %r]\n"
        "import torch, numpy as np\n"
        "from avvad import synth\n"
        "from packages.models.wavenet_autoencoder import wavenet_autoencoder\n"
        "wn = wavenet_autoencoder(2, 16, [1, 2, 4, 8, 1, 2, 4, 8], 32, 32, 16, 10, use_bias=True)\n"
        "synth.fill_module_(wn, seed=16)\n"
        "x = torch.randn(2, 16, 1000, generator=torch.Generator().manual_seed(3))\n"
        "np.save(sys.argv[1], wn.cuda().eval()(x.cuda()).cpu().numpy())\n"
    ) % (os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "audio-visual-vad_b200"),
         os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    outs = []
    for flag in ("1", "0"):
        path = str(tmp_path / f"wn_{flag}.npy")
        env = dict(os.environ, AVVAD_WAVENET_FUSED=flag)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env)
        outs.append(np.load(path))
    st = err_stats(outs[0], outs[1])
    assert st["rel_fro"] < 1e-2, st
