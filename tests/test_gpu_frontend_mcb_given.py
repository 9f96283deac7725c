"""GPU: the two whole-utterance constants given instead of computed.  The audio front end with caller peaks
(normalise == 2) equals the computed-peak run handed the same peaks, and the grouped MCB with norms_in = the norms_out
of a normal run is bit-identical to that run."""
import pytest
import torch

from avvad import engine as E
from avvad import synth

pytestmark = pytest.mark.gpu


def test_frontend_given_peaks():
    g = torch.Generator().manual_seed(3)
    B, N = 5, 30000
    ns = [30000, 1, 1023, 17000, 4097]
    wave = torch.zeros(B, N)
    for b, n in enumerate(ns):
        wave[b, :n] = torch.randn(n, generator=g) * (0.1 + b)
    wave = wave.cuda()
    nf = [E.stft_num_frames(n) for n in ns]
    t_max = max(nf)
    mean, std = (torch.from_numpy(a) for a in synth.synth_audio_stats(0))
    computed = E.frontend_logpower(wave, ns, nf, t_max, mean, std)
    peaks = torch.stack([wave[b, :n].abs().max() for b, n in enumerate(ns)])
    given = E.frontend_logpower(wave, ns, nf, t_max, mean, std, peaks=peaks)
    assert torch.equal(given, computed)
    # other peaks really are used: twice the peak is the log-power minus log(4)
    half = E.frontend_logpower(wave, ns, nf, t_max, None, None, peaks=2 * peaks)
    full = E.frontend_logpower(wave, ns, nf, t_max, None, None)
    valid = torch.arange(t_max, device="cuda").view(1, -1) < torch.tensor(nf, device="cuda").view(-1, 1)
    assert not torch.equal(half[valid], full[valid])


def test_grouped_mcb_given_norms():
    sd = synth.calibrate_mcb_bn_(synth.seeded_state_dict(synth.model_spec("av", use_mcb=True), 9), 16)
    mcb = E.Mcb()
    mcb.load(sd, "cuda")
    g = torch.Generator().manual_seed(4)
    B, t_max = 6, 37
    lens = [37, 0, 1, 20, 36, 5]
    audio = torch.randn(B, t_max, 513, generator=g).cuda()
    video = torch.randn(B, t_max, 512, generator=g).abs().cuda()
    ref = torch.zeros(B * t_max, 1024, dtype=torch.bfloat16, device="cuda")
    ref32 = torch.zeros(B * t_max, 1024, device="cuda")
    norms = torch.zeros(B, device="cuda")
    mcb.forward_grouped(audio, video, lens, t_max, out_bf16=ref, out_f32=ref32, norms_out=norms)
    plain = torch.zeros_like(ref)
    mcb.forward_grouped(audio, video, lens, t_max, out_bf16=plain)
    assert torch.equal(plain, ref)
    assert bool((norms[torch.tensor(lens, device="cuda") > 0] > 0).all())
    got = torch.zeros_like(ref)
    got32 = torch.zeros_like(ref32)
    back = torch.zeros(B, device="cuda")
    mcb.forward_grouped(audio, video, lens, t_max, out_bf16=got, out_f32=got32, norms_in=norms, norms_out=back)
    assert torch.equal(got, ref) and torch.equal(got32, ref32)
    assert torch.equal(back, norms)
    # a different norm changes the output: the given values are the ones applied
    other = torch.zeros_like(ref32)
    mcb.forward_grouped(audio, video, lens, t_max, out_f32=other, norms_in=2 * norms)
    assert not torch.equal(other[:t_max], ref32[:t_max])
