"""CPU: pin the oracle against tests/golden/ref_strong.npz -- outputs of the UNMODIFIED reference modules on
  * the assembled use_mcb=True forward (packages/models/AV_Net.py:111-121) and the stand-alone CompactBilinearPooling
    forward + hand-written backward (compact_bilinear_pooling.py:140-220), executed in the build container through the
    two-function torch.rfft / torch.irfft re-spelling of tools/make_golden.py::install_legacy_fft_shim;
  * the "strong" weight family (avvad.synth.FAMILIES) whose logits span several units;
  * one training step of DeepVAD_AV(use_mcb=True, trunk frozen) and DeepVAD_video(trunk trainable): logits, loss,
    gradient digests and BatchNorm running statistics."""
import numpy as np
import pytest
import torch

from oracle import models as om
from avvad import synth
from util import golden, ref_models, err_stats, grad_digest_of


@pytest.fixture(scope="module")
def gs():
    return golden("ref_strong.npz")


@pytest.fixture(scope="module")
def gref():
    return ref_models()


def _sd(kind, seed, family="strong", **kw):
    return synth.seeded_state_dict(synth.model_spec(kind, **kw), seed, family)


def test_standalone_mcb_forward_and_backward_match_reference(gs):
    sd = {"mcb.sketch1.h": synth.seeded_tensor("mcb.sketch1.h", (513,), torch.int64, 15),
          "mcb.sketch1.s": synth.seeded_tensor("mcb.sketch1.s", (513,), torch.float32, 15),
          "mcb.sketch2.h": synth.seeded_tensor("mcb.sketch2.h", (512,), torch.int64, 15),
          "mcb.sketch2.s": synth.seeded_tensor("mcb.sketch2.s", (512,), torch.float32, 15)}
    x = torch.tensor(gs["cbp_x"], requires_grad=True)
    y = torch.tensor(gs["cbp_y"], requires_grad=True)
    out = om.mcb(x, y, sd)
    assert err_stats(out.detach().numpy(), gs["cbp_out"])["rel_fro"] < 1e-6
    out.backward(torch.tensor(gs["cbp_go"]))
    # the reference's hand-written backward equals autograd of the restated forward
    assert err_stats(x.grad.numpy(), gs["cbp_gx"])["rel_fro"] < 1e-5
    assert err_stats(y.grad.numpy(), gs["cbp_gy"])["rel_fro"] < 1e-5


@pytest.mark.parametrize("family,seed", [("default", 22), ("strong", 42)])
def test_assembled_av_mcb_forward_matches_reference(gs, gref, family, seed):
    sd = synth.calibrate_mcb_bn_(_sd("av", seed, family, use_mcb=True), 12)
    if family == "strong":
        sd["vad_merged.bias"] = torch.tensor(gs["av_mcb_out_strong_bias"])
    a, v, lens = torch.tensor(gref["av_audio"]), torch.tensor(gref["av_video"]), gref["av_len"].tolist()
    out = om.deepvad_av_forward(a, v, lens, sd, use_mcb=True, eps=1e-8).numpy()
    ref = gs[f"av_mcb_out_{family}"]
    assert np.abs(out - ref).max() < 2e-5 * max(1.0, np.abs(ref).max()), np.abs(out - ref).max()


def _strong_sd(gs, kind, seed, key, head, **kw):
    sd = _sd(kind, seed, **kw)
    sd[head + ".bias"] = torch.tensor(gs[key + "_bias"])
    return sd


def _long_av_inputs(gs):
    v = torch.tensor(np.random.default_rng(78).standard_normal((2, 40, 67, 67)).astype(np.float32))
    a = torch.tensor(np.random.default_rng(79).standard_normal((2, 40, 513)).astype(np.float32))
    return a, v, gs["av_long_len"].tolist()


def test_strong_family_forwards_match_reference(gs, gref):
    a, v, lens = _long_av_inputs(gs)
    sd = _strong_sd(gs, "audio", 41, "audio_long_out_strong", "vad_audio")
    out = om.deepvad_audio_forward(torch.tensor(gref["audio_x"]), gref["audio_len"].tolist(), sd).numpy()
    assert err_stats(out, gs["audio_out_strong"])["rel_fro"] < 1e-5
    out = om.deepvad_video_forward(v, lens, _strong_sd(gs, "video", 43, "video_out_strong", "vad_video")).numpy()
    assert err_stats(out, gs["video_out_strong"])["rel_fro"] < 1e-4
    for y_dim, seed, key in ((1, 44, "av_out_strong"), (513, 45, "av513_out_strong")):
        out = om.deepvad_av_forward(a, v, lens, _strong_sd(gs, "av", seed, key, "vad_merged", y_dim=y_dim)).numpy()
        assert err_stats(out, gs[key])["rel_fro"] < 1e-4, key
    # the logits really span several units and both decision classes occur
    ref = gs["audio_long_out_strong"]
    assert ref.std() > 0.3 and (ref > 0).mean() > 0.5 and (ref < 0).any()
    ref = gs["av513_out_strong"]
    assert 0.4 < (ref > 0).mean() < 0.6


def test_strong_family_long_ragged_audio_matches_reference(gs):
    x = torch.tensor(np.random.default_rng(77).standard_normal((4, 317, 513)).astype(np.float32))
    sd = _strong_sd(gs, "audio", 41, "audio_long_out_strong", "vad_audio")
    out = om.deepvad_audio_forward(x, gs["audio_long_len"].tolist(), sd).numpy()
    assert err_stats(out, gs["audio_long_out_strong"])["rel_fro"] < 1e-4


def _check_digest(gs, tag, named_grads, tol):
    worst = {}
    for k, g in named_grads:
        if f"{tag}/{k}/norm" not in gs:
            assert g is None, k
            continue
        norm, sample = grad_digest_of(g)
        rn = float(gs[f"{tag}/{k}/norm"])
        assert abs(norm - rn) <= tol * max(rn, 1e-12), (k, norm, rn)
        rs = gs[f"{tag}/{k}/sample"]
        worst[k] = np.linalg.norm(sample - rs) / (np.linalg.norm(rs) + 1e-30)
        assert worst[k] <= tol, (k, worst[k])
    return worst


def _train_step(forward, sd, trainable, lens, tgt):
    p = {k: (v.clone().requires_grad_(True) if trainable(k) and v.is_floating_point() and "running" not in k else v.clone())
         for k, v in sd.items()}
    logits = forward(p)
    loss = om.batch_loss(logits, tgt, lens, 1e-8)
    loss.backward()
    return logits, loss, p


def test_training_step_av_mcb_frozen_trunk_matches_reference(gs, gref):
    a, v, lens = torch.tensor(gref["av_audio"]), torch.tensor(gref["av_video"]), gref["av_len"].tolist()
    tgt = torch.tensor(gs["train_target"])
    sd = _sd("av", 46, use_mcb=True)
    logits, loss, p = _train_step(lambda q: om.deepvad_av_forward(a, v, lens, q, use_mcb=True, eps=1e-8, training=True),
                                  sd, lambda k: not k.startswith(("features.", "bn.", "mcb.")), lens, tgt)
    assert err_stats(logits.detach().numpy(), gs["train_av_mcb_logits"])["rel_fro"] < 1e-4
    assert abs(loss.item() - float(gs["train_av_mcb_loss"])) < 1e-4 * abs(float(gs["train_av_mcb_loss"]))
    _check_digest(gs, "train_av_mcb", [(k, t.grad) for k, t in p.items() if t.requires_grad], 2e-3)


def test_training_step_video_trainable_trunk_matches_reference(gs, gref):
    v, lens = torch.tensor(gref["av_video"]), gref["av_len"].tolist()
    tgt = torch.tensor(gs["train_target"])
    sd = _sd("video", 47)
    logits, loss, p = _train_step(lambda q: om.deepvad_video_forward(v, lens, q, training=True), sd, lambda k: True,
                                  lens, tgt)
    assert err_stats(logits.detach().numpy(), gs["train_video_logits"])["rel_fro"] < 1e-4
    assert abs(loss.item() - float(gs["train_video_loss"])) < 1e-4 * abs(float(gs["train_video_loss"]))
    _check_digest(gs, "train_video", [(k, t.grad) for k, t in p.items() if t.requires_grad], 5e-3)


def test_one_call_per_utterance_matches_reference_evaluation_pattern():
    """scripts/evaluate_AV_net.py:186-236 calls the model once per utterance (x[None], v[None], lengths = [T]); the golden
    holds the UNMODIFIED reference module's logits for that call pattern.  The oracle called the same way must agree --
    and ONE batched call of the same utterances must NOT (AV_Net.py:117 normalises over the whole padded tensor), which
    is why the batched device path has a per-utterance norm (avvad_mcb_forward_grouped)."""
    from util import eval_single_inputs
    g = golden("ref_eval_single.npz")
    a, v, lens = eval_single_inputs()
    assert lens == g["lens"].tolist()
    sd = synth.calibrate_mcb_bn_(_sd("av", 43, "strong", use_mcb=True), 20)
    sd["vad_merged.bias"] = torch.tensor(g["bias"])
    worst_batched = 0.0
    for b, n in enumerate(lens):
        out = om.deepvad_av_forward(torch.tensor(a[b:b + 1, :n]), torch.tensor(v[b:b + 1, :n]), [n], sd, use_mcb=True,
                                    eps=1e-8).numpy()[0]
        assert err_stats(out, g["logits"][b, :n])["rel_fro"] < 2e-5, b
        worst_batched = max(worst_batched, float(np.abs(g["batched_call_logits"][b, :n] - g["logits"][b, :n]).max()))
    assert worst_batched > 0.5   # the reference itself: a batched call is a different function
    batched = om.deepvad_av_forward(torch.tensor(a), torch.tensor(v), lens, sd, use_mcb=True, eps=1e-8).numpy()
    for b, n in enumerate(lens):
        assert err_stats(batched[b, :n], g["batched_call_logits"][b, :n])["rel_fro"] < 2e-5, b
