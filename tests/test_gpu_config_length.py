"""GPU parity at the clip lengths of BASELINE configs 2-5 (fixtures of oracle/make_golden_long.py: outputs of the
UNMODIFIED reference on CPU).  Inputs are regenerated from their seed and checked against the stored fingerprint.
Gates: cRM <= 1e-3 rel and waveform <= 1e-4 abs (inference, both weight sets); loss rel <= 1e-3 and per-tensor gradient
rel-L2 <= 1e-2 (training, T = 188 - the recurrence 12x longer than train_full.npz)."""
import numpy as np
import pytest
import torch

from conftest import WB_GAIN, rel_l2, rel_max

pytestmark = pytest.mark.gpu
CRM_TOL, WAV_TOL = 1e-3, 1e-4
SUB = 97


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def fingerprint(y):
    a = y.numpy().astype(np.float64)
    return np.concatenate([a.reshape(-1)[:8], [a.sum(), np.abs(a).sum()]])


def check_fp(y, fp):
    assert np.allclose(fingerprint(y), fp, rtol=0, atol=1e-9), "regenerated input differs from the one the golden was made from"


@pytest.mark.parametrize("precision,crm_tol", [("fp32", 5e-5), ("auto", 5e-5)])
@pytest.mark.parametrize("tag,gain", [("wa", 1.0), ("wb", WB_GAIN)])
def test_fullsubnet_4s_clip_both_weight_sets(golden, dev, tag, gain, precision, crm_tol):
    from fullsubnet_b200.fullsubnet.model import Model
    from oracle import fullsubnet_oracle as O
    g = golden(f"model_full_4s_{tag}")
    y = O.make_noisy(1, 64000, seed=40, speechlike=True)
    check_fp(y, g["y_fp"])
    m = Model(**O.DEFAULT_MODEL_ARGS, precision=precision)
    m.load_state_dict(O.make_state_dict(seed=0, sb_fc_gain=gain), strict=True)
    m = m.to(dev).eval()
    wav, crm = m.enhance(y.to(dev), return_crm=True)
    e_crm, e_l2 = rel_max(crm.cpu(), g["crm"]), rel_l2(crm.cpu(), g["crm"])
    e_wav = float(np.abs(wav.cpu().numpy() - g["wav"]).max())
    print(f"fullsubnet 4 s {tag} {m._resolve_precision()}: cRM max-rel {e_crm:.2e} rel-l2 {e_l2:.2e}, wav max-abs {e_wav:.2e}")
    assert e_crm < crm_tol and e_l2 < crm_tol and e_wav < WAV_TOL


def test_fullsubnet_4s_single_pass_f16_mask_gate(golden, dev):
    """The opt-in single-pass mode at T = 251: cRM gate on both weight sets, waveform gate on W-a."""
    from fullsubnet_b200.fullsubnet.model import Model
    from oracle import fullsubnet_oracle as O
    y = O.make_noisy(1, 64000, seed=40, speechlike=True).to(dev)
    for tag, gain in (("wa", 1.0), ("wb", WB_GAIN)):
        g = golden(f"model_full_4s_{tag}")
        m = Model(**O.DEFAULT_MODEL_ARGS, precision="f16_tc")
        m.load_state_dict(O.make_state_dict(seed=0, sb_fc_gain=gain), strict=True)
        wav, crm = m.to(dev).eval().enhance(y, return_crm=True)
        assert rel_max(crm.cpu(), g["crm"]) < CRM_TOL and rel_l2(crm.cpu(), g["crm"]) < CRM_TOL
        if tag == "wa":
            assert np.abs(wav.cpu().numpy() - g["wav"]).max() < WAV_TOL


@pytest.mark.parametrize("prec", ["fp32", "tf32_tc"])
def test_training_step_4x3s_matches_reference(golden, dev, prec):
    """Config-3 clip length (T = 188): loss, every gradient tensor (sub-sampled + L2 norm), clip norm, Adam update."""
    from test_gpu_train import GRAD_TOL, LOSS_TOL, build, reference_like_step
    from fullsubnet_b200.loss import mse_loss
    from fullsubnet_b200.optim import FusedClipAdam
    from oracle import fullsubnet_oracle as O
    g = golden("train_full_3s")
    noisy = O.make_noisy(4, 48000, seed=41, speechlike=True)
    clean = 0.5 * O.make_noisy(4, 48000, seed=42, speechlike=True)
    check_fp(noisy, g["noisy_fp"])
    check_fp(clean, g["clean_fp"])
    args = dict(O.DEFAULT_MODEL_ARGS, weight_init=False)
    m = build(args, O.make_state_dict(seed=0, args=args, sb_fc_gain=40.0), dev, prec)
    opt = FusedClipAdam(m.parameters(), lr=1e-3, max_norm=10.0)
    loss, _, _ = reference_like_step(m, noisy.to(dev), clean.to(dev), 512, 256, mse_loss())
    assert abs(float(loss.detach()) - g["loss"][0]) <= LOSS_TOL[prec] * g["loss"][0], (float(loss), g["loss"][0])
    worst = 0.0
    for k, p in m.named_parameters():
        got = p.grad.cpu().numpy().reshape(-1)
        e = rel_l2(got[::SUB], g["gsub." + k])
        n = abs(np.sqrt((got.astype(np.float64) ** 2).sum()) - g["gl2." + k]) / g["gl2." + k]
        worst = max(worst, e, n)
        assert e < GRAD_TOL[prec] and n < GRAD_TOL[prec], (k, e, n)
    print(f"training step 4 x 3 s ({prec}): worst gradient error {worst:.2e}, loss {float(loss):.6f} (ref {g['loss'][0]:.6f})")
    opt.step()
    tol = 1e-4 if prec == "fp32" else 5e-3
    assert abs(float(opt.last_norm[0]) - g["gnorm"][0]) < tol * g["gnorm"][0]
    if prec == "fp32":
        for k, v in m.state_dict().items():
            assert np.abs(v.cpu().numpy().reshape(-1)[::SUB] - g["psub." + k]).max() < 2e-5, k


@pytest.mark.parametrize("precision,tol", [("fp32", 5e-5), ("f16x3_tc", 5e-5), ("f16_tc", CRM_TOL)])
def test_fast_fullsubnet_4s(golden, dev, precision, tol):
    from fullsubnet_b200.acoustics.feature import stft
    from fullsubnet_b200.fast_fullsubnet.model import Model
    from oracle import fast_fullsubnet_oracle as FO
    from oracle import fullsubnet_oracle as O
    g = golden("fast_full_4s")
    y = O.make_noisy(2, 64000, seed=43, speechlike=True)
    check_fp(y, g["y_fp"])
    m = Model(**FO.DEFAULT_FAST_ARGS, precision=precision)
    m.load_state_dict(FO.make_fast_state_dict(seed=3), strict=True)
    m = m.to(dev).eval()
    with torch.no_grad():
        out = m(stft(y.to(dev), 512, 256, 512)[0].unsqueeze(1))
    e, e2 = rel_max(out.cpu(), g["out"]), rel_l2(out.cpu(), g["out"])
    print(f"fast_fullsubnet 2 x 4 s {precision}: max-rel {e:.2e} rel-l2 {e2:.2e}")
    assert out.shape == g["out"].shape and e < tol and e2 < tol


@pytest.mark.parametrize("prec", ["fp32", "tf32_tc"])
@pytest.mark.parametrize("tag", ["k16", "k48", "k48_960"])
def test_improved_fullsubnet_2s(golden, dev, tag, prec):
    from fullsubnet_b200.improved_fullsubnet.model import Model
    from oracle import fullsubnet_oracle as O
    from oracle import improved_fullsubnet_oracle as IO
    g = golden("improved_2s")
    args, L = {"k16": (IO.DEFAULT_IMPROVED_ARGS, 32000), "k48": (IO.ARGS_48K_1024, 96000),
               "k48_960": (IO.ARGS_48K_960, 96000)}[tag]
    y = O.make_noisy(1, L, seed=44, speechlike=True)
    check_fp(y, g[tag + "_y_fp"])
    m = Model(**args)
    m.load_state_dict(IO.make_improved_state_dict(seed=5, args=args), strict=True)
    m.precision = prec
    with torch.no_grad():
        wav = m.to(dev).eval()(y.to(dev))
    err = float(np.abs(wav.cpu().numpy() - g[tag + "_wav"]).max())
    print(f"improved_fullsubnet 2 s {tag} {prec}: waveform max-abs {err:.2e} (scale {np.abs(g[tag + '_wav']).max():.2e})")
    assert wav.shape == g[tag + "_wav"].shape and err < WAV_TOL
