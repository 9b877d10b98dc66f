"""CPU: the oracle restatement vs. fixtures produced by the unmodified reference
(oracle/make_golden.py).  This is what pins the oracle."""
import numpy as np
import pytest
import torch

from oracle import fullsubnet_oracle as O
from conftest import rel_max, rel_l2, WB_GAIN

T = torch.from_numpy


def test_stft_matches_reference(golden):
    g = golden("dsp")
    mag, phase, real, imag = O.stft(T(g["y"]), 512, 256, 512)
    assert mag.shape == g["mag"].shape
    assert rel_max(real, g["real"]) < 2e-6 and rel_max(imag, g["imag"]) < 2e-6
    assert rel_max(mag, g["mag"]) < 2e-6
    # phase only where the magnitude is not tiny
    sel = g["mag"] > 1e-2 * g["mag"].max()
    d = np.angle(np.exp(1j * (phase.numpy() - g["phase"])))
    assert np.abs(d[sel]).max() < 1e-4
    mag3 = O.stft(T(g["y3"]), 512, 256, 512)[0]
    assert mag3.shape == g["mag3"].shape and rel_max(mag3, g["mag3"]) < 2e-6
    ms, _, rs, is_ = O.stft(T(g["y"]), 64, 32, 64)
    assert rel_max(rs, g["real_s"]) < 2e-6 and rel_max(is_, g["imag_s"]) < 2e-6


def test_istft_matches_reference(golden):
    g = golden("dsp")
    w = O.istft((T(g["real"]), T(g["imag"])), 512, 256, 512, length=g["y"].shape[-1], input_type="real_imag")
    assert rel_max(w, g["wav_rt"]) < 5e-6
    assert rel_max(w, g["y"]) < 5e-6  # round trip
    w2 = O.istft(torch.complex(T(g["real"]), T(g["imag"])), 512, 256, 512)
    assert w2.shape == g["wav_nolen"].shape and rel_max(w2, g["wav_nolen"]) < 5e-6
    w3 = O.istft((T(g["real_s"]), T(g["imag_s"])), 64, 32, 64, length=g["y"].shape[-1], input_type="real_imag")
    assert rel_max(w3, g["wav_s"]) < 5e-6
    with pytest.raises(NotImplementedError):
        O.istft((T(g["real"]), T(g["imag"])), 512, 256, 512, input_type="bogus")


def test_masks_match_reference(golden):
    g = golden("dsp")
    assert rel_max(O.decompress_cIRM(T(g["m"])), g["dec"]) < 1e-6
    assert rel_max(O.compress_cIRM(T(g["big"])), g["comp"]) < 1e-6
    _, _, cr, ci = O.stft(T(g["yc"]), 512, 256, 512)
    cirm = O.build_complex_ideal_ratio_mask(T(g["real"]), T(g["imag"]), cr, ci)
    assert cirm.shape == g["cirm"].shape
    assert np.abs(cirm.numpy() - g["cirm"]).max() < 2e-3  # cIRM is ill-conditioned where |noisy|~0


def test_drop_band_matches_reference(golden):
    g = golden("dsp")
    assert np.array_equal(O.drop_band(T(g["xb"]), 2).numpy(), g["db2"])
    assert np.array_equal(O.drop_band(T(g["xb"]), 3).numpy(), g["db3"])
    sb, sf = O.drop_band_index_map(5, 9, 2)
    x = g["xb"]
    rebuilt = np.stack([x[b][:, f, :] for b, f in zip(sb, sf)])
    assert np.array_equal(rebuilt, g["db2"])
    with pytest.raises(AssertionError):
        O.drop_band(T(g["xb"][:2]), 2)


def _small_args():
    return dict(num_freqs=33, look_ahead=2, sequence_model="LSTM", fb_num_neighbors=0, sb_num_neighbors=3,
                fb_output_activate_function="ReLU", sb_output_activate_function=False,
                fb_model_hidden_size=32, sb_model_hidden_size=24, norm_type="offline_laplace_norm",
                num_groups_in_drop_band=2, weight_init=False)


def test_small_model_matches_reference(golden):
    g = golden("model_small")
    sd = {k[3:]: T(g[k]) for k in g.files if k.startswith("sd.")}
    a = _small_args()
    regen = O.make_state_dict(seed=7, args=a)
    for k in sd:
        assert torch.equal(sd[k], regen[k]), k  # weight generator is version-stable
    mag = T(g["mag"]).unsqueeze(1)
    assert rel_max(O.model_forward(mag[:1], sd, a), g["crm_b1"]) < 1e-5
    assert rel_max(O.model_forward(mag, sd, a), g["crm_g2"]) < 1e-5
    a1 = dict(a, num_groups_in_drop_band=1)
    out, mid = O.model_forward(mag, sd, a1, return_intermediates=True)
    assert rel_max(out, g["crm_g1"]) < 1e-5
    assert rel_max(mid["fb_output"][:, 0], g["fb_out"]) < 1e-5


def test_full_model_and_inferencer_match_reference(golden):
    g = golden("model_full")
    y = T(g["y"])
    for tag, gain in (("wa", 1.0), ("wb", WB_GAIN)):
        sd = O.make_state_dict(seed=0, sb_fc_gain=gain)
        wav, crm = O.enhance(y, sd, batched=True, return_crm=True)
        assert rel_max(crm, g[f"{tag}_crm"]) < 2e-5, tag
        assert np.abs(wav.numpy() - g[f"{tag}_wav"]).max() < 2e-5 * max(1.0, np.abs(g[f"{tag}_wav"]).max()), tag
        wav1 = O.enhance(y, sd, batched=False)
        assert np.abs(wav1.numpy() - g[f"{tag}_wav"]).max() < 2e-5 * max(1.0, np.abs(g[f"{tag}_wav"]).max())
    assert np.abs(g["wb_crm"]).max() > 9.9  # the wb set exercises the clip of decompress_cIRM


def test_reflect_count_closed_form():
    c = O.reflect_count(257, 15)
    assert c.sum() == 257 * 31 and c[0] == 16 and c[256] == 16
    assert (c[1:16] == 32).all() and (c[241:256] == 32).all() and (c[16:241] == 31).all()
    # closed form of the 2nd laplace norm mean (SURVEY 8a row A6)
    mag = torch.rand(2, 1, 257, 9)
    fb = torch.rand(2, 1, 257, 9)
    cat = torch.cat([O.freq_unfold(mag, 15).reshape(2, 257, 31, 9), O.freq_unfold(fb, 0).reshape(2, 257, 1, 9)], 2)
    mu = cat.mean(dim=(1, 2, 3))
    closed = ((mag[:, 0].sum(-1) * torch.from_numpy(c).float()).sum(-1) + fb.sum(dim=(1, 2, 3))) / (257 * 32 * 9)
    assert rel_max(closed, mu) < 1e-5


def test_fast_fullsubnet_oracle_matches_reference(golden):
    from oracle import fast_fullsubnet_oracle as FO
    g = golden("fast_full")
    assert rel_max(FO.melscale_fbanks(257, 64), g["mel_fb"]) < 1e-6  # torchaudio MelScale buffer
    sd = FO.make_fast_state_dict(seed=3)
    mag = T(g["mag"]).unsqueeze(1)
    assert rel_max(FO.fast_model_forward(mag[:1], sd), g["out_b1"]) < 2e-5
    out, mid = FO.fast_model_forward(mag, sd, return_intermediates=True)
    assert out.shape == g["out_b3"].shape and rel_max(out, g["out_b3"]) < 2e-5
    # down/up-sampling restatement on odd and even lengths
    for Tn in (2, 3, 8, 9):
        x = torch.arange(Tn, dtype=torch.float32).reshape(1, 1, 1, Tn)
        d = FO.real_time_downsampling(x, 2)
        assert d.shape[-1] == 1 + (Tn - 1 + 1) // 2
        assert FO.real_time_upsampling(d, 2, Tn).shape[-1] == Tn


def test_improved_fullsubnet_oracle_matches_reference(golden):
    from oracle import improved_fullsubnet_oracle as IO
    g = golden("improved")
    for tag, args in (("k16", IO.DEFAULT_IMPROVED_ARGS), ("k48", IO.ARGS_48K_1024)):
        sd = IO.make_improved_state_dict(seed=5, args=args)
        wav = IO.improved_forward(T(g[tag + "_y"]), sd, args)
        assert wav.shape == g[tag + "_wav"].shape
        assert np.abs(wav.numpy() - g[tag + "_wav"]).max() < 2e-6 * max(1.0, np.abs(g[tag + "_wav"]).max()), tag
    with pytest.raises(ValueError):
        IO.freq_unfold(torch.zeros(1, 1, 40, 3), 0, 21, 4, 15)


# ------------------------------------------------------------------ training step (A11)
def test_train_oracle_matches_reference_small(golden):
    from oracle import train_oracle as TO
    from oracle.make_golden_train import SMALL
    g = golden("train_small")
    sd = O.make_state_dict(seed=7, args=SMALL, sb_fc_gain=8.0)
    noisy, clean = T(g["noisy"]), T(g["clean"])
    state = None
    for it in range(2):
        r = TO.train_step(noisy, clean, sd, SMALL, state=state, n_fft=64, hop=32, win=64)
        assert abs(float(r["loss"]) - g["loss"][it]) < 1e-6 * g["loss"][it]
        assert abs(float(r["gnorm"]) - g["gnorm"][it]) < 1e-5 * g["gnorm"][it]
        if it == 0:
            assert rel_max(r["cirm"], g["cirm"]) < 2e-5  # near-0/0 bins of the ratio mask carry rounding noise
            for k in sd:
                assert rel_l2(r["grads"][k], g["grad." + k]) < 1e-5, k
        sd, state = r["sd"], r["state"]
        for k in sd:
            assert np.abs(sd[k].numpy() - g[f"p{it}." + k]).max() < 2e-6, (it, k)


def test_train_oracle_matches_reference_full(golden):
    from oracle import train_oracle as TO
    g = golden("train_full")
    sd = O.make_state_dict(seed=0, sb_fc_gain=40.0)
    r = TO.train_step(T(g["noisy"]), T(g["clean"]), sd)
    assert abs(float(r["loss"]) - g["loss"][0]) < 1e-6 * g["loss"][0]
    assert abs(float(r["gnorm"]) - g["gnorm"][0]) < 1e-4 * g["gnorm"][0] and float(r["gnorm"]) > 10  # clip active
    for k in sd:
        assert rel_l2(r["grads"][k].reshape(-1)[::97], g["gsub." + k]) < 1e-4, k
        assert np.abs(r["sd"][k].numpy().reshape(-1)[::97] - g["psub." + k]).max() < 2e-6, k


def test_manual_bptt_equals_autograd(golden):
    """The hand-derived backward the CUDA kernels implement (closed-form norm gradient, drop_band row map)."""
    from oracle import train_oracle as TO
    from oracle.make_golden_train import SMALL
    g = golden("train_small")
    sd = O.make_state_dict(seed=7, args=SMALL, sb_fc_gain=8.0)
    nm, cirm = TO.targets(T(g["noisy"]), T(g["clean"]), 2, 64, 32, 64)
    loss, grads, crm = TO.manual_backward(nm, cirm, sd, SMALL)
    assert abs(float(loss) - g["loss"][0]) < 1e-6 * g["loss"][0]
    assert np.abs(crm.numpy() - g["crm"]).max() < 1e-5
    for k in sd:
        assert rel_l2(grads[k], g["grad." + k]) < 1e-5, k
    # B = 1 (no drop_band) and G = 1
    for B, G in ((1, 2), (3, 1)):
        a = dict(SMALL, num_groups_in_drop_band=G)
        if B > 1:
            nm1, cirm1 = TO.targets(T(g["noisy"])[:B], T(g["clean"])[:B], G, 64, 32, 64)
        else:  # the trainer's drop_band asserts B > G (feature.py:317-319); Model.forward itself accepts B = 1
            nm1, _, nr, ni = O.stft(T(g["noisy"])[:1], 64, 32, 64)
            cirm1 = O.build_complex_ideal_ratio_mask(nr, ni, *O.stft(T(g["clean"])[:1], 64, 32, 64)[2:])
        l0, g0, _ = TO.loss_and_grads(nm1, cirm1, sd, a)
        l1, g1, _ = TO.manual_backward(nm1, cirm1, sd, a)
        assert abs(float(l0) - float(l1)) < 1e-6 * float(l0)
        for k in sd:
            assert rel_l2(g1[k], g0[k]) < 1e-5, (B, G, k)


def test_cumulative_laplace_norm_oracle_matches_reference(golden):
    """SURVEY 8f rank 1: norm_type = cumulative_laplace_norm (base_model.py:220-251) through the whole model."""
    g = golden("model_cum")
    small = dict(num_freqs=33, look_ahead=2, sequence_model="LSTM", fb_num_neighbors=0, sb_num_neighbors=3,
                 fb_output_activate_function="ReLU", sb_output_activate_function=False, fb_model_hidden_size=32,
                 sb_model_hidden_size=24, norm_type="cumulative_laplace_norm", num_groups_in_drop_band=2)
    sd = O.make_state_dict(seed=7, args=small)
    mag = T(g["small_mag"]).unsqueeze(1)
    assert rel_max(O.model_forward(mag[:1], sd, small), g["small_b1"]) < 2e-5
    assert rel_max(O.model_forward(mag, sd, small), g["small_g2"]) < 2e-5
    full = dict(O.DEFAULT_MODEL_ARGS, norm_type="cumulative_laplace_norm")
    sdf = O.make_state_dict(seed=0, args=full, sb_fc_gain=60.0)
    wav, crm = O.enhance(T(g["full_y"]), sdf, full, return_crm=True)
    assert rel_max(crm, g["full_crm"]) < 5e-5
    assert np.abs(wav.numpy() - g["full_wav"]).max() < 1e-5


def test_improved_fullsubnet_960_oracle_matches_reference(golden):
    """The reference's own 48 kHz example (model.py:603-620): n_fft = 960, 12.18 M parameters (SURVEY A14)."""
    from oracle import improved_fullsubnet_oracle as IO
    g = golden("improved_960")
    sd = IO.make_improved_state_dict(seed=5, args=IO.ARGS_48K_960)
    assert sum(v.numel() for v in sd.values()) == 12_180_874  # "12.18 M" (SURVEY A14)
    wav = IO.improved_forward(T(g["y"]), sd, IO.ARGS_48K_960)
    assert np.abs(wav.numpy() - g["wav"]).max() < 2e-6 * max(1.0, np.abs(g["wav"]).max())
    mag, _, re, im = O.stft(T(g["y"]), 960, 480, 960)
    assert rel_max(re, g["real"]) < 5e-6 and rel_max(im, g["imag"]) < 5e-6 and rel_max(mag, g["mag"]) < 5e-6


def test_fullband_baseline_oracle_matches_reference(golden):
    """SURVEY 8f rank 3: 3 x LSTM + Linear(2F) (fullband_baseline/model.py:8-68), both norms."""
    from oracle import fullband_baseline_oracle as BO
    g = golden("fullband_baseline")
    small = dict(BO.DEFAULT_FBB_ARGS, num_freqs=33, hidden_size=32, output_activate_function="ReLU",
                 norm_type="cumulative_laplace_norm")
    for tag, a in (("small", small), ("full", dict(BO.DEFAULT_FBB_ARGS))):
        out = BO.fbb_forward(T(g[tag + "_mag"]), BO.make_fbb_state_dict(seed=11, args=a), a)
        assert out.shape == g[tag + "_out"].shape and rel_max(out, g[tag + "_out"]) < 2e-5, tag


# ------------------------------------------------------------------ the timed CPU arm and the config-length fixtures
def test_libcall_port_is_the_reference_computation(golden):
    """bench.py's CPU arm (oracle/libcall_port.py: the path written with the reference's own torch library calls)
    reproduces the outputs of the unmodified reference - so what is TIMED on the host is the reference's computation."""
    from oracle import libcall_port as P
    g = golden("model_full")
    y = T(g["y"])
    # the fixtures were made on 8 threads (make_golden.py); the LSTM's CPU GEMMs split their sums by the thread count,
    # so other counts move the waveform by a few 1e-6
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        for tag, gain in (("wa", 1.0), ("wb", WB_GAIN)):
            wav, crm = P.enhance(y, P.LibcallModel(O.make_state_dict(seed=0, sb_fc_gain=gain)), return_crm=True)
            assert rel_max(crm, g[f"{tag}_crm"]) < 1e-6
            assert np.abs(wav.numpy() - g[f"{tag}_wav"]).max() < 1e-6
    finally:
        torch.set_num_threads(threads)


def _fingerprint(y):
    a = y.numpy().astype(np.float64)
    return np.concatenate([a.reshape(-1)[:8], [a.sum(), np.abs(a).sum()]])


def test_oracle_at_config_length_4s(golden):
    """T = 251 (BASELINE configs 0/1 clip length), both weight sets: oracle vs the unmodified reference."""
    y = O.make_noisy(1, 64000, seed=40, speechlike=True)
    torch.set_num_threads(8)
    for tag, gain in (("wa", 1.0), ("wb", WB_GAIN)):
        g = golden(f"model_full_4s_{tag}")
        assert np.allclose(_fingerprint(y), g["y_fp"], rtol=0, atol=1e-9)
        with torch.no_grad():
            wav, crm = O.enhance(y, O.make_state_dict(seed=0, sb_fc_gain=gain), return_crm=True)
        assert rel_max(crm, g["crm"]) < 5e-5 and rel_l2(crm, g["crm"]) < 5e-5
        assert np.abs(wav.numpy() - g["wav"]).max() < 1e-4


def test_gru_oracle_matches_reference(golden):
    """sequence_model="GRU" (sequence_model.py:59-66): oracle gru_stack vs the unmodified reference."""
    g = golden("model_gru")
    a = dict(_small_args(), sequence_model="GRU")
    sd = O.make_state_dict(seed=7, args=a)
    assert sd["fb_model.sequence_model.weight_ih_l0"].shape == (3 * 32, 33)
    mag = T(g["small_mag"]).unsqueeze(1)
    assert rel_max(O.model_forward(mag[:1], sd, a), g["small_b1"]) < 1e-5
    assert rel_max(O.model_forward(mag, sd, a), g["small_g2"]) < 1e-5
    full = dict(O.DEFAULT_MODEL_ARGS, sequence_model="GRU")
    wav, crm = O.enhance(T(g["full_y"]), O.make_state_dict(seed=0, args=full, sb_fc_gain=60.0), full, return_crm=True)
    assert rel_max(crm, g["full_crm"]) < 2e-5
    assert np.abs(wav.numpy() - g["full_wav"]).max() < 1e-5


def test_snr_mix_oracle_matches_reference(golden):
    """Dataset.snr_mix (dataset_train.py:136-199): plain, negative SNR, reverberant and clipped cases."""
    from oracle import mix_oracle as M
    g = golden("mix")
    for i, (snr, draw, rir_len) in enumerate(g["cases"]):
        rir = g[f"c{i}_rir"] if rir_len else None
        noisy, clean = M.snr_mix(g[f"c{i}_clean"], g[f"c{i}_noise"], float(snr), -25, float(draw), rir=rir)
        assert rel_max(noisy, g[f"c{i}_noisy"]) < 2e-5 and rel_max(clean, g[f"c{i}_clean_out"]) < 2e-5, i
    assert np.abs(g["c1_noisy"]).max() > 0.98  # the clipped case really took the rescale branch (max = 0.99 - eps)
