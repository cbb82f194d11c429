"""Pin the CPU oracle against outputs of the reference modules (tests/golden)."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_APNET, GOLDEN_MODELS, GOLDEN_NSF, GOLDEN_VITS, load_golden, load_golden_apnet, load_golden_vits
from oracle import generator as og
from oracle import io as oio
from oracle import mel as om


@pytest.mark.parametrize("name", sorted(GOLDEN_MODELS))
def test_generator_matches_reference(name):
    kind, hp, _ = GOLDEN_MODELS[name]
    g, sd = load_golden(name)
    wav, stages = og.generator_forward(kind, sd, hp, g["mel"], return_stages=True)
    for i, s in enumerate(stages):
        np.testing.assert_allclose(s, g[f"stage{i}"], atol=2e-6, rtol=1e-5)
    np.testing.assert_allclose(wav, g["wav"], atol=1e-6, rtol=0)


def test_nsfhifigan_oracle_matches_reference():
    # the reference's output does not depend on the (random) harmonic source: nsfhifigan.py:269
    kind, hp, _ = GOLDEN_NSF
    g, sd = load_golden("nsfhifigan")
    np.testing.assert_array_equal(g["wav"], g["wav_other_source"])
    np.testing.assert_array_equal(g["wav"], g["wav_long_f0"])
    wav = og.generator_forward(kind, sd, hp, g["mel"], f0=g["f0"])
    np.testing.assert_allclose(wav, g["wav"], atol=1e-6, rtol=0)
    mels = [g[f"pl_mel{i}"] for i in range(3)]
    f0s = [g[f"pl_f0{i}"] for i in range(3)]
    auds = og.synthesis_audios(kind, sd, hp, mels, hop_size=16, batch_size=2, f0s=f0s)
    for i, a in enumerate(auds):
        assert a.shape == g[f"pl_audio{i}"].shape
        np.testing.assert_allclose(a, g[f"pl_audio{i}"], atol=1e-6)
    # a source shorter than the mel truncates every stage (:264-268)
    short = og.generator_forward(kind, sd, hp, g["mel"], f0=g["f0"][:, :11])
    assert short.shape[-1] == 11 * 16


def test_fold_weight_norm_matches_torch():
    _, sd = load_golden("hifigan_rb1")
    for name in ["conv_pre", "ups.0", "resblocks.2.convs1.1", "conv_post"]:
        v, g = torch.from_numpy(sd[name + ".weight_v"]), torch.from_numpy(sd[name + ".weight_g"])
        ref = torch._weight_norm(v, g, 0).numpy()
        np.testing.assert_allclose(og.fold_weight_norm(sd[name + ".weight_v"], sd[name + ".weight_g"]),
                                   ref, rtol=2e-6, atol=1e-9)


def test_numpy_primitives_match_torch_primitives():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, 5, 23)).astype(np.float32)
    w = rng.standard_normal((4, 5, 7)).astype(np.float32)
    b = rng.standard_normal(4).astype(np.float32)
    for d in (1, 3):
        p = og.get_padding(7, d)
        np.testing.assert_allclose(og.conv1d_np(x, w, b, d, p), og.conv1d(x, w, b, d, p).numpy(), atol=2e-5)
    wt = rng.standard_normal((5, 3, 8)).astype(np.float32)
    bt = rng.standard_normal(3).astype(np.float32)
    np.testing.assert_allclose(og.conv_transpose1d_np(x, wt, bt, 4, 2),
                               og.conv_transpose1d(x, wt, bt, 4, 2).numpy(), atol=2e-5)
    np.testing.assert_allclose(og.conv_transpose1d_np(x, wt[:, :, :4], bt, 2, 1),
                               og.conv_transpose1d(x, wt[:, :, :4], bt, 2, 1).numpy(), atol=2e-5)


def test_activation1d_closed_forms_match_reference():
    g, _ = load_golden("activation1d")
    up = og.upsample2x_np(g["x"], g["f_up"])
    np.testing.assert_allclose(up, g["up"], atol=2e-6)
    y = og.activation1d_np(g["x"], g["alpha"], g["beta"], True, g["f_up"], g["f_down"])
    np.testing.assert_allclose(y, g["y"], atol=3e-6)
    yt = og.activation1d(torch.from_numpy(g["x"]), g["alpha"], g["beta"], True, g["f_up"], g["f_down"]).numpy()
    np.testing.assert_allclose(yt, g["y"], atol=1e-6)
    np.testing.assert_allclose(og.kaiser_sinc_filter12(), g["f_up"], atol=1e-8)
    # short sequences: the replicate clamps overlap (T < filter reach)
    for t in (1, 2, 3, 7):
        x = torch.randn(1, 3, t)
        a = og.activation1d(x, g["alpha"][:3], g["beta"][:3], True, g["f_up"], g["f_down"]).numpy()
        b = og.activation1d_np(x.numpy(), g["alpha"][:3], g["beta"][:3], True, g["f_up"], g["f_down"])
        np.testing.assert_allclose(a, b, atol=3e-6)


def test_plumbing_matches_reference():
    kind, hp, _ = GOLDEN_MODELS["hifigan_rb1"]
    _, sd = load_golden("hifigan_rb1")
    g, _ = load_golden("plumbing")
    mels = [g[f"mel{i}"] for i in range(3)]
    auds = og.synthesis_audios(kind, sd, hp, mels, hop_size=8, batch_size=2)
    for i, a in enumerate(auds):
        assert a.shape == g[f"audio{i}"].shape
        np.testing.assert_allclose(a, g[f"audio{i}"], atol=1e-6)
    np.testing.assert_allclose(og.vocoder_inference(kind, sd, hp, g["batched_in"]), g["batched_out"], atol=1e-6)


def test_mel_oracle_matches_reference():
    g, _ = load_golden("mel")
    y, mb = g["y"], g["mel_basis"]
    lin = om.extract_linear_features(y, 1024, 256, 1024)
    np.testing.assert_allclose(lin, g["extract_linear_features"], atol=2e-4, rtol=1e-4)
    m = om.extract_mel_features(y, mb, 1024, 256, 1024, eps=1e-9)
    np.testing.assert_allclose(m, g["extract_mel_features"], atol=1e-4)
    m6 = om.extract_mel_features(y, mb, 1024, 256, 1024, eps=1e-6)
    np.testing.assert_allclose(m6, g["mel_spectrogram_torch"], atol=1e-4)
    assert g["extract_mel_features_b1"].shape == (80, 32)          # the reference's squeeze(0)
    np.testing.assert_allclose(m[0], g["extract_mel_features_b1"], atol=1e-4)
    m2 = om.extract_mel_features(g["y2"], g["mel_basis2"], 512, 160, 400)
    np.testing.assert_allclose(m2, g["extract_mel_features2"], atol=1e-4)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_mel_vjp_oracle_matches_reference_autograd(tag):
    """oracle.mel.extract_mel_features_vjp against what torch autograd computed through the reference's
    extract_mel_features (fixture made by tests/golden/gen_golden.py mel_grad)."""
    g, _ = load_golden("mel_grad")
    n_fft, hop, win, n_mel = (int(v) for v in g[tag + "_geom"])
    y, mb = g[tag + "_y_pred"], g[tag + "_mel_basis"]
    got = om.extract_mel_features_vjp(y, mb, g[tag + "_cot"], n_fft, hop, win)
    want = g[tag + "_grad_cot"]
    assert np.abs(got - want).max() <= 2e-4 * np.abs(want).max()
    # the trainers' loss: 45 * mean |mel_gt - mel_pred|  ->  cotangent 45 * sign(pred - gt) / numel
    mel_gt = om.extract_mel_features(g[tag + "_y_gt"], mb, n_fft, hop, win)
    mel_pred = om.extract_mel_features(y, mb, n_fft, hop, win)
    np.testing.assert_allclose(45 * np.abs(mel_gt - mel_pred).mean(), g[tag + "_loss"], rtol=1e-4)
    cot = 45.0 * np.sign(mel_pred - mel_gt) / mel_pred.size
    got = om.extract_mel_features_vjp(y, mb, cot, n_fft, hop, win)
    want = g[tag + "_grad_loss"]
    assert np.abs(got - want).max() <= 5e-4 * np.abs(want).max()
    silent = slice(y.shape[1] // 3 + n_fft, y.shape[1] // 3 + 2 * n_fft)   # frames wholly inside the zeroed span
    assert np.abs(want[0, silent]).max() < 1e-3 * np.abs(want).max()


def test_tacotron_oracle_matches_reference():
    g, _ = load_golden("mel")
    np.testing.assert_array_equal(g["taco_mel_basis"], g["mel_basis"])
    mel, energy = om.tacotron_mel(g["y"], g["mel_basis"], 1024, 256, 1024)
    assert mel.shape == g["taco_mel"].shape == (2, 80, 33)
    np.testing.assert_allclose(mel, g["taco_mel"], atol=2e-4)
    np.testing.assert_allclose(energy, g["taco_energy"], rtol=1e-4)
    with pytest.raises(AssertionError):
        om.tacotron_mel(g["y"] * 2, g["mel_basis"], 1024, 256, 1024)


def test_mel_filterbank_matches_torchaudio():
    ta = pytest.importorskip("torchaudio")
    fb = ta.functional.melscale_fbanks(513, 0.0, 8000.0, 80, 22050, norm="slaney", mel_scale="slaney").T.numpy()
    np.testing.assert_allclose(om.slaney_mel_filterbank(22050, 1024, 80, 0, 8000), fb, atol=5e-7)


def test_save_audio_oracle_matches_reference():
    g, _ = load_golden("save_audio")
    for ts in (0, 1):
        for sil in (0, 1):
            got = oio.save_audio_float(g["w"], 16000, add_silence=bool(sil), turn_up=bool(ts))
            np.testing.assert_array_equal(got, g[f"float_turnup{ts}_silence{sil}"])
    assert np.abs(g["float_turnup1_silence0"]).max() == np.float32(0.9) or abs(np.abs(g["float_turnup1_silence0"]).max() - 0.9) < 1e-7
    # quantiser known answers (sox: (x * 2^31 + 0x8000) >> 16, clipped)
    x = np.array([0.0, 0.5, -0.5, 1.0, -1.0, 1.5, -1.5, 1 / 32768, 1.5 / 32768, -1.5 / 32768, 0.49 / 32768, -0.51 / 32768],
                 np.float32)
    np.testing.assert_array_equal(oio.pcm16(x), [0, 16384, -16384, 32767, -32768, 32767, -32768, 1, 2, -1, 0, -1])


@pytest.mark.parametrize("tag", sorted(GOLDEN_VITS))
def test_hifigan_vits_oracle_matches_reference(tag):
    g, sd = load_golden_vits(tag)
    hp = GOLDEN_VITS[tag]
    np.testing.assert_allclose(og.hifigan_vits_forward(sd, hp, g["x"]), g["wav"], atol=1e-6, rtol=0)
    if "g" in g:
        np.testing.assert_allclose(og.hifigan_vits_forward(sd, hp, g["x"], g["g"]), g["wav_g"], atol=1e-6, rtol=0)


def test_apnet_oracle_matches_reference():
    """oracle.generator.apnet_forward / istft_same against APNet.forward of the reference (apnet.py:357-399)."""
    from oracle import generator as og
    hp, pre = GOLDEN_APNET
    g, sd = load_golden_apnet()
    logamp, pha, rea, imag, audio = og.apnet_forward(sd, hp, g["mel"], pre["n_fft"], pre["hop_size"], pre["win_size"])
    np.testing.assert_allclose(logamp, g["logamp"], atol=2e-5)
    np.testing.assert_allclose(rea, g["rea"], atol=2e-4, rtol=1e-4)
    np.testing.assert_allclose(imag, g["imag"], atol=2e-4, rtol=1e-4)
    d = np.abs(pha - g["pha"])
    assert np.minimum(d, 2 * np.pi - d).max() < 1e-3                     # the branch cut at +-pi
    assert audio.shape == g["audio"].shape == (2, 1, 23 * pre["hop_size"])
    np.testing.assert_allclose(audio, g["audio"], atol=2e-5)
    np.testing.assert_allclose(audio[:, 0], g["inference"], atol=2e-5)     # vocoder_inference takes the fifth output


def test_amplitude_phase_oracle_matches_reference():
    """oracle.mel.amplitude_phase_spectrum against utils/mel.py:244-280 (fixture amp_phase.npz)."""
    g, _ = load_golden("amp_phase")
    la, ph, re, im = om.amplitude_phase_spectrum(g["y"], 256, 64, 256)
    assert la.shape == g["logamp"].shape == (2, 129, 46) and tuple(g["b1_shape"]) == (129, 46)
    scale = np.abs(g["rea"]).max()
    np.testing.assert_allclose(re, g["rea"], atol=2e-5 * scale)
    np.testing.assert_allclose(im, g["imag"], atol=2e-5 * scale)
    np.testing.assert_allclose(la, g["logamp"], atol=2e-3)            # log of small magnitudes amplifies fp32 FFT noise
    mag = np.sqrt(g["rea"] ** 2 + g["imag"] ** 2)
    d = np.abs(ph - g["pha"])
    assert (np.minimum(d, 2 * np.pi - d) * mag).max() <= 1e-4 * scale  # phase weighted by the modulus it belongs to
