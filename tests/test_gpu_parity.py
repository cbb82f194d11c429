"""GPU parity tests proper: the CUDA path (through the C ABI / the Python
mirrors of the reference interface) against the CPU oracle and the committed
reference-generated golden fixtures.  Tolerances are stated per test; the
north-star bar is 1e-3 max-abs on the generator output, fp32."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_MODELS, GOLDEN_VITS, load_golden, load_golden_vits
from helpers import HP_BIGVGAN_BASE, HP_NSF_EXP, HP_V1, build_model, golden_model, make_cfg, randomize_snake, sd_numpy
from oracle import generator as og
from oracle import mel as om

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ws(nbytes):
    t = torch.empty(nbytes + 256, dtype=torch.uint8, device=DEV)
    return t, C.c_void_p((t.data_ptr() + 255) // 256 * 256)


def run_conv1d(x, w, b, res, k, d, pre_slope, tanh, precision="fp32"):
    from amphion_b200 import _capi
    B, cin, T = x.shape
    cout = w.shape[0]
    xd, wd = torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV)
    bd = torch.from_numpy(b).to(DEV) if b is not None else None
    rd = torch.from_numpy(res).to(DEV) if res is not None else None
    y = torch.empty(B, cout, T, device=DEV)
    prec = _capi.PRECISIONS[precision]
    n = _capi.lib.ab_conv1d_workspace_bytes(cin, cout, k, prec)
    keep, ws = _ws(n)
    _capi.check(_capi.lib.ab_conv1d_forward(_capi.ptr(xd), _capi.ptr(wd), _capi.ptr(bd), _capi.ptr(rd), _capi.ptr(y),
                                            B, cin, cout, T, k, d, pre_slope, int(tanh), prec, ws, n,
                                            _capi.stream_ptr()), "ab_conv1d_forward")
    torch.cuda.synchronize()
    return y.cpu().numpy()


def oracle_conv1d(x, w, b, res, k, d, pre_slope, tanh, operand_dtype=None):
    xa = og.leaky_relu_np(x, pre_slope) if pre_slope != 1.0 else x
    wa = w
    if operand_dtype is not None:  # model the tensor path: operands rounded, fp32+ accumulation
        xa = torch.from_numpy(xa).to(operand_dtype).double().numpy()
        wa = torch.from_numpy(w).to(operand_dtype).double().numpy()
        y = torch.nn.functional.conv1d(torch.from_numpy(xa), torch.from_numpy(wa), None, dilation=d,
                                       padding=og.get_padding(k, d)).numpy()
        y = y + (b[None, :, None].astype(np.float64) if b is not None else 0)
    else:
        y = og.conv1d(xa, wa, b, d, og.get_padding(k, d)).numpy().astype(np.float64)
    if res is not None:
        y = y + res
    if tanh:
        y = np.tanh(y)
    return y.astype(np.float32)


CONV_CASES = [
    # B, cin, cout, T, k, d, pre_slope, residual, tanh
    (2, 5, 7, 50, 3, 1, 1.0, False, False),
    (1, 16, 64, 300, 7, 3, 0.1, True, False),
    (2, 80, 96, 129, 7, 1, 1.0, False, False),       # conv_pre-like, cout not a multiple of 64
    (1, 32, 32, 1000, 11, 5, 0.1, True, False),
    (2, 24, 24, 77, 5, 12, 0.1, True, False),        # ResBlock2-style wide dilation, T < halo*2
    (3, 32, 1, 2500, 7, 1, 0.01, False, True),       # conv_post + tanh (few-out kernel, multi-tile)
    (1, 9, 2, 5, 7, 1, 1.0, False, False),           # T shorter than the filter
    (1, 4, 4, 1, 3, 1, 0.1, True, False),            # single sample
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv1d_fp32_matches_oracle(case):
    B, cin, cout, T, k, d, slope, use_res, tanh = case
    rng = np.random.default_rng(hash(case) % 2**32)
    x = rng.standard_normal((B, cin, T)).astype(np.float32)
    w = (rng.standard_normal((cout, cin, k)) / np.sqrt(cin * k)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32)
    res = rng.standard_normal((B, cout, T)).astype(np.float32) if use_res else None
    got = run_conv1d(x, w, b, res, k, d, slope, tanh)
    want = oracle_conv1d(x, w, b, res, k, d, slope, tanh)
    np.testing.assert_allclose(got, want, atol=2e-5, rtol=1e-5)   # fp32, summation order only


@pytest.mark.parametrize("case", [(2, 6, 5, 40, 8, 4), (1, 64, 32, 130, 16, 8), (2, 32, 16, 257, 4, 2),
                                  (1, 8, 8, 1, 4, 2), (1, 16, 70, 33, 8, 4), (1, 12, 12, 50, 7, 3)])
@pytest.mark.parametrize("slope", [1.0, 0.1])
def test_conv_transpose1d_matches_oracle(case, slope):
    got = run_conv_transpose1d(case, slope, "fp32")[0]
    want = oracle_conv_transpose1d(case, slope)
    np.testing.assert_allclose(got, want, atol=2e-5, rtol=1e-5)


def _convt_inputs(case):
    B, cin, cout, T, k, u = case
    rng = np.random.default_rng(sum(case))
    x = rng.standard_normal((B, cin, T)).astype(np.float32)
    w = (rng.standard_normal((cin, cout, k)) / np.sqrt(cin)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32)
    return x, w, b


def run_conv_transpose1d(case, slope, precision):
    from amphion_b200 import _capi
    B, cin, cout, T, k, u = case
    x, w, b = _convt_inputs(case)
    xd, wd, bd = (torch.from_numpy(a).to(DEV) for a in (x, w, b))
    y = torch.full((B, cout, T * u), float("nan"), device=DEV)
    prec = _capi.PRECISIONS[precision]
    n = _capi.lib.ab_conv_transpose1d_workspace_bytes(cin, cout, k, u, prec)
    keep, ws = _ws(n)
    _capi.check(_capi.lib.ab_conv_transpose1d_forward(_capi.ptr(xd), _capi.ptr(wd), _capi.ptr(bd), _capi.ptr(y), B, cin,
                                                      cout, T, k, u, slope, prec, ws, n, _capi.stream_ptr()),
                "ab_conv_transpose1d_forward")
    torch.cuda.synchronize()
    return y.cpu().numpy(), x, w, b


def oracle_conv_transpose1d(case, slope, operand_dtype=None):
    B, cin, cout, T, k, u = case
    x, w, b = _convt_inputs(case)
    xa = og.leaky_relu_np(x, slope)
    if operand_dtype is None:
        return og.conv_transpose1d(xa, w, b, u, (k - u) // 2).numpy()
    xa = torch.from_numpy(xa).to(operand_dtype).double()
    wa = torch.from_numpy(w).to(operand_dtype).double()
    y = torch.nn.functional.conv_transpose1d(xa, wa, torch.from_numpy(b).double(), stride=u, padding=(k - u) // 2)
    return y.float().numpy()


TC_CONVT_CASES = [(2, 64, 32, 130, 16, 8), (1, 512, 256, 70, 16, 8), (2, 128, 64, 300, 4, 2), (1, 64, 32, 1000, 4, 2),
                  (1, 32, 16, 257, 8, 4), (1, 48, 24, 33, 8, 4), (2, 16, 70, 33, 8, 4), (1, 12, 12, 50, 7, 3),
                  (1, 256, 128, 1, 16, 8)]


@pytest.mark.parametrize("case", TC_CONVT_CASES)
@pytest.mark.parametrize("prec", ["tc_f16", "tc_bf16"])
def test_tc_conv_transpose1d_matches_operand_rounded_oracle(case, prec):
    got = run_conv_transpose1d(case, 0.1, prec)[0]
    assert np.isfinite(got).all()          # every output element written exactly once (buffer pre-filled with NaN)
    dt = torch.float16 if prec == "tc_f16" else torch.bfloat16
    np.testing.assert_allclose(got, oracle_conv_transpose1d(case, 0.1, dt), atol=3e-5, rtol=1e-5)
    assert np.abs(got - oracle_conv_transpose1d(case, 0.1)).max() < (3e-3 if prec == "tc_f16" else 3e-2)


def test_conv_transpose1d_rejects_odd_geometry():
    from amphion_b200 import _capi
    x = torch.zeros(1, 2, 4, device=DEV)
    w = torch.zeros(2, 2, 5, device=DEV)
    y = torch.zeros(1, 2, 8, device=DEV)
    keep, ws = _ws(1024)
    rc = _capi.lib.ab_conv_transpose1d_forward(_capi.ptr(x), _capi.ptr(w), None, _capi.ptr(y), 1, 2, 2, 4, 5, 2, 1.0,
                                               0, ws, 1024, _capi.stream_ptr())
    assert rc == -2 and "even" in _capi.last_error()


def test_activation1d_matches_reference_fixture_and_oracle():
    from amphion_b200.vocoders.activations import Activation1d, SnakeBeta, Snake
    g, _ = load_golden("activation1d")
    act = Activation1d(SnakeBeta(6, alpha_logscale=True)).to(DEV)
    with torch.no_grad():
        act.act.alpha.copy_(torch.from_numpy(g["alpha"]))
        act.act.beta.copy_(torch.from_numpy(g["beta"]))
    y = act(torch.from_numpy(g["x"]).to(DEV)).cpu().numpy()
    np.testing.assert_allclose(y, g["y"], atol=5e-6)     # reference module output
    rng = np.random.default_rng(1)
    for (B, Cn, T, logscale, cls) in [(1, 3, 1, True, SnakeBeta), (2, 2, 2, False, Snake), (1, 5, 7, True, Snake),
                                      (2, 4, 1024, True, SnakeBeta), (1, 3, 2049, False, SnakeBeta),
                                      (1, 2, 5000, True, SnakeBeta)]:
        a = Activation1d(cls(Cn, alpha_logscale=logscale)).to(DEV)
        with torch.no_grad():
            a.act.alpha.normal_(0.0 if logscale else 1.0, 0.3)
            if cls is SnakeBeta:
                a.act.beta.normal_(0.0 if logscale else 1.0, 0.3)
        x = (rng.standard_normal((B, Cn, T)) * 3).astype(np.float32)
        got = a(torch.from_numpy(x).to(DEV)).cpu().numpy()
        beta = a.act.beta if cls is SnakeBeta else a.act.alpha
        want = og.activation1d_np(x, a.act.alpha.detach().cpu().numpy(), beta.detach().cpu().numpy(), logscale,
                                  g["f_up"], g["f_down"])
        np.testing.assert_allclose(got, want, atol=2e-5, rtol=1e-5)


@pytest.mark.parametrize("name", sorted(GOLDEN_MODELS))
def test_generator_fp32_matches_reference_fixture(name):
    kind, hp, g, sd, model = golden_model(name)
    model = model.to(DEV)
    model.precision = "fp32"
    wav = model(torch.from_numpy(g["mel"]).to(DEV))
    assert wav.shape == g["wav"].shape and wav.dtype == torch.float32 and wav.is_cuda
    np.testing.assert_allclose(wav.cpu().numpy(), g["wav"], atol=2e-5)   # bar: 1e-3
    assert model.last_launches > 0


@pytest.mark.parametrize("name", sorted(GOLDEN_MODELS))
def test_generator_tensor_core_matches_reference_fixture(name):
    kind, hp, g, sd, model = golden_model(name)
    model = model.to(DEV)
    for prec, tol in (("tc_f16", 5e-4), ("tc_bf16", 4e-3)):   # bf16 is a non-default mode (8-bit mantissa)
        model.precision = prec
        wav = model(torch.from_numpy(g["mel"]).to(DEV)).cpu().numpy()
        assert np.isfinite(wav).all()
        assert np.abs(wav - g["wav"]).max() <= tol, (prec, np.abs(wav - g["wav"]).max())


TC_CASES = [
    # C, T, k, d   (single conv through the tcgen05 kernel)
    (64, 128, 1, 1),      # pure GEMM: no tap shifts
    (64, 200, 3, 1),      # tap shifts of one row
    (32, 1000, 3, 3),
    (128, 700, 7, 3),
    (256, 600, 11, 5),    # V1 stage-0 worst case, multi-tile
    (48, 333, 5, 2),      # channels padded 48 -> 48 (16-multiple), K chunk of 16 left over
    (24, 90, 3, 1),       # channels padded 24 -> 32
    (256, 50, 11, 1),     # sequence shorter than one tile
]


@pytest.mark.parametrize("case", TC_CASES)
@pytest.mark.parametrize("prec", ["tc_f16", "tc_bf16"])
def test_tc_conv1d_matches_operand_rounded_oracle(case, prec):
    C_, T, k, d = case
    rng = np.random.default_rng(C_ * 1000 + T + k)
    x = rng.standard_normal((2, C_, T)).astype(np.float32)
    w = (rng.standard_normal((C_, C_, k)) / np.sqrt(C_ * k)).astype(np.float32)
    b = rng.standard_normal(C_).astype(np.float32)
    res = rng.standard_normal((2, C_, T)).astype(np.float32)
    got = run_conv1d(x, w, b, res, k, d, 0.1, False, precision=prec)
    dt = torch.float16 if prec == "tc_f16" else torch.bfloat16
    want = oracle_conv1d(x, w, b, res, k, d, 0.1, False, operand_dtype=dt)
    # identical operands, fp32 accumulation in a different order: tight
    np.testing.assert_allclose(got, want, atol=3e-5, rtol=1e-5)
    exact = oracle_conv1d(x, w, b, res, k, d, 0.1, False)
    assert np.abs(got - exact).max() < (3e-3 if prec == "tc_f16" else 3e-2)


TC_WIDE_CASES = [
    # B, cin, cout, T, k, d, pre_slope, residual, tanh   (N-blocked tensor-core kernel, conv mode)
    (2, 80, 512, 300, 7, 1, 1.0, False, False),      # conv_pre of HiFi-GAN V1 (2 N blocks, K = 80)
    (1, 100, 96, 130, 7, 1, 1.0, False, False),      # conv_pre-like, BigVGAN mel count, N padded
    (2, 32, 1, 2500, 7, 1, 0.01, False, True),       # conv_post + tanh (N = 16 with one live column)
    (1, 64, 320, 77, 3, 2, 0.1, True, False),        # residual, dilation, T < tile
]


@pytest.mark.parametrize("case", TC_WIDE_CASES)
def test_tc_wide_conv1d_matches_operand_rounded_oracle(case):
    B, cin, cout, T, k, d, slope, use_res, tanh = case
    rng = np.random.default_rng(cin * 7 + cout)
    x = rng.standard_normal((B, cin, T)).astype(np.float32)
    w = (rng.standard_normal((cout, cin, k)) / np.sqrt(cin * k)).astype(np.float32)
    b = rng.standard_normal(cout).astype(np.float32)
    res = rng.standard_normal((B, cout, T)).astype(np.float32) if use_res else None
    got = run_conv1d(x, w, b, res, k, d, slope, tanh, precision="tc_f16")
    want = oracle_conv1d(x, w, b, res, k, d, slope, tanh, operand_dtype=torch.float16)
    np.testing.assert_allclose(got, want, atol=3e-5, rtol=1e-5)


def _full_size_case(kind, hp, n_mel, B, T, seed):
    model = build_model(kind, hp, n_mel, seed=seed)
    if kind == "bigvgan":
        randomize_snake(model, seed + 1, hp["snake_logscale"])
    g = torch.Generator().manual_seed(seed + 2)
    mel = torch.randn(B, n_mel, T, generator=g)
    want = og.generator_forward(kind, sd_numpy(model), hp, mel.numpy())
    return model.to(DEV), mel, want


@pytest.mark.parametrize("prec,tol", [("fp32", 5e-5), ("tc_f16", 1e-3)])
def test_hifigan_v1_full_width_matches_oracle(prec, tol):
    """BASELINE config 1/2 architecture (512 ch, rates 8.8.2.2) at a CPU-checkable size."""
    model, mel, want = _full_size_case("hifigan", HP_V1, 80, 2, 40, seed=1234)
    model.precision = prec
    got = model(mel.to(DEV)).cpu().numpy()
    assert got.shape == (2, 1, 40 * 256)
    assert np.abs(got - want).max() <= tol, np.abs(got - want).max()


@pytest.mark.parametrize("prec,tol", [("fp32", 1e-4), ("tc_f16", 1e-3)])
def test_bigvgan_base_full_width_matches_oracle(prec, tol):
    """BASELINE config 3 architecture (snakebeta, logscale, 100 mels) at a CPU-checkable size."""
    model, mel, want = _full_size_case("bigvgan", HP_BIGVGAN_BASE, 100, 1, 24, seed=77)
    model.precision = prec
    got = model(mel.to(DEV)).cpu().numpy()
    assert np.abs(got - want).max() <= tol, np.abs(got - want).max()


def test_bigvgan_wide_layers_match_oracle():
    """BigVGAN-large style widths: stage 0 has 384 channels (> 256: streaming N-blocked tensor-core kernel),
    stage 1 has 192 (pair kernel); CPU-checkable length."""
    hp = dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4], upsample_initial_channel=768,
              resblock_kernel_sizes=[3, 11], resblock_dilation_sizes=[[1, 3, 5]] * 2, activation="snakebeta",
              snake_logscale=True)
    model, mel, want = _full_size_case("bigvgan", hp, 20, 2, 37, seed=5)
    for prec, tol in (("fp32", 1e-4), ("tc_f16", 1e-3)):
        model.precision = prec
        got = model(mel.to(DEV)).cpu().numpy()
        assert np.isfinite(got).all()
        assert np.abs(got - want).max() <= tol, (prec, np.abs(got - want).max())
    # BigVGAN-large widths: the first ConvTranspose is 1536 -> 768 (C_in beyond a resident tile: streaming
    # conv-transpose with fp32 loader warps), stage 0 runs 768 channels
    hp = dict(hp, upsample_initial_channel=1536, resblock_kernel_sizes=[3], resblock_dilation_sizes=[[1, 3]])
    model, mel, want = _full_size_case("bigvgan", hp, 12, 1, 19, seed=8)
    model.precision = "tc_f16"
    got = model(mel.to(DEV)).cpu().numpy()
    assert np.isfinite(got).all()
    assert np.abs(got - want).max() <= 1e-3, np.abs(got - want).max()


def test_nsfhifigan_matches_reference_fixture():
    """NSFHiFiGAN.forward (nsfhifigan.py:262-283) against the output of the reference module: the fixture
    pins that the (random) harmonic source never reaches the samples, only `x = x + x` does."""
    from amphion_b200.vocoders.gan_vocoder_inference import synthesis_audios, vocoder_inference
    kind, hp, g, sd, model = golden_model("nsfhifigan")
    model = model.to(DEV)
    mel, f0 = torch.from_numpy(g["mel"]).to(DEV), torch.from_numpy(g["f0"]).to(DEV)
    for prec, tol in (("fp32", 2e-5), ("tc_f16", 5e-4), ("tc_bf16", 4e-3)):
        model.precision = prec
        wav = model(mel, f0)
        assert wav.shape == g["wav"].shape and wav.is_cuda
        assert np.abs(wav.cpu().numpy() - g["wav"]).max() <= tol, (prec, np.abs(wav.cpu().numpy() - g["wav"]).max())
    model.precision = "fp32"
    longer = model(mel, torch.cat([f0, f0[:, :4]], dim=1))          # f0 longer than the mel: nothing is truncated
    np.testing.assert_allclose(longer.cpu().numpy(), g["wav_long_f0"], atol=2e-5)
    with pytest.raises(ValueError):
        model(mel, f0[:1])
    # f0 shorter than the mel: the reference truncates every stage to the source length (:264-268)
    sdn = {k: v for k, v in sd.items()}
    for prec, tol in (("fp32", 2e-5), ("tc_f16", 5e-4)):
        model.precision = prec
        short = model(mel, f0[:, :11])
        want = og.generator_forward(kind, sdn, hp, g["mel"], f0=g["f0"][:, :11])
        assert short.shape == want.shape and short.shape[-1] < g["wav"].shape[-1]
        assert np.abs(short.cpu().numpy() - want).max() <= tol, (prec, np.abs(short.cpu().numpy() - want).max())
    model.precision = "fp32"
    # f0-aware plumbing (gan_vocoder_inference.py:36, :76-95)
    mels = [torch.from_numpy(g[f"pl_mel{i}"]) for i in range(3)]
    f0s = [torch.from_numpy(g[f"pl_f0{i}"]) for i in range(3)]
    auds = synthesis_audios(model.cfg, model, mels, f0s=f0s, batch_size=2)
    for i, a in enumerate(auds):
        assert a.device.type == "cpu" and a.shape == g[f"pl_audio{i}"].shape
        np.testing.assert_allclose(a.numpy(), g[f"pl_audio{i}"], atol=2e-5)
    out = vocoder_inference(model.cfg, model, mel.cpu(), f0s=f0.cpu(), device=DEV)
    np.testing.assert_allclose(out.numpy(), g["wav"][:, 0], atol=2e-5)


def test_nsfhifigan_exp_config_matches_oracle():
    """The shipped recipe's architecture (egs/vocoder/gan/nsfhifigan/exp_config.json: 768 channels, rates
    8.4.2.2.2 — the first ConvTranspose is 768 -> 384, streaming kernel) at a CPU-checkable length."""
    model = build_model("nsfhifigan", HP_NSF_EXP, 100, seed=3)
    g = torch.Generator().manual_seed(4)
    mel = torch.randn(1, 100, 14, generator=g)
    f0 = torch.rand(1, 14, generator=g) * 400 + 60
    want = og.generator_forward("nsfhifigan", sd_numpy(model), HP_NSF_EXP, mel.numpy(), f0=f0.numpy())
    model = model.to(DEV)
    for prec, tol in (("fp32", 1e-4), ("tc_f16", 1e-3)):
        model.precision = prec
        got = model(mel.to(DEV), f0.to(DEV)).cpu().numpy()
        assert got.shape == (1, 1, 14 * 256)
        assert np.abs(got - want).max() <= tol, (prec, np.abs(got - want).max())


@pytest.mark.parametrize("prec", ["fp32", "tc_f16"])
def test_generator_properties_at_scale(prec):
    """Size-independent properties on a batch the CPU oracle cannot afford:
    batch independence, strided (transposed-view) input == contiguous input,
    time-tiling invariance (a long sequence equals the oracle on a window far
    from the edges is covered above; here: same mel twice in a batch gives
    bit-identical rows), output range of tanh."""
    model = build_model("hifigan", HP_V1, 80, seed=5).to(DEV)
    model.precision = prec
    g = torch.Generator().manual_seed(9)
    mel = torch.randn(4, 80, 512, generator=g).to(DEV)
    mel[3] = mel[1]
    wav = model(mel)
    assert wav.shape == (4, 1, 512 * 256)
    assert torch.isfinite(wav).all() and wav.abs().max() <= 1.0
    assert torch.equal(wav[3], wav[1])                                   # batch independence, deterministic
    single = model(mel[2:3])
    assert torch.equal(single[0], wav[2])                                # B=1 == row of the batch
    tview = mel.transpose(1, 2).contiguous().transpose(1, 2)             # [B,T,n_mel] storage, as vocoder_inference.py:349
    assert not tview.is_contiguous()
    assert torch.equal(model(tview), wav)
    # zero-padding on the right only changes samples near the pad (receptive field), SURVEY Q12
    padded = torch.nn.functional.pad(mel[:1], (0, 64))
    wp = model(padded)[..., : 512 * 256]
    far = (512 - 40) * 256
    assert torch.equal(wp[..., :far], wav[:1, :, :far])


def test_config2_full_size_is_consistent_with_checked_sizes():
    """BASELINE config 2 at its FULL size (HiFi-GAN V1, B=64, 80x1024 -> 64 x 262144 samples, default precision):
    the CPU oracle cannot afford it (40 TFLOP), so it is tied to sizes the oracle does check through
    size-independent properties: every row equals the same utterance run alone (B=1), a row equals its own
    T=256 prefix run away from the right edge (tiling / padding locality), and a 1-utterance, 40-frame window
    in the middle of the batch agrees with the oracle on its interior."""
    hp = HP_V1
    model = build_model("hifigan", hp, 80, seed=1234)
    sd = sd_numpy(model)
    model = model.to(DEV)
    g = torch.Generator().manual_seed(0)
    mel = torch.randn(64, 80, 1024, generator=g).to(DEV)
    wav = model(mel)
    assert wav.shape == (64, 1, 262144) and torch.isfinite(wav).all() and wav.abs().max() <= 1.0
    for b in (0, 17, 63):
        assert torch.equal(model(mel[b:b + 1])[0], wav[b])                        # batch independence at full size
    prefix = model(mel[5:6, :, :256])
    far = (256 - 40) * 256
    assert torch.equal(prefix[..., :far], wav[5:6, :, :far])                      # right-edge locality (receptive field)
    # oracle on a 72-frame window [480, 552) of utterance 33: interior 24 frames are free of edge effects
    lo, hi = 480, 552
    want = og.generator_forward("hifigan", sd, hp, mel[33:34, :, lo:hi].cpu().numpy())
    got = wav[33:34, :, lo * 256: hi * 256].cpu().numpy()
    mid = slice(24 * 256, 48 * 256)
    assert np.abs(got[..., mid] - want[..., mid]).max() <= 1e-3, np.abs(got[..., mid] - want[..., mid]).max()


def test_plumbing_matches_reference_fixture():
    from amphion_b200.vocoders.gan_vocoder_inference import synthesis_audios, vocoder_inference
    kind, hp, g0, sd, model = golden_model("hifigan_rb1")
    model = model.to(DEV)
    model.precision = "fp32"
    g, _ = load_golden("plumbing")
    cfg = model.cfg
    mels = [torch.from_numpy(g[f"mel{i}"]) for i in range(3)]
    auds = synthesis_audios(cfg, model, mels, batch_size=2)
    for i, a in enumerate(auds):
        assert a.device.type == "cpu" and a.dtype == torch.float32
        assert a.shape == g[f"audio{i}"].shape
        np.testing.assert_allclose(a.numpy(), g[f"audio{i}"], atol=2e-5)
    out = vocoder_inference(cfg, model, torch.from_numpy(g["batched_in"]), device=DEV)
    assert out.device.type == "cpu" and out.shape == g["batched_out"].shape
    np.testing.assert_allclose(out.numpy(), g["batched_out"], atol=2e-5)


def test_synthesis_loads_reference_checkpoint_formats(tmp_path):
    from amphion_b200.vocoders.vocoder_inference import synthesis
    kind, hp, g0, sd, model = golden_model("hifigan_rb1")
    cfg = model.cfg
    cfg.model.generator = "hifigan"
    tsd = {("module." + k): torch.from_numpy(v) for k, v in sd.items()}
    p = tmp_path / "legacy.pt"
    torch.save({"generator_state_dict": tsd}, p)
    g, _ = load_golden("plumbing")
    pred = [g[f"mel{i}"].T.copy() for i in range(3)]            # [T, n_mel] as the recipes pass them
    auds = synthesis(cfg, str(p), 3, pred, batch_size=2)
    for i, a in enumerate(auds):
        assert np.abs(a.numpy() - g[f"audio{i}"]).max() < 1e-3  # default precision (tensor cores)


def test_mel_matches_reference_fixture():
    from types import SimpleNamespace as NS
    from amphion_b200 import mel
    g, _ = load_golden("mel")
    cfgp = NS(sample_rate=22050, n_fft=1024, n_mel=80, fmin=0, fmax=8000, win_size=1024, hop_size=256)
    y = torch.from_numpy(g["y"]).to(DEV)
    m = mel.extract_mel_features(y, cfgp)
    assert m.shape == (2, 80, 32) and m.is_cuda
    np.testing.assert_allclose(m.cpu().numpy(), g["extract_mel_features"], atol=2e-4)
    np.testing.assert_allclose(mel.mel_spectrogram_torch(y, cfgp).cpu().numpy(), g["mel_spectrogram_torch"], atol=2e-4)
    np.testing.assert_allclose(mel.extract_linear_features(y, cfgp).cpu().numpy(), g["extract_linear_features"],
                               atol=2e-4, rtol=1e-4)
    assert mel.extract_mel_features(y[:1], cfgp).shape == (80, 32)       # the reference's squeeze(0)
    cfg2 = NS(sample_rate=16000, n_fft=512, n_mel=40, fmin=50, fmax=7600, win_size=400, hop_size=160)
    m2 = mel.extract_mel_features(torch.from_numpy(g["y2"]).to(DEV), cfg2)
    np.testing.assert_allclose(m2.cpu().numpy(), g["extract_mel_features2"], atol=2e-4)


def test_mel_magnitude_is_bit_identical_to_torch_stft_on_device():
    """North-star: 'mel extractor bit-pattern-equal given identical FFT backend'.
    Same fp32 window multiply, same cuFFT, same |.| arithmetic as utils/mel.py:145-166
    executed by torch on this GPU."""
    from types import SimpleNamespace as NS
    from amphion_b200 import mel
    cfgp = NS(sample_rate=22050, n_fft=1024, n_mel=80, fmin=0, fmax=8000, win_size=1024, hop_size=256)
    g = torch.Generator().manual_seed(3)
    y = ((torch.rand(4, 22050, generator=g) * 2 - 1) * 0.9).to(DEV)
    win = torch.hann_window(1024).to(DEV)
    yp = torch.nn.functional.pad(y.unsqueeze(1), (384, 384), mode="reflect").squeeze(1)
    spec = torch.stft(yp, 1024, hop_length=256, win_length=1024, window=win, center=False, pad_mode="reflect",
                      normalized=False, onesided=True, return_complex=True)
    ref = torch.sqrt(torch.view_as_real(spec).pow(2).sum(-1) + 1e-9)
    got = mel.extract_linear_features(y, cfgp)
    assert got.shape == ref.shape
    nbad = int((got != ref).sum())
    assert nbad == 0, f"{nbad} of {ref.numel()} magnitudes differ, max abs {float((got - ref).abs().max())}"
    basis = mel.librosa_mel_fn(22050, 1024, 80, 0, 8000).to(DEV)
    torch.backends.cuda.matmul.allow_tf32 = False
    ref_mel = torch.log(torch.clamp(torch.matmul(basis, ref), min=1e-5))
    assert (mel.extract_mel_features(y, cfgp) - ref_mel).abs().max() <= 1e-5   # cuBLAS summation order only


def test_tacotron_stft_matches_reference_fixture():
    from amphion_b200.stft import TacotronSTFT
    g, _ = load_golden("mel")
    taco = TacotronSTFT(1024, 256, 1024, 80, 22050, 0, 8000)
    np.testing.assert_allclose(taco.mel_basis.numpy(), g["taco_mel_basis"], atol=1e-7)
    m, e = taco.mel_spectrogram(torch.from_numpy(g["y"]))                # CPU in, CPU out, like the reference
    assert m.device.type == "cpu" and m.shape == (2, 80, 33) and e.shape == (2, 33)
    np.testing.assert_allclose(m.numpy(), g["taco_mel"], atol=3e-4)
    np.testing.assert_allclose(e.numpy(), g["taco_energy"], rtol=2e-4)
    with pytest.raises(AssertionError):
        taco.mel_spectrogram(torch.from_numpy(g["y"]) * 2)


def test_mel_full_size_properties():
    """BASELINE config 4 shape: 64 x 10 s @ 22.05 kHz -> mel [64, 80, 862]."""
    from amphion_b200.stft import TacotronSTFT
    g = torch.Generator().manual_seed(0)
    y = (torch.rand(64, 220500, generator=g) * 2 - 1) * 0.9
    taco = TacotronSTFT(1024, 256, 1024, 80, 22050, 0, 8000)
    m, e = taco.mel_spectrogram(y)
    assert m.shape == (64, 80, 862) and e.shape == (64, 862)
    assert torch.isfinite(m).all() and m.min() >= np.log(1e-5) - 1e-6
    mo, eo = om.tacotron_mel(y[:1, :8192].numpy(), taco.mel_basis.numpy(), 1024, 256, 1024)
    # frames whose support lies inside the first 8192-512 samples are identical to the short run
    np.testing.assert_allclose(m[0, :, :28].numpy(), mo[0, :, :28], atol=3e-4)
    m2, _ = taco.mel_spectrogram(y[5:6])
    # batch independence (cuFFT may pick a different plan for another batch count: not bit-equal)
    torch.testing.assert_close(m2[0], m[5], atol=2e-5, rtol=0)


def test_save_audio_matches_oracle(tmp_path):
    """utils/io.py:49-76 on the device: bit-exact against the oracle (float stage pinned by the reference
    fixture, quantiser restated — see oracle/io.py)."""
    import wave
    from oracle import io as oio
    from amphion_b200.io import save_audio, save_audios, waveform_to_pcm16
    g, _ = load_golden("save_audio")
    for ts in (0, 1):
        for sil in (0, 1):
            p = tmp_path / f"a{ts}{sil}.wav"
            save_audio(p, g["w"], 16000, add_silence=bool(sil), turn_up=bool(ts))
            with wave.open(str(p)) as f:
                assert (f.getnchannels(), f.getsampwidth(), f.getframerate()) == (1, 2, 16000)
                got = np.frombuffer(f.readframes(f.getnframes()), "<i2")
            want = oio.pcm16(g[f"float_turnup{ts}_silence{sil}"])[0]
            np.testing.assert_array_equal(got, want)
    # batch with ragged lengths (down to one sample), odd sizes, a constant row and clipping
    gen = torch.Generator().manual_seed(3)
    wav = torch.randn(5, 4097, generator=gen) * 0.7
    wav[4] = 0.25
    lens = [4097, 1, 1000, 333, 4096]
    pcm = waveform_to_pcm16(wav.to(DEV), lens, silence=7, turn_up=True, volume_peak=0.9).cpu().numpy()
    assert pcm.shape == (5, 4097 + 14 + 1)
    for b, n in enumerate(lens):
        want = oio.pcm16(oio.save_audio_float(wav[b, :n].numpy(), 140, add_silence=True, turn_up=True))[0]
        np.testing.assert_array_equal(pcm[b, : n + 14], want)
        assert not pcm[b, n + 14:].any()
    plain = waveform_to_pcm16((wav * 3).to(DEV)).cpu().numpy()
    np.testing.assert_array_equal(plain[:, :4097], oio.pcm16((wav * 3).numpy()))
    paths = [tmp_path / f"b{i}.wav" for i in range(5)]
    save_audios(paths, wav.to(DEV), 22050, lengths=lens, add_silence=True)
    with wave.open(str(paths[2])) as f:
        assert f.getnframes() == 1000 + 2 * (22050 // 20)
    # full-size property: a config-2 sized batch quantises to the same values as the oracle's formula
    big = torch.rand(8, 262144, generator=gen) * 2 - 1
    got = waveform_to_pcm16(big.to(DEV)).cpu().numpy()
    np.testing.assert_array_equal(got, oio.pcm16(big.numpy()))


@pytest.mark.parametrize("tag", sorted(GOLDEN_VITS))
def test_hifigan_vits_matches_reference_fixture(tag):
    """HiFiGAN_vits.forward(x, g) (hifigan.py:427-445), the VITS waveform decoder."""
    from amphion_b200.vocoders import HiFiGAN_vits
    g, sd = load_golden_vits(tag)
    model = HiFiGAN_vits(**GOLDEN_VITS[tag])
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    model = model.to(DEV).eval()
    x = torch.from_numpy(g["x"]).to(DEV)
    for prec, tol in (("fp32", 2e-5), ("tc_f16", 5e-4)):
        model.precision = prec
        got = model(x).cpu().numpy()
        assert got.shape == g["wav"].shape
        assert np.abs(got - g["wav"]).max() <= tol, (prec, np.abs(got - g["wav"]).max())
        if "g" in g:
            cond = torch.from_numpy(g["g"]).to(DEV)
            got = model(x, g=cond).cpu().numpy()
            assert np.abs(got - g["wav_g"]).max() <= tol, (prec, np.abs(got - g["wav_g"]).max())
            got2 = model(x, g=cond[:, :, 0]).cpu().numpy()            # [B, gin] is accepted too
            np.testing.assert_array_equal(got, got2)
    if "g" not in g:
        with pytest.raises(AttributeError):                            # the reference has no `cond` module either
            model(x, g=torch.zeros(x.shape[0], 4, 1, device=DEV))


def test_hifigan_vits_decoder_size_matches_oracle():
    """VITS decoder geometry (config/vits.json: inter_channels 192, 512 ch, rates 8.8.2.2, gin 256), CPU-checkable."""
    from amphion_b200.vocoders import HiFiGAN_vits
    args = dict(initial_channel=192, resblock="1", resblock_kernel_sizes=[3, 7, 11], resblock_dilation_sizes=[[1, 3, 5]] * 3,
                upsample_rates=[8, 8, 2, 2], upsample_initial_channel=512, upsample_kernel_sizes=[16, 16, 4, 4],
                gin_channels=256)
    torch.manual_seed(6)
    model = HiFiGAN_vits(**args).eval()
    gen = torch.Generator().manual_seed(7)
    x, cond = torch.randn(2, 192, 21, generator=gen), torch.randn(2, 256, 1, generator=gen)
    want = og.hifigan_vits_forward(sd_numpy(model), args, x.numpy(), cond.numpy())
    model = model.to(DEV)
    got = model(x.to(DEV), g=cond.to(DEV)).cpu().numpy()
    assert got.shape == (2, 1, 21 * 256)
    assert np.abs(got - want).max() <= 1e-3, np.abs(got - want).max()


# ---- persistent fused ResBlock kernel (ab_kernels_rb.cu): execution-plan modes -------------------------------
def _fusion_outputs(model, mel, modes):
    outs = {}
    for mode in modes:
        model.set_option("resblock_fusion", mode)
        outs[mode] = model(mel)
    model.set_option("resblock_fusion", 2)
    return outs


@pytest.mark.parametrize("B,T", [(2, 40), (3, 150), (1, 37)])
def test_resblock_fusion_modes_agree_on_v1(B, T):
    """HiFi-GAN V1 (stages of 256/128/64/32 channels).  The persistent kernel one pair per launch (1), the
    cost-model plan (2) and whole-block fusion with halo recompute (3) run the same arithmetic in the same order
    and must agree to the last bit (recomputed halo rows == the rows another tile owns).  The per-pair kernel (0)
    adds the residual after the convolution instead of accumulating on top of it: fp32 summation order only.
    T=150 gives several tiles per sequence and an odd tile count, T=37 a ragged single tile."""
    model = build_model("hifigan", HP_V1, 80, seed=4321).to(DEV)
    mel = torch.randn(B, 80, T, generator=torch.Generator().manual_seed(T)).to(DEV)
    outs = _fusion_outputs(model, mel, (0, 1, 2, 3, 4))
    for mode in (1, 2, 3, 4):
        assert torch.isfinite(outs[mode]).all()
    assert torch.equal(outs[1], outs[3])
    # the per-pair kernel (0) adds the residual after the convolution; plans with the TMEM-resident residual (2, 4)
    # accumulate every conv2 of a block on top of x without intermediate rounding of x_p: fp32 summation order only
    for mode in (0, 2, 4):
        diff = (outs[mode] - outs[3]).abs().max().item()
        assert diff <= 3e-5, (mode, diff)


@pytest.mark.parametrize("name", ["hifigan_rb1", "hifigan_rb2"])
@pytest.mark.parametrize("mode", [0, 1, 3, 4])
def test_resblock_fusion_modes_match_reference_fixture(name, mode):
    """ResBlock1 and ResBlock2 (single conv per residual step) fixtures through every plan, incl. bf16."""
    kind, hp, g, sd, model = golden_model(name)
    model = model.to(DEV)
    model.set_option("resblock_fusion", mode)
    for prec, tol in (("tc_f16", 5e-4), ("tc_bf16", 4e-3)):
        model.precision = prec
        wav = model(torch.from_numpy(g["mel"]).to(DEV)).cpu().numpy()
        assert np.abs(wav - g["wav"]).max() <= tol, (prec, mode, np.abs(wav - g["wav"]).max())


def test_resblock_fusion_odd_channels_and_wide_kernel():
    """Channel counts that are not multiples of 32 (K chunk of 16 left over, generic issue path) and a kernel /
    dilation set whose fused halo does not fit (falls back to one pair per launch), against the CPU oracle."""
    hp = dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4], upsample_initial_channel=96,
              resblock_kernel_sizes=[3, 13], resblock_dilation_sizes=[[1, 2, 4], [1, 7, 9]])
    model, mel, want = _full_size_case("hifigan", hp, 20, 2, 300, seed=11)
    for mode in (0, 1, 3, 4):
        model.set_option("resblock_fusion", mode)
        got = model(mel.to(DEV)).cpu().numpy()
        assert np.abs(got - want).max() <= 1e-3, (mode, np.abs(got - want).max())


# ---- parity where 16-bit operands can bite (VERDICT r1 #4) -------------------------------------------------------
def _trained_like(model, seed):
    """Give a random-init model the dynamic range of a trained checkpoint without changing its fp32 function much:
    every (c1, c2) pair of a ResBlock gets c1 scaled by s and c2 by 1/s, s = 10^U(-1.5, 1.5) (leaky_relu is
    positively homogeneous, so only the intermediate's magnitude moves: 0.03x .. 30x), the weight-norm gains carry
    the scale (weight_g spanning three decades), and ~1 % of the direction entries are 10x outliers."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, mod in model.named_modules():
            if hasattr(mod, "convs1") and hasattr(mod, "convs2"):
                for c1, c2 in zip(mod.convs1, mod.convs2):
                    s = float(10.0 ** (torch.rand((), generator=g) * 3.0 - 1.5))
                    c1.weight_g.mul_(s)
                    c1.bias.mul_(s)
                    c2.weight_g.div_(s)
        for n, p in model.named_parameters():
            if n.endswith("weight_v"):
                mask = torch.rand(p.shape, generator=g) < 0.01
                p[mask] *= 10.0
    if hasattr(model, "invalidate"):
        model.invalidate()
    return model


@pytest.mark.parametrize("kind,hp,n_mel,B,T,seed", [("hifigan", HP_V1, 80, 2, 40, 21), ("bigvgan", HP_BIGVGAN_BASE, 100, 1, 24, 22)])
@pytest.mark.parametrize("stress", ["logmel_input", "trained_like_weights", "both"])
def test_tensor_core_path_holds_1e3_under_trained_like_dynamic_range(kind, hp, n_mel, B, T, seed, stress):
    """Full-width V1 / BigVGAN-base on the default tensor-core path (fp16 operands, fp32 accumulate) against the
    fp32 CPU oracle with (i) mel ~ U(-11.5, 2), the log-mel range of utils/mel.py:11 (SURVEY 8d), and (ii) weight-norm
    gains spanning three decades plus outlier weights.  Bar: 1e-3 max-abs (north star)."""
    model = build_model(kind, hp, n_mel, seed=seed)
    if kind == "bigvgan":
        randomize_snake(model, seed + 1, hp["snake_logscale"])
    if stress in ("trained_like_weights", "both"):
        _trained_like(model, seed + 2)
    gm = torch.Generator().manual_seed(seed + 3)
    mel = torch.rand(B, n_mel, T, generator=gm) * 13.5 - 11.5 if stress != "trained_like_weights" else torch.randn(B, n_mel, T, generator=gm)
    want = og.generator_forward(kind, sd_numpy(model), hp, mel.numpy())
    model = model.to(DEV)
    model.precision = "tc_f16"
    got = model(mel.to(DEV)).cpu().numpy()
    assert np.isfinite(got).all()
    err = np.abs(got - want).max()
    print(f"max|tc_f16 - oracle| {kind} {stress}: {err:.3e} (|wav| max {np.abs(want).max():.3f})")
    assert err <= 1e-3, (stress, err)


def _full_size_consistency(kind, hp, n_mel, B, T, seed, win_lo):
    """Full BASELINE size on the default precision, tied to oracle-checked sizes through size-independent
    properties (the CPU oracle cannot afford the full batch): batch independence, right-edge locality and an
    oracle-checked interior window."""
    hop = int(np.prod(hp["upsample_rates"]))
    model = build_model(kind, hp, n_mel, seed=seed)
    if kind == "bigvgan":
        randomize_snake(model, seed + 1, hp["snake_logscale"])
    sd = sd_numpy(model)
    model = model.to(DEV)
    mel = torch.randn(B, n_mel, T, generator=torch.Generator().manual_seed(seed + 2)).to(DEV)
    wav = model(mel)
    assert wav.shape == (B, 1, T * hop) and torch.isfinite(wav).all() and wav.abs().max() <= 1.0
    for b in (0, B - 1):
        assert torch.equal(model(mel[b:b + 1])[0], wav[b])                        # batch independence
    prefix = model(mel[1:2, :, :256])
    far = (256 - 48) * hop
    assert torch.equal(prefix[..., :far], wav[1:2, :, :far])                      # right-edge locality
    lo, hi = win_lo, win_lo + 72                                                  # 72-frame window, interior 24 frames
    want = og.generator_forward(kind, sd, hp, mel[B // 2: B // 2 + 1, :, lo:hi].cpu().numpy())
    got = wav[B // 2: B // 2 + 1, :, lo * hop: hi * hop].cpu().numpy()
    mid = slice(24 * hop, 48 * hop)
    err = np.abs(got[..., mid] - want[..., mid]).max()
    print(f"full-size {kind} B={B} T={T}: interior max|cuda - oracle| = {err:.3e}")
    assert err <= 1e-3, err


def test_config3_full_size_is_consistent_with_checked_sizes():
    """BASELINE config 3: BigVGAN-base 24 kHz, batch 32, 100 x 1024 mel."""
    _full_size_consistency("bigvgan", HP_BIGVGAN_BASE, 100, 32, 1024, seed=303, win_lo=480)


def test_config5_shard_full_size_is_consistent_with_checked_sizes():
    """BASELINE config 5, one GPU's shard: BigVGAN-large 24 kHz (1536 ch, six stages), batch 32, 100 x 2048 mel."""
    hp = dict(resblock="1", upsample_rates=[4, 4, 2, 2, 2, 2], upsample_kernel_sizes=[8, 8, 4, 4, 4, 4],
              upsample_initial_channel=1536, resblock_kernel_sizes=[3, 7, 11],
              resblock_dilation_sizes=[[1, 3, 5]] * 3, activation="snakebeta", snake_logscale=True)
    _full_size_consistency("bigvgan", hp, 100, 32, 2048, seed=505, win_lo=1000)


def test_fused_mel_kernel_matches_the_cufft_pipeline_and_the_oracle():
    """ab_mel_forward_fused (frame -> window -> own 1024-point FFT -> |.| -> mel -> log in one kernel): log-mel
    within 1e-5 of the cuFFT pipeline (whose spectrum is bit-identical to torch.stft), energy within 2e-6 relative,
    on ragged lengths (partial frame groups, reflect padding at both ends), the three parameterisations of
    SURVEY Q8 (eps 0 / 1e-9 / 1e-6; pad n_fft/2 and (n_fft-hop)/2; win < n_fft) and 24 kHz / 100 mels."""
    from amphion_b200 import mel
    cases = [  # B, T, hop, win, n_mel, sr, fmax, pad, eps
        (3, 22050, 256, 1024, 80, 22050, 8000, 512, 0.0),        # TacotronSTFT (config 4 parameters)
        (2, 9000, 256, 1024, 80, 22050, 8000, 384, 1e-9),        # extract_mel_features
        (1, 4097, 240, 960, 100, 24000, 12000, 392, 1e-6),       # mel_spectrogram_torch, BigVGAN 24 kHz, win < n_fft
        (5, 1300, 256, 1024, 128, 22050, None, 512, 0.0),        # fewer frames than a group of 8, 128 mels
    ]
    for B, T, hop, win, n_mel, sr, fmax, pad, eps in cases:
        g = torch.Generator().manual_seed(T)
        y = ((torch.rand(B, T, generator=g) * 2 - 1) * 0.9).to(DEV)
        window = torch.hann_window(win).to(DEV)
        basis = mel.librosa_mel_fn(sr, 1024, n_mel, 0, fmax).to(DEV)
        _, m0, e0 = mel.native_stft_mel(y, 1024, hop, win, window, basis, pad, eps, want_energy=True)
        _, m1, e1 = mel.native_stft_mel(y, 1024, hop, win, window, basis, pad, eps, want_energy=True, fused=True)
        assert m1.shape == m0.shape and e1.shape == e0.shape
        assert (m1 - m0).abs().max() <= 1e-5, ((B, T), float((m1 - m0).abs().max()))
        assert ((e1 - e0).abs() / e0.abs().clamp_min(1e-3)).max() <= 2e-6
    want, _ = om.tacotron_mel(y[:1, :1300].cpu().numpy()[:, :1300], basis.cpu().numpy(), 1024, 256, 1024)
    np.testing.assert_allclose(m1[:1].cpu().numpy(), want, atol=3e-4)      # CPU oracle (conv-DFT restatement)


def test_bucketed_synthesis_and_generate_to_files(tmp_path):
    """SURVEY 8(f) rank 1: length bucketing (opt-in) and the fused generate + trim + PCM16 + save loop.  Every
    utterance's samples away from its last receptive field equal the unbucketed result; an utterance grouped with
    the same neighbours is bit-identical; the files hold exactly the PCM16 of the returned audio."""
    import wave
    from oracle import io as oio
    from amphion_b200.vocoders import synthesis_audios, synthesize_to_files
    kind, hp, g0, sd, model = golden_model("hifigan_rb1")
    model = model.to(DEV)
    cfg = model.cfg
    cfg.preprocess.sample_rate = 16000
    hop = cfg.preprocess.hop_size
    gen = torch.Generator().manual_seed(9)
    lens = [71, 49, 80, 52, 73, 50]
    mels = [torch.randn(g0["mel"].shape[1], n, generator=gen) for n in lens]
    plain = synthesis_audios(cfg, model, mels, batch_size=2)
    buck = synthesis_audios(cfg, model, mels, batch_size=2, bucket=True)
    assert [a.shape[0] for a in buck] == [n * hop for n in lens]                 # input order, trimmed lengths
    rf = 32 * hop      # > receptive field (rates [4, 2], k = 11, d = 1,3,5: 60 samples per block = 15 + 7.5 frames, + conv_pre 3)
    for a, b, n in zip(plain, buck, lens):
        keep = max(n * hop - rf, 0)
        assert torch.equal(a[:keep], b[:keep])
    paths = [str(tmp_path / f"u{i}.wav") for i in range(len(mels))]
    synthesize_to_files(cfg, model, mels, paths, batch_size=2, bucket=True, turn_up=True)
    for p, a in zip(paths, buck):
        with wave.open(p) as f:
            assert (f.getnchannels(), f.getsampwidth(), f.getframerate()) == (1, 2, 16000)
            got = np.frombuffer(f.readframes(f.getnframes()), "<i2")
        want = oio.pcm16(oio.save_audio_float(a.numpy(), 16000, turn_up=True))[0]
        assert got.shape == want.shape and np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= 1


def test_nsfhifigan_odd_source_stride_truncates_like_the_reference():
    """rates [4, 3, 3]: noise_convs with an odd stride give a source one sample short, so the reference cuts the
    stage (nsfhifigan.py:264-268) and everything after it; CUDA path against the CPU oracle's restatement."""
    hp = dict(resblock="1", harmonic_num=8, upsample_rates=[4, 3, 3], upsample_kernel_sizes=[8, 5, 5],
              upsample_initial_channel=128, resblock_kernel_sizes=[3, 7], resblock_dilation_sizes=[[1, 3, 5]] * 2)
    model = build_model("nsfhifigan", hp, 20, seed=8)
    gm = torch.Generator().manual_seed(2)
    mel, f0 = torch.randn(2, 20, 30, generator=gm), torch.rand(2, 30, generator=gm) * 300 + 80
    want = og.generator_forward("nsfhifigan", sd_numpy(model), hp, mel.numpy(), f0=f0.numpy())
    model = model.to(DEV)
    for prec, tol in (("fp32", 5e-5), ("tc_f16", 1e-3)):
        model.precision = prec
        got = model(mel.to(DEV), f0.to(DEV)).cpu().numpy()
        assert got.shape == want.shape and got.shape[-1] < 30 * 36
        assert np.abs(got - want).max() <= tol, (prec, np.abs(got - want).max())


@pytest.mark.parametrize("n_in,tag", [(256, "JETS: HiFiGAN(hifi_cfg) with n_mel = attention_dim (models/tts/jets/jets.py:454-458)"),
                                      (192, "VITS-SVC: self.dec = HiFiGAN(temp_cfg) with n_mel = inter_channels (models/svc/vits/vits.py:131-139)")])
def test_in_model_generators_of_jets_and_vits_svc_are_the_registry_class(n_in, tag):
    """The end-to-end TTS / SVC models build their waveform decoder from the vocoder registry class with the
    model's hidden width as `n_mel` — the same native class, fed a [B, hidden, T] latent instead of a mel."""
    hp = dict(HP_V1, upsample_initial_channel=256)
    model, z, want = _full_size_case("hifigan", hp, n_in, 2, 33, seed=n_in)
    for prec, tol in (("fp32", 5e-5), ("tc_f16", 1e-3)):
        model.precision = prec
        got = model(z.to(DEV)).cpu().numpy()
        assert got.shape == (2, 1, 33 * 256)
        assert np.abs(got - want).max() <= tol, (tag, prec, np.abs(got - want).max())


@pytest.mark.parametrize("T", [1, 3])
def test_v1_shorter_than_every_halo(T):
    """A mel of one or three frames: every tile of every stage is mostly zero padding (the fused kernel's rows are
    nearly all outside [0, T)); all plans against the CPU oracle."""
    model, mel, want = _full_size_case("hifigan", HP_V1, 80, 2, T, seed=60 + T)
    for mode in (0, 2, 3):
        model.set_option("resblock_fusion", mode)
        got = model(mel.to(DEV)).cpu().numpy()
        assert got.shape == want.shape
        assert np.abs(got - want).max() <= 1e-3, (mode, np.abs(got - want).max())


# ---------------------------------------------------------------------------
# (f)4: the mel front end under autograd (the trainers' mel loss, gan_vocoder_trainer.py:368-396)
# ---------------------------------------------------------------------------
_MEL_GRAD_CFG = {"a": dict(sample_rate=22050, n_fft=1024, n_mel=80, fmin=0, fmax=8000, win_size=1024, hop_size=256),
                 "b": dict(sample_rate=16000, n_fft=512, n_mel=40, fmin=50, fmax=7600, win_size=400, hop_size=160)}


@pytest.mark.parametrize("tag", ["a", "b"])
def test_mel_loss_gradient_matches_reference_autograd(tag):
    """L1(mel(y_gt), mel(y_pred)) * 45 differentiated through the native backward equals what torch autograd gave
    through the reference's extract_mel_features (tests/golden/mel_grad.npz), and a random cotangent likewise."""
    from types import SimpleNamespace as NS
    from amphion_b200 import mel
    g, _ = load_golden("mel_grad")
    cfgp = NS(**_MEL_GRAD_CFG[tag])
    y_gt = torch.from_numpy(g[tag + "_y_gt"]).to(DEV)
    y_pred = torch.from_numpy(g[tag + "_y_pred"]).to(DEV).requires_grad_(True)
    mel_gt = mel.extract_mel_features(y_gt, cfgp)
    mel_pred = mel.extract_mel_features(y_pred, cfgp)
    assert mel_pred.requires_grad and not mel_gt.requires_grad
    loss = torch.nn.L1Loss(reduction="mean")(mel_gt, mel_pred) * 45
    np.testing.assert_allclose(loss.item(), g[tag + "_loss"], rtol=1e-4)
    (gl,) = torch.autograd.grad(loss, y_pred, retain_graph=True)
    want = g[tag + "_grad_loss"]
    # sign(pred - gt) may flip where the two mels agree to the last bits: compare in the aggregate and pointwise loosely
    err = np.abs(gl.cpu().numpy() - want)
    assert err.max() <= 2e-2 * np.abs(want).max() and err.mean() <= 1e-4 * np.abs(want).max(), (err.max(), err.mean())
    (gc,) = torch.autograd.grad(mel_pred, y_pred, torch.from_numpy(g[tag + "_cot"]).to(DEV))
    want = g[tag + "_grad_cot"]
    assert np.abs(gc.cpu().numpy() - want).max() <= 5e-4 * np.abs(want).max()
    silent = slice(y_pred.shape[1] // 3 + cfgp.n_fft, y_pred.shape[1] // 3 + 2 * cfgp.n_fft)
    assert np.abs(gc[0, silent].cpu().numpy()).max() <= 1e-3 * np.abs(want).max()      # frames below the log clamp


def test_mel_gradient_odd_lengths_and_the_1e6_variant_match_the_oracle():
    """Edge geometry (length not a multiple of the hop, one frame only) and mel_spectrogram_torch's eps = 1e-6."""
    from types import SimpleNamespace as NS
    from amphion_b200 import mel
    from oracle import mel as om
    cfgp = NS(**_MEL_GRAD_CFG["a"])
    basis = om.slaney_mel_filterbank(22050, 1024, 80, 0, 8000)
    rng = np.random.default_rng(5)
    for T, eps, fn in ((2999, 1e-9, mel.extract_mel_features), (1024 - 256 + 3, 1e-9, mel.extract_mel_features),
                       (4100, 1e-6, mel.mel_spectrogram_torch)):
        y = ((rng.random((2, T)) * 2 - 1) * 0.7).astype(np.float32)
        yt = torch.from_numpy(y).to(DEV).requires_grad_(True)
        m = fn(yt, cfgp)
        cot = rng.standard_normal(tuple(m.shape)).astype(np.float32)
        (gy,) = torch.autograd.grad(m, yt, torch.from_numpy(cot).to(DEV))
        want = om.extract_mel_features_vjp(y, basis, cot, 1024, 256, 1024, eps=eps)
        assert gy.shape == yt.shape
        assert np.abs(gy.cpu().numpy() - want).max() <= 5e-4 * np.abs(want).max(), (T, eps)
    # no graph, no gradient: the inference path is untouched
    with torch.no_grad():
        assert not mel.extract_mel_features(yt, cfgp).requires_grad


def test_feature_directory_round_trip(tmp_path):
    """(f)4 data format: wav -> native mel -> <processed_dir>/<dataset>/mels/<uid>.npy (reference layout, float32
    [n_mel, T]) -> VocoderDataset -> batched synthesis to <uid>.wav.  The stored mel equals the oracle's, and the
    files equal those written from the in-memory mels."""
    import wave
    from types import SimpleNamespace as NS
    from amphion_b200 import features
    from amphion_b200.vocoders import synthesize_to_files
    from oracle import mel as om
    kind, hp, g0, sd, model = golden_model("hifigan_rb1")
    model = model.to(DEV)
    n_mel = g0["mel"].shape[1]
    root = str(tmp_path / "processed_data")
    pre = model.cfg.preprocess
    pre.sample_rate, pre.n_fft, pre.win_size, pre.fmin, pre.fmax = 16000, 256, 256, 0, 8000
    pre.processed_dir, pre.train_file, pre.valid_file, pre.mel_dir = root, "train.json", "valid.json", "mels"
    pre.use_mel, pre.use_frame_pitch, pre.extract_mel = True, False, True
    pre.extract_amplitude_phase = True
    hop = pre.hop_size
    rng = np.random.default_rng(3)
    utts = [{"Dataset": "toy", "Uid": f"utt{i:02d}"} for i in range(5)]
    basis = om.slaney_mel_filterbank(16000, 256, n_mel, 0, 8000)
    mels = []
    for u, n in zip(utts, (40, 57, 33, 64, 48)):
        wav = ((rng.random(n * hop) * 2 - 1) * 0.6).astype(np.float32)
        m = features.extract_utt_mel_features(os.path.join(root, "toy"), model.cfg, u, torch.from_numpy(wav).to(DEV))
        stored = np.load(os.path.join(root, "toy", "mels", u["Uid"] + ".npy"))
        assert stored.dtype == np.float32 and stored.shape == (n_mel, n)
        np.testing.assert_array_equal(stored, m.cpu().numpy())
        np.testing.assert_allclose(stored, om.extract_mel_features(wav[None], basis, 256, hop, 256)[0], atol=2e-4)
        mels.append(torch.from_numpy(stored))
        la = np.load(os.path.join(root, "toy", "log_amplitudes", u["Uid"] + ".npy"))      # APNet features, squeezed
        re_, im_ = (np.load(os.path.join(root, "toy", d, u["Uid"] + ".npy")) for d in ("reals", "imaginarys"))
        assert la.shape == re_.shape == (129, n) and os.path.exists(os.path.join(root, "toy", "phases", u["Uid"] + ".npy"))
        np.testing.assert_allclose(la, np.log(np.sqrt(re_ ** 2 + im_ ** 2) + 1e-5), atol=1e-5)
    pre.extract_amplitude_phase = False          # synthesis below is the mel -> wav path of this (HiFi-GAN) model
    features.write_metadata(root, "toy", utts, "valid.json")
    ds = features.VocoderDataset(model.cfg, "toy", is_valid=True)
    out = features.synthesize_dataset(model.cfg, model, ds, str(tmp_path / "out"), batch_size=2)
    ref_paths = [str(tmp_path / f"ref{i}.wav") for i in range(len(mels))]
    synthesize_to_files(model.cfg, model, mels, ref_paths, batch_size=2, bucket=True)
    for p, q, u in zip(out, ref_paths, utts):
        assert os.path.basename(p) == u["Uid"] + ".wav"
        with wave.open(p) as f, wave.open(q) as h:
            assert f.getframerate() == 16000 and f.getnframes() == h.getnframes()
            assert f.readframes(f.getnframes()) == h.readframes(h.getnframes())


# ---------------------------------------------------------------------------
# (f)4: iSTFT-head generator (APNet, apnet.py:283-399)
# ---------------------------------------------------------------------------
def _apnet_model(hp, pre, sd=None, seed=None):
    from types import SimpleNamespace as NS
    from amphion_b200.vocoders import APNet
    if seed is not None:
        torch.manual_seed(seed)
    m = APNet(NS(preprocess=NS(**pre), model=NS(generator="apnet", apnet=NS(**hp))))
    if sd is not None:
        m.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()}, strict=True)
    return m.eval().to(DEV)


def _phase_err(a, b):
    d = np.abs(a - b)
    return np.minimum(d, 2 * np.pi - d)


@pytest.mark.parametrize("precision,tol", [("fp32", 5e-5), ("tc_f16", 2e-3)])
def test_apnet_matches_reference_fixture(precision, tol):
    """fp32 arithmetic reproduces the reference to 5e-5.  With 16-bit conv operands the log-amplitude and the (R, I)
    pair carry ~1e-3 of rounding, which exp() and atan2 turn into ~1e-3 RELATIVE error of the spectrum: the audio
    bound is 2e-3 (measured 1e-3-class), stated here rather than hidden."""
    from conftest import GOLDEN_APNET, load_golden_apnet
    from amphion_b200.vocoders.gan_vocoder_inference import vocoder_inference
    hp, pre = GOLDEN_APNET
    g, sd = load_golden_apnet()
    model = _apnet_model(hp, pre, sd)
    model.precision = precision
    logamp, pha, rea, imag, audio = model(torch.from_numpy(g["mel"]).to(DEV))
    assert audio.shape == (2, 1, 23 * pre["hop_size"]) and audio.is_cuda
    errs = dict(logamp=np.abs(logamp.cpu().numpy() - g["logamp"]).max(),
                audio=np.abs(audio.cpu().numpy() - g["audio"]).max())
    amp = np.exp(g["logamp"])
    errs["rea"] = (np.abs(rea.cpu().numpy() - g["rea"]) / (1 + amp)).max()
    errs["imag"] = (np.abs(imag.cpu().numpy() - g["imag"]) / (1 + amp)).max()
    print("apnet fixture", precision, {k: float(v) for k, v in errs.items()})
    assert errs["logamp"] <= tol * 3, errs
    assert errs["rea"] <= tol * 3 and errs["imag"] <= tol * 3, errs
    # the phase is ill-conditioned where |R + iI| is small: compare it weighted by that modulus (what reaches the audio)
    if precision == "fp32":
        assert _phase_err(pha.cpu().numpy(), g["pha"]).max() <= 2e-2
    assert np.abs(audio.cpu().numpy() - g["audio"]).max() <= tol
    from types import SimpleNamespace as NS
    out = vocoder_inference(model.cfg, model, torch.from_numpy(g["mel"]))
    assert not out.is_cuda and np.abs(out.numpy() - g["inference"]).max() <= tol


def test_istft_module_matches_the_oracle():
    """ISTFT "same" (apnet.py:46-104) on a random complex spectrum, two geometries."""
    from amphion_b200.vocoders.apnet import ISTFT
    from oracle import generator as og
    rng = np.random.default_rng(11)
    for n_fft, hop, B, T in ((64, 16, 3, 9), (1024, 256, 2, 37), (256, 64, 1, 1)):
        re = rng.standard_normal((B, n_fft // 2 + 1, T)).astype(np.float32)
        im = rng.standard_normal((B, n_fft // 2 + 1, T)).astype(np.float32)
        spec = torch.complex(torch.from_numpy(re), torch.from_numpy(im)).to(DEV)
        got = ISTFT(n_fft, hop, n_fft)(spec, torch.hann_window(n_fft))
        want = og.istft_same(re, im, n_fft, hop, n_fft)
        assert got.shape == want.shape == (B, T * hop)
        assert np.abs(got.cpu().numpy() - want).max() <= 2e-5 * max(1.0, np.abs(want).max())


def test_apnet_recipe_width_matches_the_oracle():
    """egs/vocoder/gan/apnet/exp_config.json: 512-channel streams, n_fft 1024, hop 256, 80 mels (the wide ResBlocks run
    on the streaming tensor-core kernel).  Random weights with the output convolutions scaled to a generic phase."""
    from helpers import sd_numpy
    from oracle import generator as og
    hp = dict(ASP_channel=512, ASP_resblock_kernel_sizes=[3, 7, 11], ASP_resblock_dilation_sizes=[[1, 3, 5]] * 3,
              ASP_input_conv_kernel_size=7, ASP_output_conv_kernel_size=7,
              PSP_channel=512, PSP_resblock_kernel_sizes=[3, 7, 11], PSP_resblock_dilation_sizes=[[1, 3, 5]] * 3,
              PSP_input_conv_kernel_size=7, PSP_output_R_conv_kernel_size=7, PSP_output_I_conv_kernel_size=7)
    pre = dict(n_mel=80, n_fft=1024, hop_size=256, win_size=1024, extract_amplitude_phase=True, sample_rate=22050)
    model = _apnet_model(hp, pre, seed=5)
    with torch.no_grad():
        for conv, gain in ((model.ASP_output_conv, 3.0), (model.PSP_output_R_conv, 20.0), (model.PSP_output_I_conv, 20.0)):
            conv.weight_g.mul_(gain)
    mel = torch.randn(2, 80, 40, generator=torch.Generator().manual_seed(6))
    want = og.apnet_forward(sd_numpy(model), hp, mel.numpy(), 1024, 256, 1024)
    for precision, tol in (("fp32", 1e-4), ("tc_f16", 2e-3)):
        model.precision = precision
        logamp, pha, rea, imag, audio = model(mel.to(DEV))
        scale = max(1.0, float(np.abs(want[4]).max()))
        e_log, e_aud = np.abs(logamp.cpu().numpy() - want[0]).max(), np.abs(audio.cpu().numpy() - want[4]).max()
        print("apnet recipe width", precision, float(e_log), float(e_aud), "audio absmax", scale)
        assert e_log <= 3 * tol, (precision, e_log)
        assert e_aud <= tol * scale, (precision, e_aud)
    assert model.last_launches > 0


def test_vocos_istft_head_matches_the_oracle():
    """ISTFTHead.forward (models/codec/kmeans/vocos.py:333-361) on the codec's geometry (n_fft 800, hop 200: a
    non-power-of-two FFT) with the magnitude clip exercised."""
    from amphion_b200.vocoders import ISTFTHead
    from oracle import generator as og
    torch.manual_seed(3)
    head = ISTFTHead(dim=48, n_fft=800, hop_length=200).to(DEV)
    with torch.no_grad():
        head.out.weight.mul_(8.0)                                   # some log-magnitudes beyond log(1e2)
    x = torch.randn(2, 21, 48, generator=torch.Generator().manual_seed(4))
    got = head(x.to(DEV))
    y = (x.double() @ head.out.weight.detach().cpu().double().T + head.out.bias.detach().cpu().double()).transpose(1, 2).numpy()
    mag = np.minimum(np.exp(y[:, :401]), 1e2)
    assert (mag == 1e2).any() and (mag < 1e2).any()
    want = og.istft_same(mag * np.cos(y[:, 401:]), mag * np.sin(y[:, 401:]), 800, 200, 800)
    assert got.shape == want.shape == (2, 21 * 200)
    assert np.abs(got.cpu().numpy() - want).max() <= 1e-3 * max(1.0, np.abs(want).max())   # TF32-free fp32 GEMM + fp32 FFT


@pytest.mark.parametrize("B,T", [(1, 1), (3, 5), (1, 130)])
def test_apnet_odd_shapes(B, T):
    """Channel counts that are not multiples of 16, a single frame, a tile boundary: against the oracle."""
    from helpers import sd_numpy
    from oracle import generator as og
    hp = dict(ASP_channel=24, ASP_resblock_kernel_sizes=[3, 5], ASP_resblock_dilation_sizes=[[1, 3, 5], [1, 2, 4]],
              ASP_input_conv_kernel_size=3, ASP_output_conv_kernel_size=5,
              PSP_channel=40, PSP_resblock_kernel_sizes=[7], PSP_resblock_dilation_sizes=[[1, 3, 5]],
              PSP_input_conv_kernel_size=7, PSP_output_R_conv_kernel_size=3, PSP_output_I_conv_kernel_size=3)
    pre = dict(n_mel=10, n_fft=32, hop_size=8, win_size=32, extract_amplitude_phase=True, sample_rate=16000)
    model = _apnet_model(hp, pre, seed=21)
    with torch.no_grad():
        for conv, gain in ((model.ASP_output_conv, 3.0), (model.PSP_output_R_conv, 20.0), (model.PSP_output_I_conv, 20.0)):
            conv.weight_g.mul_(gain)
    mel = torch.randn(B, 10, T, generator=torch.Generator().manual_seed(22))
    want = og.apnet_forward(sd_numpy(model), hp, mel.numpy(), 32, 8, 32)
    for precision, tol in (("fp32", 1e-4), ("tc_f16", 2e-3)):
        model.precision = precision
        got = model(mel.to(DEV))
        assert got[4].shape == (B, 1, T * 8)
        scale = max(1.0, float(np.abs(want[4]).max()))
        assert np.abs(got[0].cpu().numpy() - want[0]).max() <= 3 * tol, precision
        assert np.abs(got[4].cpu().numpy() - want[4]).max() <= tol * scale, precision


def test_amplitude_phase_spectrum_matches_reference_fixture():
    """utils/mel.py:244-280 on the native STFT: re / im against the reference fixture, log-amplitude and phase
    consistent with them, and the squeezed B == 1 form."""
    from types import SimpleNamespace as NS
    from amphion_b200 import mel
    g, _ = load_golden("amp_phase")
    cfgp = NS(sample_rate=22050, n_fft=256, n_mel=40, fmin=0, fmax=8000, win_size=256, hop_size=64)
    y = torch.from_numpy(g["y"]).to(DEV)
    la, ph, re, im = (t.cpu().numpy() for t in mel.amplitude_phase_spectrum(y, cfgp))
    scale = np.abs(g["rea"]).max()
    assert la.shape == (2, 129, 46)
    assert np.abs(re - g["rea"]).max() <= 2e-5 * scale and np.abs(im - g["imag"]).max() <= 2e-5 * scale
    np.testing.assert_allclose(la, g["logamp"], atol=2e-3)
    np.testing.assert_allclose(la, np.log(np.sqrt(re * re + im * im) + 1e-5), atol=1e-5)
    mag = np.sqrt(g["rea"] ** 2 + g["imag"] ** 2)
    d = np.abs(ph - g["pha"])
    assert (np.minimum(d, 2 * np.pi - d) * mag).max() <= 1e-4 * scale
    np.testing.assert_allclose(ph, np.arctan2(im, re), atol=1e-5)
    assert tuple(mel.amplitude_phase_spectrum(y[:1], cfgp)[0].shape) == (129, 46)
