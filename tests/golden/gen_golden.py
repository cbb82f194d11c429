"""Generate the golden fixtures in this directory by RUNNING THE REFERENCE.

Run only in the build container (needs /root/reference, which does not exist on
the GPU box):   python tests/golden/gen_golden.py

What it does: imports the reference's own modules (generator classes,
Activation1d, utils/mel.py, utils/stft.py, gan_vocoder_inference.py) with
import-time stubs for packages that are absent here (lhotse, json5, ruamel,
accelerate, librosa), builds small seeded models, runs them on CPU fp32 and
stores inputs / state dicts / outputs as ``.npz``.  The librosa stand-in is
``oracle.mel.slaney_mel_filterbank`` (cross-checked against torchaudio in
tests/test_oracle.py); the mel basis is stored in the fixture so parity never
depends on how it was generated.
"""
import os
import sys
import types
from types import SimpleNamespace as NS

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)


class _Stub(types.ModuleType):
    """Module whose every attribute is a dummy class (never executed)."""
    __path__ = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return type(name, (), {})


for _m in ["lhotse", "lhotse.dataset", "lhotse.dataset.collation", "lhotse.dataset.input_strategies",
           "lhotse.utils", "json5", "ruamel", "ruamel.yaml", "ruamel_yaml", "accelerate"]:
    if _m not in sys.modules:
        sys.modules[_m] = _Stub(_m)

from oracle import mel as omel  # noqa: E402

_librosa = types.ModuleType("librosa")
_filters = types.ModuleType("librosa.filters")
_util = types.ModuleType("librosa.util")


def _mel(sr=None, n_fft=None, n_mels=128, fmin=0.0, fmax=None, *a, **k):
    return omel.slaney_mel_filterbank(sr, n_fft, n_mels, fmin, fmax)


_filters.mel = _mel
_util.pad_center = lambda data, size, **k: omel.pad_center(data, size)
_util.tiny = lambda x: np.finfo(np.float32).tiny
_util.normalize = lambda x, norm=None: x
_librosa.filters, _librosa.util = _filters, _util
sys.modules.update({"librosa": _librosa, "librosa.filters": _filters, "librosa.util": _util})

import warnings  # noqa: E402

warnings.filterwarnings("ignore")

from models.vocoders.gan.generator.hifigan import HiFiGAN, HiFiGAN_vits  # noqa: E402
from models.vocoders.gan.generator.bigvgan import BigVGAN  # noqa: E402
from models.vocoders.gan.generator.nsfhifigan import NSFHiFiGAN  # noqa: E402
from modules.anti_aliasing.act import Activation1d  # noqa: E402
from modules.activation_functions.snake import SnakeBeta  # noqa: E402
import utils.mel as rmel  # noqa: E402
import utils.stft as rstft  # noqa: E402


def sd_np(module):
    return {k: v.detach().cpu().numpy() for k, v in module.state_dict().items()}


def run_with_stage_hooks(model, mel, nk):
    outs = {}
    hooks = []
    for n, rb in enumerate(model.resblocks):
        hooks.append(rb.register_forward_hook(lambda m, i, o, n=n: outs.__setitem__(n, o.detach().clone())))
    with torch.no_grad():
        y = model(mel)
    for h in hooks:
        h.remove()
    stages = []
    for i in range(len(model.resblocks) // nk):
        xs = outs[i * nk]
        for j in range(1, nk):
            xs = xs + outs[i * nk + j]
        stages.append((xs / nk).numpy())
    return y.numpy(), stages


def gen_generator(name, kind, hp, n_mel, B, T, seed, mel_dist="randn"):
    pre = NS(n_mel=n_mel, hop_size=int(np.prod(hp["upsample_rates"])), extract_amplitude_phase=False)
    cfg = NS(preprocess=pre, model=NS(**{kind: NS(**hp)}))
    torch.manual_seed(seed)
    model = (HiFiGAN if kind == "hifigan" else BigVGAN)(cfg).eval()
    g = torch.Generator().manual_seed(seed + 1)
    if kind == "bigvgan":
        with torch.no_grad():
            for n, p in model.named_parameters():
                if n.endswith(".alpha") or n.endswith(".beta"):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.3 + (0.0 if hp["snake_logscale"] else 1.0))
    if mel_dist == "randn":
        mel = torch.randn(B, n_mel, T, generator=g)
    else:  # log-mel range (utils/mel.py:11)
        mel = torch.rand(B, n_mel, T, generator=g) * 13.5 - 11.5
    wav, stages = run_with_stage_hooks(model, mel, len(hp["resblock_kernel_sizes"]))
    out = {"mel": mel.numpy(), "wav": wav}
    for i, s in enumerate(stages):
        out[f"stage{i}"] = s
    for k, v in sd_np(model).items():
        out["sd:" + k] = v
    np.savez(os.path.join(HERE, name + ".npz"), **out)
    print(name, "wav", wav.shape, "absmax", float(np.abs(wav).max()),
          "bytes", os.path.getsize(os.path.join(HERE, name + ".npz")))
    return cfg, model


HP_HIFIGAN_RB1 = dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4],
                      upsample_initial_channel=64, resblock_kernel_sizes=[3, 7, 11],
                      resblock_dilation_sizes=[[1, 3, 5]] * 3)
HP_HIFIGAN_RB2 = dict(resblock="2", upsample_rates=[4, 4], upsample_kernel_sizes=[8, 8],
                      upsample_initial_channel=32, resblock_kernel_sizes=[3, 5, 7],
                      resblock_dilation_sizes=[[1, 2], [2, 6], [3, 12]])
HP_BIGVGAN_RB1 = dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4],
                      upsample_initial_channel=64, resblock_kernel_sizes=[3, 7, 11],
                      resblock_dilation_sizes=[[1, 3, 5]] * 3, activation="snakebeta", snake_logscale=True)
HP_BIGVGAN_RB2 = dict(resblock="2", upsample_rates=[2, 2], upsample_kernel_sizes=[4, 4],
                      upsample_initial_channel=32, resblock_kernel_sizes=[3, 5],
                      resblock_dilation_sizes=[[1, 2], [2, 6]], activation="snake", snake_logscale=False)


HP_NSF = dict(resblock="1", harmonic_num=8, upsample_rates=[4, 2, 2], upsample_kernel_sizes=[8, 4, 4],
              upsample_initial_channel=64, resblock_kernel_sizes=[3, 7, 11], resblock_dilation_sizes=[[1, 3, 5]] * 3)


def gen_nsfhifigan():
    """NSF-HiFiGAN (nsfhifigan.py:181-283).  The harmonic source is random (SineGen draws rand/randn), yet the
    output is not: `x_source = x[:, :, :length]` (:269) adds x to itself, so the source only contributes its
    length.  The fixture stores two runs under different torch seeds to pin exactly that, plus the f0-aware
    plumbing (gan_vocoder_inference.py:76-95)."""
    import models.vocoders.gan.gan_vocoder_inference as gvi
    n_mel, B, T = 20, 2, 17
    pre = NS(n_mel=n_mel, hop_size=int(np.prod(HP_NSF["upsample_rates"])), sample_rate=24000,
             extract_amplitude_phase=False)
    cfg = NS(preprocess=pre, model=NS(nsfhifigan=NS(**HP_NSF)))
    torch.manual_seed(41)
    model = NSFHiFiGAN(cfg).eval()
    g = torch.Generator().manual_seed(42)
    mel = torch.randn(B, n_mel, T, generator=g)
    f0 = torch.rand(B, T, generator=g) * 300 + 80
    f0[:, 3:6] = 0.0                                  # unvoiced frames
    with torch.no_grad():
        torch.manual_seed(1)
        wav = model(mel, f0).numpy()
        torch.manual_seed(2)
        wav2 = model(mel, f0 * 0.5).numpy()           # other source, other noise: same samples
        wav_long_f0 = model(mel, torch.cat([f0, f0[:, :4]], dim=1)).numpy()   # f0 longer than the mel: no truncation
    out = {"mel": mel.numpy(), "f0": f0.numpy(), "wav": wav, "wav_other_source": wav2, "wav_long_f0": wav_long_f0}
    mels = [torch.randn(n_mel, t, generator=g) for t in (7, 11, 4)]
    f0s = [torch.rand(t, generator=g) * 200 + 100 for t in (7, 11, 4)]
    auds = gvi.synthesis_audios(cfg, model, mels, f0s=f0s, batch_size=2)
    for i, (m, f, a) in enumerate(zip(mels, f0s, auds)):
        out[f"pl_mel{i}"], out[f"pl_f0{i}"], out[f"pl_audio{i}"] = m.numpy(), f.numpy(), a.numpy()
    for k, v in sd_np(model).items():
        out["sd:" + k] = v
    np.savez(os.path.join(HERE, "nsfhifigan.npz"), **out)
    print("nsfhifigan wav", wav.shape, "absmax", float(np.abs(wav).max()), "source-independent:",
          bool((wav == wav2).all()), bool((wav == wav_long_f0).all()), [a.shape for a in auds])


VITS_ARGS = dict(initial_channel=24, resblock="1", resblock_kernel_sizes=[3, 7, 11],
                 resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[4, 2], upsample_initial_channel=64,
                 upsample_kernel_sizes=[8, 4], gin_channels=10)
VITS_ARGS_RB2 = dict(initial_channel=12, resblock="2", resblock_kernel_sizes=[3, 5], resblock_dilation_sizes=[[1, 2], [2, 6]],
                     upsample_rates=[2, 2], upsample_initial_channel=32, upsample_kernel_sizes=[4, 4], gin_channels=0)


def gen_hifigan_vits():
    """HiFiGAN_vits (hifigan.py:376-449), the decoder inside VITS: with and without the global conditioning."""
    out = {}
    for tag, args, seed, B, T in (("a", VITS_ARGS, 51, 2, 19), ("b", VITS_ARGS_RB2, 52, 1, 23)):
        torch.manual_seed(seed)
        model = HiFiGAN_vits(**args).eval()
        gen = torch.Generator().manual_seed(seed + 1)
        x = torch.randn(B, args["initial_channel"], T, generator=gen)
        out[f"{tag}:x"] = x.numpy()
        with torch.no_grad():
            out[f"{tag}:wav"] = model(x).numpy()
            if args["gin_channels"]:
                g = torch.randn(B, args["gin_channels"], 1, generator=gen)
                out[f"{tag}:g"] = g.numpy()
                out[f"{tag}:wav_g"] = model(x, g=g).numpy()
        for k, v in sd_np(model).items():
            out[f"{tag}:sd:" + k] = v
    np.savez(os.path.join(HERE, "hifigan_vits.npz"), **out)
    print("hifigan_vits", out["a:wav"].shape, out["b:wav"].shape, float(np.abs(out["a:wav_g"] - out["a:wav"]).max()))


def gen_save_audio():
    """utils/io.py:49-76 with torchaudio.save intercepted: the float tensor it is handed is the fixture."""
    import utils.io as rio
    got = {}
    rio.torchaudio.save = lambda path, wav, fs, **kw: got.__setitem__(path, (wav.numpy().copy(), fs, dict(kw)))
    g = torch.Generator().manual_seed(9)
    w = (torch.randn(3000, generator=g) * 0.2).numpy()
    w[100] = -0.73                                     # the peak is a negative sample
    out = {"w": w}
    for ts in (0, 1):
        for sil in (0, 1):
            rio.save_audio(f"k{ts}{sil}", w, 16000, add_silence=bool(sil), turn_up=bool(ts))
            out[f"float_turnup{ts}_silence{sil}"] = got[f"k{ts}{sil}"][0]
    assert got["k00"][2] == dict(encoding="PCM_S", bits_per_sample=16)
    np.savez(os.path.join(HERE, "save_audio.npz"), **out)
    print("save_audio", {k: v.shape for k, v in out.items()})


def gen_activation1d():
    torch.manual_seed(7)
    act = Activation1d(activation=SnakeBeta(6, alpha_logscale=True))
    with torch.no_grad():
        act.act.alpha.normal_(0, 0.3)
        act.act.beta.normal_(0, 0.3)
    x = torch.randn(2, 6, 37) * 2
    with torch.no_grad():
        up = act.upsample(x)
        y = act(x)
    np.savez(os.path.join(HERE, "activation1d.npz"), x=x.numpy(), up=up.numpy(), y=y.numpy(),
             alpha=act.act.alpha.detach().numpy(), beta=act.act.beta.detach().numpy(),
             f_up=act.upsample.filter.numpy().reshape(-1), f_down=act.downsample.lowpass.filter.numpy().reshape(-1))
    print("activation1d", y.shape, act.upsample.filter.reshape(-1)[:6].tolist())


def gen_mel():
    cfgp = NS(sample_rate=22050, n_fft=1024, n_mel=80, fmin=0, fmax=8000, win_size=1024, hop_size=256)
    g = torch.Generator().manual_seed(0)
    y = (torch.rand(2, 8192, generator=g) * 2 - 1) * 0.9
    out = {"y": y.numpy(), "mel_basis": omel.slaney_mel_filterbank(22050, 1024, 80, 0, 8000)}
    rmel.mel_basis.clear(); rmel.hann_window.clear()
    out["extract_mel_features"] = rmel.extract_mel_features(y, cfgp).numpy()
    rmel.mel_basis.clear(); rmel.hann_window.clear()
    out["mel_spectrogram_torch"] = rmel.mel_spectrogram_torch(y, cfgp).numpy()
    out["extract_linear_features"] = rmel.extract_linear_features(y, cfgp).numpy()
    rmel.mel_basis.clear(); rmel.hann_window.clear()
    out["extract_mel_features_b1"] = rmel.extract_mel_features(y[:1], cfgp).numpy()   # squeeze(0) case
    # TacotronSTFT hard-codes .cuda() (utils/stft.py:168-169): identity shim for the CPU run
    torch.Tensor.cuda = lambda self, *a, **k: self
    taco = rstft.TacotronSTFT(1024, 256, 1024, 80, 22050, 0, 8000)
    m, e = taco.mel_spectrogram(y)
    out["taco_mel"], out["taco_energy"] = m.numpy(), e.numpy()
    out["taco_mel_basis"] = taco.mel_basis.numpy()
    # odd geometry: win < n_fft, different hop
    cfg2 = NS(sample_rate=16000, n_fft=512, n_mel=40, fmin=50, fmax=7600, win_size=400, hop_size=160)
    y2 = (torch.rand(3, 3000, generator=g) * 2 - 1) * 0.5
    rmel.mel_basis.clear(); rmel.hann_window.clear()
    out["y2"] = y2.numpy()
    out["mel_basis2"] = omel.slaney_mel_filterbank(16000, 512, 40, 50, 7600)
    out["extract_mel_features2"] = rmel.extract_mel_features(y2, cfg2).numpy()
    np.savez(os.path.join(HERE, "mel.npz"), **out)
    print("mel", out["extract_mel_features"].shape, out["taco_mel"].shape, out["extract_mel_features2"].shape)


def gen_mel_grad():
    """The trainers' mel loss differentiated by the reference itself (gan_vocoder_trainer.py:368-396:
    L1(extract_mel_features(y_gt), extract_mel_features(y_pred)) * 45), plus a plain random cotangent."""
    out = {}
    g = torch.Generator().manual_seed(17)
    for tag, cfgp, B, T in (("a", NS(sample_rate=22050, n_fft=1024, n_mel=80, fmin=0, fmax=8000, win_size=1024, hop_size=256), 2, 6144),
                            ("b", NS(sample_rate=16000, n_fft=512, n_mel=40, fmin=50, fmax=7600, win_size=400, hop_size=160), 3, 2000)):
        y_gt = (torch.rand(B, T, generator=g) * 2 - 1) * 0.8
        y_pred = (y_gt + 0.2 * torch.randn(B, T, generator=g)).clamp(-1, 1)
        y_pred[0, T // 3: T // 3 + 3 * cfgp.n_fft] = 0.0                 # silence: frames below the log clamp (zero gradient)
        y_pred.requires_grad_(True)
        rmel.mel_basis.clear(); rmel.hann_window.clear()
        mel_gt = rmel.extract_mel_features(y_gt, cfgp)
        mel_pred = rmel.extract_mel_features(y_pred, cfgp)
        loss = torch.nn.L1Loss(reduction="mean")(mel_gt, mel_pred) * 45
        (gl,) = torch.autograd.grad(loss, y_pred, retain_graph=True)
        cot = torch.randn(mel_pred.shape, generator=g)
        (gc,) = torch.autograd.grad(mel_pred, y_pred, cot)
        basis = omel.slaney_mel_filterbank(cfgp.sample_rate, cfgp.n_fft, cfgp.n_mel, cfgp.fmin, cfgp.fmax)
        out.update({f"{tag}_y_gt": y_gt.numpy(), f"{tag}_y_pred": y_pred.detach().numpy(), f"{tag}_loss": loss.detach().numpy(),
                    f"{tag}_grad_loss": gl.numpy(), f"{tag}_cot": cot.numpy(), f"{tag}_grad_cot": gc.numpy(),
                    f"{tag}_mel_basis": basis, f"{tag}_geom": np.array([cfgp.n_fft, cfgp.hop_size, cfgp.win_size, cfgp.n_mel])})
        print("mel_grad", tag, float(loss), float(gl.abs().max()), float(gc.abs().max()))
    np.savez(os.path.join(HERE, "mel_grad.npz"), **out)


HP_APNET = dict(ASP_channel=32, ASP_resblock_kernel_sizes=[3, 7, 11], ASP_resblock_dilation_sizes=[[1, 3, 5]] * 3,
                ASP_input_conv_kernel_size=7, ASP_output_conv_kernel_size=7,
                PSP_channel=48, PSP_resblock_kernel_sizes=[3, 7], PSP_resblock_dilation_sizes=[[1, 3, 5], [1, 2, 4]],
                PSP_input_conv_kernel_size=5, PSP_output_R_conv_kernel_size=7, PSP_output_I_conv_kernel_size=7)
APNET_PRE = dict(n_mel=12, n_fft=64, hop_size=16, win_size=64, extract_amplitude_phase=True)


def gen_apnet():
    """APNet.forward (apnet.py:357-399) and the inference plumbing that unpacks its fifth output."""
    from models.vocoders.gan.generator.apnet import APNet
    import models.vocoders.gan.gan_vocoder_inference as gvi
    cfg = NS(preprocess=NS(**APNET_PRE), model=NS(generator="apnet", apnet=NS(**HP_APNET)))
    torch.manual_seed(77)
    model = APNet(cfg).eval()
    g = torch.Generator().manual_seed(78)
    with torch.no_grad():   # the output convolutions are initialised with std 0.01: scale them so the phase is generic
        for conv, gain in ((model.ASP_output_conv, 3.0), (model.PSP_output_R_conv, 20.0), (model.PSP_output_I_conv, 20.0)):
            conv.weight_g.mul_(gain)
            conv.bias.copy_(torch.randn(conv.bias.shape, generator=g) * 0.3)
    mel = torch.randn(2, APNET_PRE["n_mel"], 23, generator=g)
    with torch.no_grad():
        logamp, pha, rea, imag, audio = model(mel)
    out = {"mel": mel.numpy(), "logamp": logamp.numpy(), "pha": pha.numpy(), "rea": rea.numpy(), "imag": imag.numpy(),
           "audio": audio.numpy()}
    out["inference"] = gvi.vocoder_inference(cfg, model, mel, device="cpu").numpy()
    # the weights are not stored: tests/conftest.py:load_golden_apnet draws them again from the same seeds
    # and checks them against this digest
    sys.path.insert(0, os.path.dirname(HERE))
    from conftest import state_dict_sha256
    sd = sd_np(model)
    out["sd_keys"] = np.array(list(sd))
    out["sd_sha256"] = np.array(state_dict_sha256(list(sd), sd))
    np.savez(os.path.join(HERE, "apnet.npz"), **out)
    print("apnet", audio.shape, float(audio.abs().max()), float(logamp.abs().max()), os.path.getsize(os.path.join(HERE, "apnet.npz")))


def gen_amp_phase():
    """amplitude_phase_spectrum (utils/mel.py:244-280), batched and the squeezed B == 1 case."""
    cfgp = NS(sample_rate=22050, n_fft=256, n_mel=40, fmin=0, fmax=8000, win_size=256, hop_size=64)
    g = torch.Generator().manual_seed(33)
    y = (torch.rand(2, 3000, generator=g) * 2 - 1) * 0.8
    la, ph, re, im = rmel.amplitude_phase_spectrum(y, cfgp)
    out = {"y": y.numpy(), "logamp": la.numpy(), "pha": ph.numpy(), "rea": re.numpy(), "imag": im.numpy(),
           "b1_shape": np.array(rmel.amplitude_phase_spectrum(y[:1], cfgp)[0].shape)}
    np.savez(os.path.join(HERE, "amp_phase.npz"), **out)
    print("amp_phase", la.shape, out["b1_shape"])


def gen_plumbing(cfg, model):
    import models.vocoders.gan.gan_vocoder_inference as gvi
    g = torch.Generator().manual_seed(5)
    mels = [torch.randn(16, t, generator=g) for t in (9, 14, 5)]
    auds = gvi.synthesis_audios(cfg, model, mels, batch_size=2)
    out = {f"mel{i}": m.numpy() for i, m in enumerate(mels)}
    out.update({f"audio{i}": a.numpy() for i, a in enumerate(auds)})
    batched = gvi.vocoder_inference(cfg, model, torch.stack([mels[1], mels[1].flip(-1)]), device="cpu")
    out["batched_in"] = torch.stack([mels[1], mels[1].flip(-1)]).numpy()
    out["batched_out"] = batched.numpy()
    np.savez(os.path.join(HERE, "plumbing.npz"), **out)
    print("plumbing", [a.shape for a in auds], batched.shape)


if __name__ == "__main__":
    LATER = {"nsfhifigan": gen_nsfhifigan, "save_audio": gen_save_audio, "hifigan_vits": gen_hifigan_vits,
             "mel_grad": gen_mel_grad, "apnet": gen_apnet, "amp_phase": gen_amp_phase}
    if sys.argv[1:] and set(sys.argv[1:]) <= set(LATER):   # later additions regenerate alone
        for name in sys.argv[1:]:
            LATER[name]()
        sys.exit(0)
    cfg, model = gen_generator("hifigan_rb1", "hifigan", HP_HIFIGAN_RB1, 16, 2, 24, seed=1234)
    gen_plumbing(cfg, model)
    gen_generator("hifigan_rb2", "hifigan", HP_HIFIGAN_RB2, 20, 1, 19, seed=11, mel_dist="logmel")
    gen_generator("bigvgan_rb1", "bigvgan", HP_BIGVGAN_RB1, 20, 2, 21, seed=21)
    gen_generator("bigvgan_rb2", "bigvgan", HP_BIGVGAN_RB2, 12, 1, 33, seed=31)
    gen_activation1d()
    gen_mel()
    gen_nsfhifigan()
    gen_save_audio()
    gen_hifigan_vits()
    gen_mel_grad()
    gen_apnet()
    gen_amp_phase()
