"""CPU-only checks of the host side: the C-ABI library loads and exports every
symbol the header declares, argument errors surface as exceptions, the module
mirrors keep the reference's parameter names / init order, and nothing falls
back to the CPU."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN_MODELS, GOLDEN_NSF, GOLDEN_VITS, ROOT, load_golden, load_golden_vits
from helpers import build_model, make_cfg


def test_library_exports_every_declared_symbol():
    from amphion_b200 import _capi
    header = open(os.path.join(ROOT, "include", "amphion_b200.h")).read()
    declared = set(re.findall(r"\b(ab_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    for name in declared:
        assert hasattr(_capi.lib, name), name
    assert _capi.lib.ab_version() >= 100
    assert os.path.dirname(_capi.LIB_PATH).endswith("amphion_b200")  # in-tree, not site-packages


def test_create_rejects_bad_configs():
    from amphion_b200 import _capi
    h = C.c_void_p()
    cfg = _capi.GeneratorConfig()
    assert _capi.lib.ab_generator_create(C.byref(cfg), C.byref(h)) == -1
    assert "n_mel" in _capi.last_error()
    with pytest.raises(RuntimeError, match="ab_generator_create"):
        _capi.check(_capi.lib.ab_generator_create(C.byref(cfg), C.byref(h)), "ab_generator_create")
    assert _capi.lib.ab_generator_create(None, C.byref(h)) == -1
    m = C.c_void_p()
    assert _capi.lib.ab_mel_create(C.byref(_capi.MelConfig(1023, 256, 1024, 80, 0, 0.0, 1e-5)), C.byref(m)) == -1


def test_handle_lifecycle_and_tensor_table_without_gpu():
    from amphion_b200 import _capi
    kind, hp, n_mel = GOLDEN_MODELS["bigvgan_rb1"]
    model = build_model(kind, hp, n_mel)
    h = model._ensure_handle()
    names = [_capi.lib.ab_generator_tensor_name(h, i).decode() for i in range(_capi.lib.ab_generator_num_tensors(h))]
    sd = model.state_dict()
    for n in names:  # every tensor the library wants exists in the module (folded or weight-normed)
        assert n in sd or (n + "_v" in sd and n + "_g" in sd), n
    assert "ups.0.0.weight" in names and "resblocks.5.activations.5.act.beta" in names
    assert _capi.lib.ab_generator_param_bytes(h) > sum(v.numel() * 4 for k, v in sd.items() if k.endswith("_v"))
    assert _capi.lib.ab_generator_workspace_bytes(h, 2, 21) > 0
    # forward before bind/finalize is a state error, not a crash
    rc = _capi.lib.ab_generator_forward(h, C.c_void_p(8), 1, 4, _capi.shape_array((1, 1, 1)), C.c_void_p(8),
                                        C.c_void_p(256), 1 << 30, None)
    assert rc == -4 and "finalize" in _capi.last_error()


@pytest.mark.parametrize("name", sorted(GOLDEN_MODELS))
def test_state_dict_keys_and_shapes_match_reference(name):
    kind, hp, n_mel = GOLDEN_MODELS[name]
    _, sd = load_golden(name)
    model = build_model(kind, hp, n_mel)
    msd = model.state_dict()
    assert list(msd.keys()) == list(sd.keys())          # same names, same order
    for k in sd:
        assert tuple(msd[k].shape) == sd[k].shape, k
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)


def test_nsfhifigan_module_matches_reference_layout():
    from amphion_b200 import _capi
    kind, hp, n_mel = GOLDEN_NSF
    _, sd = load_golden("nsfhifigan")
    model = build_model(kind, hp, n_mel, seed=41)        # the fixture's seed: same construction order => same weights
    msd = model.state_dict()
    assert list(msd.keys()) == list(sd.keys())
    for k, v in msd.items():
        np.testing.assert_array_equal(v.numpy(), sd[k], err_msg=k)
    # tensor table of the C ABI = HiFi-GAN's; the source / noise-conv parameters are not consumed
    h = model._ensure_handle()
    names = [_capi.lib.ab_generator_tensor_name(h, i).decode() for i in range(_capi.lib.ab_generator_num_tensors(h))]
    assert "ups.0.weight" in names and not any(n.startswith(("m_source", "noise_convs")) for n in names)
    # the reference's ResBlock2 cannot be constructed (nsfhifigan.py:111): same TypeError here
    with pytest.raises(TypeError):
        build_model(kind, dict(hp, resblock="2"), n_mel)
    # stage lengths when the harmonic source is shorter than a stage (short f0 / odd source stride):
    # `length = min(x.shape[-1], x_source.shape[-1])` (nsfhifigan.py:264-268), restated by the C ABI
    hop = int(np.prod(hp["upsample_rates"]))
    assert _capi.lib.ab_generator_output_samples(h, 10, 0) == 10 * hop
    assert _capi.lib.ab_generator_output_samples(h, 10, 12) == 10 * hop     # f0 longer than the mel: nothing cut
    assert _capi.lib.ab_generator_output_samples(h, 10, 7) == 7 * hop       # every stage cut to the source length
    odd = build_model(kind, dict(hp, upsample_rates=[4, 3, 3], upsample_kernel_sizes=[8, 5, 5]), n_mel)
    ho = odd._ensure_handle()
    T, src = 5, 5 * 36
    l0 = min(T * 4, (src + 2 * (9 // 2) - 18) // 9 + 1)      # stage 0: s = 9
    l1 = min(l0 * 3, (src + 2 * (3 // 2) - 6) // 3 + 1)       # stage 1: s = 3
    assert _capi.lib.ab_generator_output_samples(ho, T, T) == min(l1 * 3, src) < T * 36
    with pytest.raises(RuntimeError, match="CUDA"):      # no CPU fallback
        model(torch.zeros(1, n_mel, 4), torch.zeros(1, 4))


def test_seeded_init_reproduces_reference_weights():
    # the reference fixture was built with torch.manual_seed(1234); HiFiGAN(cfg):
    # same construction order => same RNG stream => identical parameters
    kind, hp, n_mel = GOLDEN_MODELS["hifigan_rb1"]
    _, sd = load_golden("hifigan_rb1")
    model = build_model(kind, hp, n_mel, seed=1234)
    for k, v in model.state_dict().items():
        np.testing.assert_array_equal(v.numpy(), sd[k], err_msg=k)


def test_remove_weight_norm_keeps_loadable_names(capsys):
    kind, hp, n_mel = GOLDEN_MODELS["hifigan_rb2"]
    model = build_model(kind, hp, n_mel, seed=3)
    w = torch._weight_norm(model.conv_pre.weight_v, model.conv_pre.weight_g, 0).detach().clone()
    model.remove_weight_norm()
    assert "conv_pre.weight" in model.state_dict() and "conv_pre.weight_v" not in model.state_dict()
    torch.testing.assert_close(model.conv_pre.weight.detach(), w)
    assert "Removing weight norm" in capsys.readouterr().out


def test_no_cpu_fallback():
    kind, hp, n_mel = GOLDEN_MODELS["hifigan_rb1"]
    model = build_model(kind, hp, n_mel, seed=0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model(torch.zeros(1, n_mel, 8))
    from amphion_b200.vocoders.activations import Activation1d, SnakeBeta
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Activation1d(SnakeBeta(4))(torch.zeros(1, 4, 8))
    from amphion_b200 import mel
    cfgp = make_cfg("hifigan", hp, 80).preprocess
    cfgp.sample_rate, cfgp.n_fft, cfgp.fmin, cfgp.fmax, cfgp.win_size = 22050, 1024, 0, 8000, 1024
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mel.extract_mel_features(torch.zeros(1, 4096), cfgp)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "amphion_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), os.path.join(dirpath, f)


def test_pad_mels_to_tensors_matches_reference_layout():
    from amphion_b200.util import pad_mels_to_tensors
    from oracle import generator as og
    mels = [torch.randn(5, t) for t in (7, 3, 9, 4, 6)]
    for bs in (None, 2, 5, 8):
        ts, fr = pad_mels_to_tensors(mels, bs)
        ots, ofr = og.pad_mels([m.numpy() for m in mels], bs)
        assert len(ts) == len(ots)
        for a, b, f, of in zip(ts, ots, fr, ofr):
            np.testing.assert_array_equal(a.numpy(), b)
            np.testing.assert_array_equal(f.numpy(), of)
    assert pad_mels_to_tensors([], 4) == ([], [])


def test_kaiser_filter_matches_reference_buffer():
    from amphion_b200.vocoders.activations import kaiser_sinc_filter1d
    g, _ = load_golden("activation1d")
    np.testing.assert_allclose(kaiser_sinc_filter1d(0.25, 0.3, 12).reshape(-1).numpy(), g["f_up"], atol=1e-8)


def test_mel_filterbank_host_matches_oracle():
    from amphion_b200 import mel
    from oracle import mel as om
    for args in [(22050, 1024, 80, 0, 8000), (16000, 512, 40, 50, 7600), (24000, 1024, 100, 0, None)]:
        np.testing.assert_allclose(mel.librosa_mel_fn(*args).numpy(), om.slaney_mel_filterbank(*args), atol=1e-7)


def test_wav_writer_roundtrip(tmp_path):
    import wave
    from amphion_b200.io import write_wav_pcm16
    x = (np.arange(-5, 6) * 3000).astype(np.int16)
    write_wav_pcm16(tmp_path / "a.wav", x, 24000)
    with wave.open(str(tmp_path / "a.wav")) as f:
        assert (f.getnchannels(), f.getsampwidth(), f.getframerate(), f.getnframes()) == (1, 2, 24000, 11)
        np.testing.assert_array_equal(np.frombuffer(f.readframes(11), "<i2"), x)
    # no CPU fallback: the quantiser only exists as a CUDA kernel, so where no device is visible save_audio raises
    # (checked in a child process with every device hidden, so that it holds on a GPU machine as well)
    code = ("import sys; import numpy as np; from amphion_b200.io import save_audio\n"
            "try:\n    save_audio(sys.argv[1], np.zeros(16, np.float32), 16000)\nexcept RuntimeError:\n    sys.exit(3)\n")
    r = subprocess.run([sys.executable, "-c", code, str(tmp_path / "b.wav")], cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 3 and not (tmp_path / "b.wav").exists()


@pytest.mark.parametrize("tag,seed", [("a", 51), ("b", 52)])
def test_hifigan_vits_module_matches_reference_layout(tag, seed):
    from amphion_b200 import _capi
    from amphion_b200.vocoders import HiFiGAN_vits
    _, sd = load_golden_vits(tag)
    torch.manual_seed(seed)
    model = HiFiGAN_vits(**GOLDEN_VITS[tag])
    msd = model.state_dict()
    assert list(msd.keys()) == list(sd.keys())
    for k, v in msd.items():
        np.testing.assert_array_equal(v.numpy(), sd[k], err_msg=k)
    h = model._ensure_handle()
    names = [_capi.lib.ab_generator_tensor_name(h, i).decode() for i in range(_capi.lib.ab_generator_num_tensors(h))]
    assert "conv_post.bias" not in names and ("cond.weight" in names) == (GOLDEN_VITS[tag]["gin_channels"] > 0)


def test_f0_padding_and_argument_checks_run_before_any_device_work():
    from oracle import generator as og
    from amphion_b200.util import pad_f0_to_tensors
    from amphion_b200.vocoders import HiFiGAN_vits
    f0s = [torch.arange(n, dtype=torch.float32) + 1 for n in (5, 9, 2, 7, 3)]
    for bs in (None, 2, 5):
        got = pad_f0_to_tensors(f0s, bs)
        want = og.pad_f0s([f.numpy() for f in f0s], bs)
        assert len(got) == len(want)
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a.numpy(), b)
    assert pad_f0_to_tensors([], 4) == []
    kind, hp, n_mel = GOLDEN_NSF
    model = build_model(kind, hp, n_mel, seed=1)
    mel = torch.zeros(2, n_mel, 6)
    with pytest.raises(TypeError):
        model(mel, None)
    with pytest.raises(ValueError):
        model(mel, torch.zeros(3, 6))                       # batch mismatch
    with pytest.raises(RuntimeError, match="CUDA"):
        model(mel, torch.zeros(2, 4))                       # a shorter source is computed (stage truncation), on CUDA only
    vits = HiFiGAN_vits(**GOLDEN_VITS["b"])                  # gin_channels == 0
    with pytest.raises(AttributeError):
        vits(torch.zeros(1, 12, 4), g=torch.zeros(1, 3, 1))
    vits_g = HiFiGAN_vits(**GOLDEN_VITS["a"])
    with pytest.raises(ValueError):
        vits_g(torch.zeros(2, 24, 4), g=torch.zeros(2, 7, 1))   # wrong gin
    with pytest.raises(NotImplementedError):
        vits_g(torch.zeros(2, 24, 4), g=torch.zeros(2, 10, 4))  # time-varying conditioning


def test_checkpoint_resolution_follows_the_reference_layout(tmp_path):
    """models/vocoders/vocoder_inference.py:443-451: an experiment directory is searched under checkpoint/ for the
    highest epoch (names with "audio" skipped); accelerate writes pytorch_model.bin or model.safetensors; a directory
    that is one epoch-*_step-* checkpoint, or a plain file, is taken as is."""
    import torch
    from safetensors.torch import save_file
    from amphion_b200.vocoders.vocoder_inference import _read_state_dict, resolve_checkpoint
    exp = tmp_path / "exp"
    for name, fname in (("epoch-0002_step-0000200_loss-0.9", "pytorch_model.bin"),
                        ("epoch-0011_step-0001100_loss-0.5", "model.safetensors"),
                        ("epoch-0007_step-0000700_loss-0.7", "pytorch_model.bin"),
                        ("epoch-0099_audio", "pytorch_model.bin")):
        d = exp / "checkpoint" / name
        d.mkdir(parents=True)
        sd = {"conv_pre.bias": torch.full((3,), float(name.split("-")[1][:4]))}
        if fname.endswith(".bin"):
            torch.save(sd, d / fname)
        else:
            save_file(sd, str(d / fname))
    best = resolve_checkpoint(str(exp))
    assert best.endswith("epoch-0011_step-0001100_loss-0.5/model.safetensors")
    assert float(_read_state_dict(best)["conv_pre.bias"][0]) == 11.0
    one = str(exp / "checkpoint" / "epoch-0007_step-0000700_loss-0.7")
    assert resolve_checkpoint(one) == os.path.join(one, "pytorch_model.bin")
    pt = tmp_path / "legacy.pt"
    torch.save({"generator_state_dict": {"module.conv_pre.bias": torch.zeros(3)}}, pt)
    assert resolve_checkpoint(str(pt)) == str(pt)
    assert list(_read_state_dict(str(pt))) == ["module.conv_pre.bias"]
    with pytest.raises(FileNotFoundError):
        resolve_checkpoint(str(tmp_path))


def test_native_state_is_not_copied_or_pickled(tmp_path):
    """The ctypes handle / packed arena are derived state: deepcopy and torch.save of a model work (also after the
    handle exists) and the copy starts without native state; in-place `.data` edits need `invalidate()`."""
    import copy
    import torch
    kind, hp, n_mel = GOLDEN_MODELS["hifigan_rb1"]
    m = build_model(kind, hp, n_mel, seed=3)
    m.remove_weight_norm()                   # torch cannot deepcopy the derived .weight of old-style weight_norm
    m._ensure_handle()                       # what a first forward leaves behind (no GPU needed for the handle)
    m._arena_key = ("fake",)
    c = copy.deepcopy(m)
    assert c._handle is None and c._arena_key is None and m._handle is not None
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), c.state_dict().values()))
    torch.save(m, tmp_path / "m.pt")
    r = torch.load(tmp_path / "m.pt", weights_only=False)
    assert r._handle is None and list(r.state_dict()) == list(m.state_dict())
    m._arena_key = ("fake",)
    m.load_state_dict(c.state_dict())
    assert m._arena_key is None              # load_state_dict invalidates the packed weights
    m._arena_key = ("fake",)
    m.invalidate()
    assert m._arena_key is None


def test_feature_files_keep_the_reference_layout(tmp_path):
    """utils/io.py:12-30 + vocoder_dataset.py:20-197: <processed_dir>/<dataset>/mels/<uid>.npy [n_mel, T] float32,
    metadata json, __getitem__ contract, overrides=False keeps an existing file."""
    from types import SimpleNamespace as NS
    from amphion_b200 import features
    root = str(tmp_path / "processed_data")
    pre = NS(processed_dir=root, train_file="train.json", valid_file="valid.json", mel_dir="mels", pitch_dir="pitches",
             n_mel=4, use_mel=True, use_frame_pitch=True)
    cfg = NS(preprocess=pre)
    rng = np.random.default_rng(0)
    utts = [{"Dataset": "toy", "Uid": f"u{i}", "Duration": 1.0} for i in range(3)]
    mels = [rng.standard_normal((4, t)).astype(np.float32) for t in (5, 9, 7)]
    for u, m in zip(utts, mels):
        p = features.save_feature(os.path.join(root, "toy"), "mels", u["Uid"], torch.from_numpy(m))
        assert p == os.path.join(root, "toy", "mels", u["Uid"] + ".npy")
        features.save_feature(os.path.join(root, "toy"), "pitches", u["Uid"], np.arange(m.shape[1] + 2, dtype=np.float32))
    features.save_feature(os.path.join(root, "toy"), "mels", "u0", np.zeros((4, 5), np.float32), overrides=False)
    features.write_metadata(root, "toy", utts, "valid.json")
    ds = features.VocoderDataset(cfg, "toy", is_valid=True)
    assert len(ds) == 3 and ds.get_dataset_name() == "toy"
    for i, m in enumerate(mels):
        item = ds[i]
        np.testing.assert_array_equal(item["mel"], m)                      # u0 was not overwritten
        assert item["mel"].dtype == np.float32 and item["target_len"] == m.shape[1]
        np.testing.assert_array_equal(item["frame_pitch"], np.arange(m.shape[1], dtype=np.float32))
    np.testing.assert_array_equal(features.align_length(np.ones(3, np.float32), 5), [1, 1, 1, 0, 0])
    assert features.align_length(np.ones((2, 6)), 4).shape == (2, 4)


def test_apnet_state_dict_matches_the_reference_layout():
    """Keys, order and shapes of APNet's state dict equal the reference module's (fixture made from
    models/vocoders/gan/generator/apnet.py), so its checkpoints load unchanged."""
    from types import SimpleNamespace as NS
    from conftest import GOLDEN_APNET, load_golden_apnet
    from amphion_b200.vocoders import APNet, _vocoders
    hp, pre = GOLDEN_APNET
    g, sd = load_golden_apnet()
    model = APNet(NS(preprocess=NS(**pre), model=NS(generator="apnet", apnet=NS(**hp))))
    assert _vocoders["apnet"] is APNet
    own = model.state_dict()
    assert list(own.keys()) == list(sd.keys())
    for k, v in sd.items():
        assert tuple(own[k].shape) == tuple(v.shape), k
    model.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()}, strict=True)
    # the trunks see effective weights under the native names; R and I filters stacked
    t = model._trunk_tensors("PSP")
    assert t["conv_post.weight"].shape == (2 * 33, hp["PSP_channel"], 7) and t["conv_pre.weight"].shape == (48, 12, 5)
    w = torch.as_tensor(sd["PSP_output_I_conv.weight_v"])
    gg = torch.as_tensor(sd["PSP_output_I_conv.weight_g"])
    want = w * (gg / w.flatten(1).norm(dim=1).view(-1, 1, 1))
    torch.testing.assert_close(t["conv_post.weight"][33:], want)
    with pytest.raises(RuntimeError, match="CUDA"):
        model(torch.zeros(1, 12, 8))


def test_vocoder_inference_names_follow_the_reference_layout():
    """models/vocoders/vocoder_inference.py is a module (synthesis, load_nnvocoder); the function vocoder_inference
    lives in gan/gan_vocoder_inference.py.  The package attribute is the module whatever was imported first."""
    import types
    import amphion_b200.vocoders as v
    from amphion_b200.vocoders import load_nnvocoder, synthesis
    from amphion_b200.vocoders.gan_vocoder_inference import vocoder_inference
    assert isinstance(v.vocoder_inference, types.ModuleType) and v.vocoder_inference.synthesis is synthesis
    assert callable(vocoder_inference) and callable(load_nnvocoder)
    assert v._vocoder_forward_funcs["hifigan"] is vocoder_inference


def test_apnet_copies_and_pickles_without_native_state():
    """The two trunk handles are derived state: deepcopy / pickle rebuild them, parameters survive."""
    import copy
    import pickle
    from types import SimpleNamespace as NS
    from conftest import GOLDEN_APNET
    from amphion_b200.vocoders import APNet
    hp, pre = GOLDEN_APNET
    torch.manual_seed(1)
    model = APNet(NS(preprocess=NS(**pre), model=NS(generator="apnet", apnet=NS(**hp))))
    model.remove_weight_norm()
    for clone in (copy.deepcopy(model), pickle.loads(pickle.dumps(model))):
        assert set(clone._trunks) == {"ASP", "PSP"} and clone._trunks["ASP"]._owner is clone
        assert clone._trunks["ASP"]._handle is None
        for (ka, va), (kb, vb) in zip(model.state_dict().items(), clone.state_dict().items()):
            assert ka == kb and torch.equal(va, vb)
    # without weight norm the trunk sees the plain weights
    t = model._trunk_tensors("ASP")
    assert torch.equal(t["conv_pre.weight"], model.ASP_input_conv.weight.detach())
