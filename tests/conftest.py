import hashlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


# The CPU oracle (oneDNN convs on small channel counts) gets slower, not faster, beyond ~16 threads: on the
# 128-thread GPU box the wide-model oracle took minutes.  Cap the threads the test process uses.
try:
    import torch
    torch.set_num_threads(min(16, os.cpu_count() or 1))
except Exception:  # pragma: no cover
    pass


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    d = {k: z[k] for k in z.files}
    sd = {k[3:]: v for k, v in d.items() if k.startswith("sd:")}
    rest = {k: v for k, v in d.items() if not k.startswith("sd:")}
    return rest, sd


# hyper-parameters of the golden fixtures (must match tests/golden/gen_golden.py)
GOLDEN_MODELS = {
    "hifigan_rb1": ("hifigan", dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4],
                                    upsample_initial_channel=64, resblock_kernel_sizes=[3, 7, 11],
                                    resblock_dilation_sizes=[[1, 3, 5]] * 3), 16),
    "hifigan_rb2": ("hifigan", dict(resblock="2", upsample_rates=[4, 4], upsample_kernel_sizes=[8, 8],
                                    upsample_initial_channel=32, resblock_kernel_sizes=[3, 5, 7],
                                    resblock_dilation_sizes=[[1, 2], [2, 6], [3, 12]]), 20),
    "bigvgan_rb1": ("bigvgan", dict(resblock="1", upsample_rates=[4, 2], upsample_kernel_sizes=[8, 4],
                                    upsample_initial_channel=64, resblock_kernel_sizes=[3, 7, 11],
                                    resblock_dilation_sizes=[[1, 3, 5]] * 3, activation="snakebeta",
                                    snake_logscale=True), 20),
    "bigvgan_rb2": ("bigvgan", dict(resblock="2", upsample_rates=[2, 2], upsample_kernel_sizes=[4, 4],
                                    upsample_initial_channel=32, resblock_kernel_sizes=[3, 5],
                                    resblock_dilation_sizes=[[1, 2], [2, 6]], activation="snake",
                                    snake_logscale=False), 12),
}


# NSF-HiFiGAN fixture (needs f0 and cfg.preprocess.sample_rate; no per-stage hooks) — tests/golden/gen_golden.py:gen_nsfhifigan
GOLDEN_NSF = ("nsfhifigan", dict(resblock="1", harmonic_num=8, upsample_rates=[4, 2, 2], upsample_kernel_sizes=[8, 4, 4],
                                 upsample_initial_channel=64, resblock_kernel_sizes=[3, 7, 11],
                                 resblock_dilation_sizes=[[1, 3, 5]] * 3), 20)


# APNet fixture (tests/golden/gen_golden.py:gen_apnet): cfg.model.apnet and cfg.preprocess
GOLDEN_APNET = (dict(ASP_channel=32, ASP_resblock_kernel_sizes=[3, 7, 11], ASP_resblock_dilation_sizes=[[1, 3, 5]] * 3,
                     ASP_input_conv_kernel_size=7, ASP_output_conv_kernel_size=7,
                     PSP_channel=48, PSP_resblock_kernel_sizes=[3, 7], PSP_resblock_dilation_sizes=[[1, 3, 5], [1, 2, 4]],
                     PSP_input_conv_kernel_size=5, PSP_output_R_conv_kernel_size=7, PSP_output_I_conv_kernel_size=7),
                dict(n_mel=12, n_fft=64, hop_size=16, win_size=64, extract_amplitude_phase=True, sample_rate=16000))


def state_dict_sha256(keys, sd):
    """Digest of a state dict: every key, its shape and its float32 bytes, in the given order."""
    h = hashlib.sha256()
    for k in keys:
        v = np.ascontiguousarray(sd[k], dtype=np.float32)
        h.update(f"{k}{v.shape}".encode())
        h.update(v.tobytes())
    return h.hexdigest()


def load_golden_apnet():
    """apnet.npz keeps the reference's inputs, outputs, state-dict key order and the SHA-256 of its weights; the
    weights themselves (1.2 MB of random initialisation) are drawn again.  APNet built under torch.manual_seed(77)
    draws the reference's initial weights (same construction order), and the output convolutions are then rescaled
    as gen_golden.py:gen_apnet did; the digest pins the result to the weights the reference ran with."""
    from types import SimpleNamespace as NS
    import torch
    from amphion_b200.vocoders import APNet
    g, _ = load_golden("apnet")
    hp, pre = GOLDEN_APNET
    torch.manual_seed(77)
    model = APNet(NS(preprocess=NS(**pre), model=NS(generator="apnet", apnet=NS(**hp))))
    gen = torch.Generator().manual_seed(78)
    with torch.no_grad():
        for conv, gain in ((model.ASP_output_conv, 3.0), (model.PSP_output_R_conv, 20.0), (model.PSP_output_I_conv, 20.0)):
            conv.weight_g.mul_(gain)
            conv.bias.copy_(torch.randn(conv.bias.shape, generator=gen) * 0.3)
    own = {k: v.numpy().copy() for k, v in model.state_dict().items()}
    keys = [str(k) for k in g.pop("sd_keys")]
    assert list(own) == keys, "APNet state-dict keys differ from the reference's"
    assert state_dict_sha256(keys, own) == str(g.pop("sd_sha256")), "APNet(seed 77) no longer draws the reference's weights"
    return g, own


# HiFiGAN_vits fixtures (positional constructor; tests/golden/gen_golden.py:gen_hifigan_vits)
GOLDEN_VITS = {
    "a": dict(initial_channel=24, resblock="1", resblock_kernel_sizes=[3, 7, 11], resblock_dilation_sizes=[[1, 3, 5]] * 3,
              upsample_rates=[4, 2], upsample_initial_channel=64, upsample_kernel_sizes=[8, 4], gin_channels=10),
    "b": dict(initial_channel=12, resblock="2", resblock_kernel_sizes=[3, 5], resblock_dilation_sizes=[[1, 2], [2, 6]],
              upsample_rates=[2, 2], upsample_initial_channel=32, upsample_kernel_sizes=[4, 4], gin_channels=0),
}


def load_golden_vits(tag):
    z = np.load(os.path.join(GOLDEN, "hifigan_vits.npz"))
    d = {k[len(tag) + 1:]: z[k] for k in z.files if k.startswith(tag + ":")}
    sd = {k[3:]: v for k, v in d.items() if k.startswith("sd:")}
    return {k: v for k, v in d.items() if not k.startswith("sd:")}, sd


@pytest.fixture(scope="session")
def golden_models():
    return GOLDEN_MODELS
