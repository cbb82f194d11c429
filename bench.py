#!/usr/bin/env python
"""bench.py — vocoder audio samples/s on B200 (BASELINE.json metric, headline = config 2).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)

Headline workload (config.workload): HiFi-GAN V1 22.05 kHz generator forward, batch 64 per GPU, 80x1024
synthetic mel (random-init weights, torch.manual_seed(1234)).  A "step" is one generator forward over the
per-GPU batch (+, when N > 1, the path's one exchange: the gather of the wav shards to rank 0 — weak scaling,
the utterance batch grows with N).  `value` times the device-resident path with CUDA events; `e2e` times the
reference-facing call (`vocoder_inference` / `sharded_vocoder_inference`) with pinned HOST buffers, H2D and D2H
inside the timed region.  One JSON line on stdout (rank 0).  The same line carries, under `also`, the other
BASELINE configs measured the same way in the same process (config 3 BigVGAN-base, config 4 mel, the config-5
BigVGAN-large shard — at N > 1 the sharded config 5 itself), and under `gpu_eager` the reference's op sequence in
eager PyTorch on the same GPU (cuDNN, TF32 off / on) as the informative same-box rival.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "vocoder_audio_samples_per_sec_22.05kHz"
UNIT = "samples/s"
HOP = 256
HP_V1 = dict(resblock="1", upsample_rates=[8, 8, 2, 2], upsample_kernel_sizes=[16, 16, 4, 4],
             upsample_initial_channel=512, resblock_kernel_sizes=[3, 7, 11],
             resblock_dilation_sizes=[[1, 3, 5]] * 3)
HP_BIGVGAN_BASE = dict(HP_V1, activation="snakebeta", snake_logscale=True)
# egs/vocoder/gan/bigvgan_large/exp_config.json:14-57 (SURVEY 8, config 5)
HP_BIGVGAN_LARGE = dict(resblock="1", upsample_rates=[4, 4, 2, 2, 2, 2], upsample_kernel_sizes=[8, 8, 4, 4, 4, 4],
                        upsample_initial_channel=1536, resblock_kernel_sizes=[3, 7, 11],
                        resblock_dilation_sizes=[[1, 3, 5]] * 3, activation="snakebeta", snake_logscale=True)
# flop = SURVEY.md §8(d): conv FLOPs per output sample
WORKLOADS = {
    "hifigan_v1": dict(kind="hifigan", hp=HP_V1, n_mel=80, batch=64, frames=1024, flop=2398848,
                       label="HiFi-GAN V1 22.05kHz", config="config 2"),
    "bigvgan_base": dict(kind="bigvgan", hp=HP_BIGVGAN_BASE, n_mel=100, batch=32, frames=1024, flop=2399408,
                         label="BigVGAN-base 24kHz", config="config 3"),
    "bigvgan_large": dict(kind="bigvgan", hp=HP_BIGVGAN_LARGE, n_mel=100, batch=32, frames=2048, flop=7047456,
                          label="BigVGAN-large 24kHz", config="config 5 (per-GPU shard: 32 of 256 utterances)"),
}
N_MEL = 80   # kept for scripts that import it
DUMP_BYTES = 32 << 20   # --dump-outputs: the full config-2 waveform is 64 MiB, half of its utterances are kept


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="utterances per GPU (default: the workload's)")
    ap.add_argument("--frames", type=int, default=0)
    ap.add_argument("--precision", default=os.environ.get("AMPHION_B200_PRECISION", "tc_f16"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="only the headline workload (quick iteration)")
    ap.add_argument("--workload", default="hifigan_v1", choices=list(WORKLOADS),
                    help="headline workload of the line; hifigan_v1 = BASELINE config 2 (default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the waveform the headline workload's last timed step returned "
                         "as DIR/wav.npy (float32; beyond %d MiB a fixed seeded sample of its utterances)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native path's outputs")
    return args


def dump_output(out_dir, name, wav):
    """Write a generator output [B, 1, N] as out_dir/<name>.npy in float32.  If it is larger than DUMP_BYTES, keep
    the utterances of a fixed seeded draw (in batch order) and, should one utterance alone exceed the budget, its
    leading samples: two builds run with the same arguments then write the same selection."""
    import numpy as np
    import torch
    B, N = wav.shape[0], wav[0].numel()
    rows = min(B, max(1, DUMP_BYTES // (4 * N)))
    cols = min(N, DUMP_BYTES // (4 * rows))
    if rows < B:
        idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:rows].sort().values
        wav = wav[idx.to(wav.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), wav[..., :cols].float().cpu().numpy())


def make_cfg(workload="hifigan_v1"):
    from types import SimpleNamespace as NS
    w = WORKLOADS[workload]
    pre = NS(n_mel=w["n_mel"], hop_size=HOP, extract_amplitude_phase=False)
    return NS(preprocess=pre, model=NS(generator=w["kind"], **{w["kind"]: NS(**w["hp"])}))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"], tensor=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, source="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------
# CPU legs: the oracle port (oracle/generator.py follows the reference's hifigan.py:203-219 / bigvgan.py:313-331
# op for op on the same torch CPU primitives).  This module never imports the product on this path.
# --------------------------------------------------------------------------
_CPU_THREADS = {}


def _oracle_forward(workload):
    from oracle import generator as og
    w = WORKLOADS[workload]
    fn = og.hifigan_forward if w["kind"] == "hifigan" else og.bigvgan_forward
    return lambda params, mel: fn(params, w["hp"], mel)


def _pick_cpu_threads(workload, params, fwd, torch):
    """torch's CPU convolutions are often FASTER with fewer threads than cores on many-core hosts (oneDNN on small
    channel counts).  Probe a short forward at a few thread counts; the baseline of record is the fastest, and the
    all-cores rate is reported next to it."""
    if workload in _CPU_THREADS:
        return _CPU_THREADS[workload]
    ncpu = os.cpu_count() or 1
    cands = sorted({ncpu, min(ncpu, 64), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True)
    n_mel = WORKLOADS[workload]["n_mel"]
    probe = torch.randn(2, n_mel, 48, generator=torch.Generator().manual_seed(1))
    best = (float("inf"), ncpu)
    for n in cands:
        torch.set_num_threads(n)
        fwd(params, probe[:, :, :16])
        t0 = time.perf_counter()
        fwd(params, probe)
        dt = time.perf_counter() - t0
        if dt < best[0]:
            best = (dt, n)
    _CPU_THREADS[workload] = best[1]
    return best[1]


def cpu_oracle_rate(workload, batch, frames, repeats=1, all_cores_too=False):
    """samples/s of the oracle port on a [batch, n_mel, frames] slice (the generator has no cross-batch or
    long-range op, so cost is linear in batch x frames)."""
    import torch
    from oracle.params import random_generator_params
    w = WORKLOADS[workload]
    params = random_generator_params(w["kind"], w["hp"], w["n_mel"], seed=1234)
    fwd = _oracle_forward(workload)
    cores = _pick_cpu_threads(workload, params, fwd, torch)
    mel = torch.randn(batch, w["n_mel"], frames, generator=torch.Generator().manual_seed(0))
    out = {}
    for label, n in ([("all_cores", os.cpu_count() or 1)] if all_cores_too and cores != (os.cpu_count() or 1) else []) + [("best", cores)]:
        torch.set_num_threads(n)
        fwd(params, mel[:1, :, : min(frames, 32)])      # warm-up
        best = float("inf")
        for _ in range(repeats):
            t0 = time.perf_counter()
            fwd(params, mel)
            best = min(best, time.perf_counter() - t0)
        out[label] = (batch * frames * HOP / best, n, best)
    v, n, dt = out["best"]
    sample = "B=%d slice at T=%d of the workload, best of %d, %d of %d host threads (fastest probed)" % (
        batch, frames, repeats, n, os.cpu_count() or 1)
    res = dict(value=v, unit=UNIT, cores=n, kind="port", sample=sample, seconds=dt)
    if "all_cores" in out:
        res["all_cores"] = dict(value=out["all_cores"][0], cores=out["all_cores"][1], seconds=out["all_cores"][2])
    return res


def run_reference(args, rank):
    """The reference's own CPU path for the headline workload (the oracle port: identical op sequence on the same
    torch CPU primitives).  Each step is a bounded sample of the batch: 8 utterances at the full frame count."""
    if rank != 0:
        return 0
    w = WORKLOADS[args.workload]
    B, T = args.batch or w["batch"], args.frames or w["frames"]
    sb = min(8, B)
    steps = max(1, args.steps)
    per, total_t, last = [], 0.0, None
    for i in range(steps):
        last = cpu_oracle_rate(args.workload, sb, T, repeats=1, all_cores_too=(i == 0))
        if i == 0:
            first = last
        per.append(last["seconds"])
        total_t += last["seconds"] + (first.get("all_cores", {}).get("seconds", 0.0) if i == 0 else 0.0)
        if total_t > 120:      # keep the whole run within a few minutes
            steps = i + 1
            break
    ms = statistics.mean(per) * 1e3
    value = sb * T * HOP / (ms / 1e3)
    cores = last["cores"]
    sample = "each step = %d of the %d utterances of the batch at full T=%d, %d of %d host threads (fastest probed)" % (
        sb, B, T, cores, os.cpu_count() or 1)
    cb = dict(value=value, unit=UNIT, cores=cores, kind="port", sample=sample)
    if "all_cores" in first:
        cb["all_cores"] = first["all_cores"]
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=w["label"] + " generator forward, batch=%d per GPU, %dx%d synthetic mel" % (B, w["n_mel"], T),
                            global_batch=args.gpus * B, frames=T, hop=HOP, precision="fp32 (CPU)", sample=sample),
                cpu_baseline=cb,
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, f"/tmp/ab_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in open(self.path):
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons),
                    power_w_max=max(pw), samples=len(sm))


def _traffic(workload, B, T, precision, dom):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture of the same workload
    (profiles/r2_traffic.json, written by scripts/ncu_traffic.py); None when no capture matches."""
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        e = tr[workload]
        if (e["batch"], e["frames"], e["precision"]) == (B, T, precision) and dom in e["kernels"]:
            k = e["kernels"][dom]
            return k["bytes_per_launch"], "profiles/r2_traffic.json (ncu dram__bytes_read+write, mean of the %d %s launches of one forward)" % (k["launches"], dom)
    except (OSError, KeyError, ValueError, TypeError):
        pass
    return None, None


def _roofline(prof, ms_total, samples_rank_step, flop, workload, B, T, precision):
    pk = peaks()
    dom = max(prof, key=lambda k: prof[k]["ms"])
    d = prof[dom]
    tf = d["flops"] / (d["ms"] / 1e3) / 1e12 if d["ms"] > 0 else 0.0
    gbs = d["bytes"] / (d["ms"] / 1e3) / 1e9 if d["ms"] > 0 else 0.0
    hbm_bound = dom == "activation1d"     # the anti-aliased Snake is a streaming kernel
    steps_ms = ms_total
    r = dict(bound="hbm" if hbm_bound else "tensor", kernel=dom + "_kernel",
             achieved=gbs if hbm_bound else tf, peak=pk["hbm"] if hbm_bound else pk["tensor"],
             unit="GB/s" if hbm_bound else "TFLOP/s",
             frac=(gbs / pk["hbm"]) if hbm_bound else (tf / pk["tensor"]), traffic=None,
             peak_source=pk["source"] + (", copy" if hbm_bound else ", bf16 sustained"),
             launches=d["launches"], avg_launch_ms=d["ms"] / max(d["launches"], 1),
             share_of_step=d["ms"] / steps_ms,
             tensor=dict(achieved=tf, peak=pk["tensor"], unit="TFLOP/s", frac=tf / pk["tensor"]),
             hbm=dict(achieved=gbs, peak=pk["hbm"], unit="GB/s", frac=gbs / pk["hbm"],
                      note="algorithmic bytes: fp32 x read + y write (+ branch sum) + weights once"),
             classes={k: dict(launches=v["launches"], ms=round(v["ms"], 3)) for k, v in prof.items() if v["launches"]})
    r["algorithmic_bytes_per_launch"] = d["bytes"] / max(d["launches"], 1)
    r["traffic"], src = _traffic(workload, B, T, precision, dom)
    if src:
        r["traffic_source"] = src
    return r


def measure_generator(workload, args, dev, rank, world, steps, warmup, want_cpu, clocks_on_rank0=True, shape=None,
                      dump_dir=None):
    """One workload on the native path: device-resident `value` (CUDA events, max over ranks), `e2e` through the
    reference-facing call with pinned host buffers, per-class roofline from the C ABI's launch events.  With
    `dump_dir`, the output of the last timed step is written there (dump_output)."""
    import torch
    import torch.distributed as dist
    from amphion_b200.dist import sharded_vocoder_inference, _sharded_forward
    from amphion_b200.vocoders import _vocoders
    from amphion_b200.vocoders.gan_vocoder_inference import vocoder_inference

    w = WORKLOADS[workload]
    cfg = make_cfg(workload)
    torch.manual_seed(1234)
    model = _vocoders[w["kind"]](cfg).to(dev).eval()
    if w["kind"] == "bigvgan":
        gsn = torch.Generator().manual_seed(1)
        with torch.no_grad():       # alpha/beta ~ N(0, 0.3) (SURVEY 8d): the default 0 is too benign
            for n, prm in model.named_parameters():
                if n.endswith(".alpha") or n.endswith(".beta"):
                    prm.copy_((torch.randn(prm.shape, generator=gsn) * 0.3).to(dev))
    model.precision = args.precision
    B = args.batch if (args.batch and workload == args.workload) else w["batch"]
    T = args.frames if (args.frames and workload == args.workload) else w["frames"]
    if shape is not None:
        B, T = shape
    n_mel = w["n_mel"]
    mel = torch.randn(B, n_mel, T, generator=torch.Generator().manual_seed(rank)).to(dev)
    samples_step = world * B * T * HOP

    def step():
        if world > 1:   # the path's one exchange: gather of the wav shards to rank 0 (SURVEY.md §8e)
            return _sharded_forward(model, mel, world * B, rank, world, None, 0, 4)
        return model(mel)

    def barrier():
        if world > 1:
            dist.barrier()

    with torch.no_grad():
        nwarm = warmup if os.environ.get("AB_BENCH_PROFILE") else max(warmup, 3)
        for _ in range(nwarm):
            step()
        torch.cuda.synchronize()
        sampler = ClockSampler(dev.index)
        if rank == 0 and clocks_on_rank0:
            sampler.start()
        model.set_profiling(True)
        model.get_profile()
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            step()
        last = step()
        e1.record()
        torch.cuda.synchronize(); barrier()
        ms_total = e0.elapsed_time(e1)
        prof = model.get_profile()
        model.set_profiling(False)
        clocks = sampler.stop() if (rank == 0 and clocks_on_rank0) else None
        launches = model.last_launches * steps * world      # whole job (every rank runs the same pipeline)
        if dump_dir is not None and last is not None:       # ranks other than the gather's destination hold None
            dump_output(dump_dir, "wav", last)
        del last

        # ---- end to end through the reference-facing call, host buffers in, host result out ----
        mel_host = mel.cpu().pin_memory()

        def e2e_step():
            if world == 1:
                return vocoder_inference(cfg, model, mel_host, device=dev)          # H2D + forward + D2H (+ sync)
            return sharded_vocoder_inference(cfg, model, mel_host, world * B, device=dev)   # + gather to rank 0

        for _ in range(0 if os.environ.get("AB_BENCH_PROFILE") else 2):
            e2e_step()
        barrier(); torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            e2e_step()
        t1.record()
        torch.cuda.synchronize(); barrier()
        e2e_ms_total = t0.elapsed_time(t1)

    tms = torch.tensor([ms_total, e2e_ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_total_max, e2e_ms_total = tms.tolist()
    ms_step = ms_total_max / steps
    res = dict(workload=w["label"] + " generator forward, batch=%d per GPU, %dx%d synthetic mel" % (B, n_mel, T),
               baseline_config=w["config"], value=samples_step / (ms_step / 1e3), unit=UNIT, ms_per_step=ms_step,
               steps=steps, batch_per_gpu=B, frames=T,
               e2e=dict(value=samples_step / (e2e_ms_total / steps / 1e3), unit=UNIT,
                        h2d_bytes_per_step=world * B * n_mel * T * 4,
                        d2h_bytes_per_step=world * B * T * HOP * 4, ms_per_step=e2e_ms_total / steps,
                        api="vocoder_inference(cfg, model, pinned_host_mel)" if world == 1 else
                            "sharded_vocoder_inference(cfg, model, pinned_host_mel_shard, global_batch): gather to rank 0, D2H of the whole batch there"),
               gpu_launches=launches, clocks=clocks)
    if rank == 0:
        res["roofline"] = _roofline(prof, ms_total, B * T * HOP, w["flop"], workload, B, T, args.precision)
        tfl = B * T * HOP * w["flop"] / (ms_step / 1e3) / 1e12
        res["roofline"]["whole_step"] = dict(tflops=tfl, frac_of_tensor_peak=tfl / peaks()["tensor"])
        if want_cpu:
            sb, st = {"hifigan_v1": (min(2, B), T), "bigvgan_base": (1, 256), "bigvgan_large": (1, 128)}[workload]
            res["cpu_baseline"] = cpu_oracle_rate(workload, sb, st, repeats=2 if workload == "hifigan_v1" else 1,
                                                  all_cores_too=workload == "hifigan_v1")
        else:
            res["cpu_baseline"] = None
    del model, mel
    torch.cuda.empty_cache()
    return res


def measure_mel(dev, steps=10, want_cpu=True):
    """Config 4: TacotronSTFT(1024,256,1024,80,22050,0,8000).mel_spectrogram on 64 x 10 s @ 22.05 kHz."""
    import torch
    from amphion_b200 import mel as M
    from amphion_b200.stft import TacotronSTFT
    y = ((torch.rand(64, 220500, generator=torch.Generator().manual_seed(0)) * 2 - 1) * 0.9)
    yd = y.to(dev)
    taco = TacotronSTFT(1024, 256, 1024, 80, 22050, 0, 8000)
    win, basis = taco.stft_fn.fft_window, taco.mel_basis.to(dev)
    fused = os.environ.get("AMPHION_B200_MEL", "fused") != "cufft"   # what TacotronSTFT.mel_spectrogram runs

    def step():
        return M.native_stft_mel(yd, 1024, 256, 1024, win, basis, 512, 0.0, want_energy=True, fused=fused)

    for _ in range(5):
        out = step()
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(steps):
        flush.zero_()                      # inputs (56 MB) fit in L2: flush between timed iterations
        e0.record(); out = step(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    ms = statistics.median(ts)
    F = out[1].shape[-1]
    algo = yd.numel() * 4 + out[1].numel() * 4 + out[2].numel() * 4
    pk = peaks()
    # e2e: the reference-facing call with a pinned host wav; it returns CPU tensors (utils/stft.py:172)
    yh = y.pin_memory()
    for _ in range(2):
        taco.mel_spectrogram(yh)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        mel_h, en_h = taco.mel_spectrogram(yh)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) / steps * 1e3
    res = dict(workload="TacotronSTFT(1024,256,1024,80,22050,0,8000).mel_spectrogram, 64 x 10 s @ 22.05 kHz",
               baseline_config="config 4", metric="audio samples/s through the mel front end", unit=UNIT,
               value=yd.numel() / ms * 1e3, ms_per_step=ms, best_ms=min(ts), frames=int(64 * F), steps=steps,
               l2="256 MB flush between timed iterations",
               roofline=dict(bound="hbm", kernel="mel_fused_kernel" if fused else "frame_window + cuFFT R2C + mag_mel", achieved=algo / ms / 1e6,
                             peak=pk["hbm"], unit="GB/s", frac=algo / ms / 1e6 / pk["hbm"], traffic=None,
                             algorithmic_bytes=algo, peak_source=pk["source"] + ", copy"),
               e2e=dict(value=yd.numel() / e2e_ms * 1e3, unit=UNIT, ms_per_step=e2e_ms, h2d_bytes_per_step=yd.numel() * 4,
                        d2h_bytes_per_step=(mel_h.numel() + en_h.numel()) * 4,
                        api="TacotronSTFT.mel_spectrogram(pinned_host_wav) -> CPU (mel, energy)"))
    tr, src = _traffic("mel", 64, 220500, "fp32", "mel")
    if tr:
        res["roofline"]["traffic"], res["roofline"]["traffic_source"] = tr, src
    if want_cpu:
        import numpy as np
        from oracle import mel as om
        yb = y[:8].numpy()
        mb = basis.cpu().numpy()
        om.tacotron_mel(yb[:1], mb, 1024, 256, 1024)
        t0 = time.perf_counter()
        om.tacotron_mel(yb, mb, 1024, 256, 1024)
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = dict(value=yb.size / dt, unit=UNIT, cores=torch.get_num_threads(), kind="port",
                                   sample="8 of the 64 utterances (10 s each), oracle/mel.py tacotron_mel (conv-DFT as utils/stft.py:152-181)",
                                   seconds=dt)
    del flush
    torch.cuda.empty_cache()
    return res


def measure_gpu_eager(args, dev, steps=2):
    """The reference's op sequence (hifigan.py:203-219) in eager PyTorch on the same GPU — cuDNN convolutions,
    one kernel per elementwise op — with TF32 off (the parity setting) and on (what bins/vocoder/inference.py:28-30
    enables).  Informative rival, labelled separately from the CPU baseline of record."""
    import torch
    import torch.nn.functional as F
    from oracle.params import random_generator_params
    w = WORKLOADS["hifigan_v1"]
    hp = w["hp"]
    B, T = w["batch"], w["frames"]
    P = {k: torch.from_numpy(v).to(dev) for k, v in random_generator_params("hifigan", hp, w["n_mel"]).items()}
    mel = torch.randn(B, w["n_mel"], T, device=dev)

    def conv(x, name, d=1, pad=0):
        return F.conv1d(x, P[name + ".weight"], P[name + ".bias"], dilation=d, padding=pad)

    def forward(x):
        x = conv(x, "conv_pre", pad=3)
        nk = len(hp["resblock_kernel_sizes"])
        for i, (u, k) in enumerate(zip(hp["upsample_rates"], hp["upsample_kernel_sizes"])):
            x = F.leaky_relu(x, 0.1)
            x = F.conv_transpose1d(x, P[f"ups.{i}.weight"], P[f"ups.{i}.bias"], stride=u, padding=(k - u) // 2)
            xs = None
            for j in range(nk):
                kk = hp["resblock_kernel_sizes"][j]
                r = x
                for q, d in enumerate(hp["resblock_dilation_sizes"][j]):
                    xt = F.leaky_relu(r, 0.1)
                    xt = conv(xt, f"resblocks.{i * nk + j}.convs1.{q}", d, (kk * d - d) // 2)
                    xt = F.leaky_relu(xt, 0.1)
                    xt = conv(xt, f"resblocks.{i * nk + j}.convs2.{q}", 1, (kk - 1) // 2)
                    r = xt + r
                xs = r if xs is None else xs + r
            x = xs / nk
        x = F.leaky_relu(x)
        return torch.tanh(conv(x, "conv_post", pad=3))

    out = {}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    with torch.no_grad():
        for tag, tf32 in (("tf32_off", False), ("tf32_on", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            forward(mel); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                forward(mel)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[tag] = dict(ms_per_step=ms, value=B * T * HOP / ms * 1e3, unit=UNIT)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    out["what"] = ("HiFi-GAN V1, batch=%d, 80x%d: the reference's eager op sequence with torch.nn.functional on this GPU "
                   "(cuDNN), %d timed steps after 1 warm-up; weights folded (remove_weight_norm)" % (B, T, steps))
    torch.cuda.empty_cache()
    return out


def run_native(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    want_cpu = world == 1 and not args.no_cpu_baseline
    main = measure_generator(args.workload, args, dev, rank, world, args.steps, args.warmup, want_cpu,
                             dump_dir=args.dump_outputs)
    also, eager = {}, None
    if not args.no_also and not os.environ.get("AB_BENCH_PROFILE"):
        if world == 1:
            for wl in ("bigvgan_base", "bigvgan_large"):
                if wl != args.workload:
                    also[wl] = measure_generator(wl, args, dev, rank, world, 3, 3, want_cpu, clocks_on_rank0=False)
            also["mel"] = measure_mel(dev, want_cpu=want_cpu)
            # BASELINE config 1: HiFi-GAN V1, batch 1, 80x200 mel through the egs/vocoder plumbing (CPU leg timed in full)
            r = measure_generator("hifigan_v1", args, dev, rank, world, 20, 3, want_cpu, clocks_on_rank0=False, shape=(1, 200))
            r["baseline_config"] = "config 1 (batch 1, 80x200 mel; the reference runs it on the CPU)"
            also["hifigan_v1_b1_t200"] = r
            eager = measure_gpu_eager(args, dev)
        elif args.workload != "bigvgan_large":
            # BASELINE config 5: BigVGAN-large, 32 utterances per GPU, 100x2048 mel, gather to rank 0
            r = measure_generator("bigvgan_large", args, dev, rank, world, 3, 3, False, clocks_on_rank0=False)
            if rank == 0:
                r["baseline_config"] = "config 5 (batch %d sharded 32/GPU across %d GPUs, gather to rank 0)" % (32 * world, world)
                also["bigvgan_large"] = r
    if rank == 0:
        w = WORKLOADS[args.workload]
        dt = {"fp32": "f32", "tc_f16": "f16 operands, f32 accumulate (tcgen05); f32 elsewhere",
              "tc_bf16": "bf16 operands, f32 accumulate (tcgen05); f32 elsewhere"}[args.precision]
        line = dict(metric=METRIC, value=main["value"], unit=UNIT, n_gpus=world, steps=args.steps,
                    warmup=max(args.warmup, 3), ms_per_step=main["ms_per_step"], higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype=dt, data="synthetic",
                    config=dict(workload=main["workload"], global_batch=world * main["batch_per_gpu"],
                                frames=main["frames"], hop=HOP, precision=args.precision,
                                parallelism="utterance-batch sharding dp%d, gather of the wav shards to rank 0 (NCCL send/recv, chunked under the last layer)" % world
                                if world > 1 else "single GPU",
                                l2="no explicit flush: each step streams > 8 GB of stage tensors (>> 126 MB L2)"),
                    e2e=main["e2e"], gpu_launches=main["gpu_launches"], clocks=main["clocks"],
                    roofline=main["roofline"], cpu_baseline=main.get("cpu_baseline"), impl="native")
        if also:
            line["also"] = also
        if eager:
            line["gpu_eager"] = eager
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # convenience: re-launch under torchrun exactly as the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if args.impl == "reference":
        return run_reference(args, rank)
    return run_native(args, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
