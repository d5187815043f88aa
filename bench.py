#!/usr/bin/env python
"""bench.py -- throughput of the sigmaVAE / Oobleck hot path on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W                      (this repo's CUDA path)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                               (the reference's CPU arithmetic, host cores)

Workload (BASELINE.json configs[1]): SAO-shape autoencoder (channels 128, c_mults 1/2/4/8/16, strides
2/4/4/8/8, 44.1 kHz stereo, random init, synthetic audio), one step = encode -> split mean/scale ->
sample('fix') -> decode of 16 clips x 10.03 s per GPU in bf16 mode.  Batch items are independent, so N GPUs
run N independent shards with no data-path collective (weak scaling: 16 clips per GPU).

The JSON line:
  value        audio-seconds round-tripped per second, whole job, inputs resident in HBM
  e2e          same through the public module API with pinned HOST buffers: H2D of the audio and D2H of the
               decoded waveform inside the timed region
  decode_only  decode leg alone (the metric's name), same batch
  roofline     tensor-core roofline of the dominant kernel family (conv_umma2_kernel and its fused ResidualUnit
               form conv_ru2_kernel): algorithmic FLOPs of its
               launches / their CUDA-event time, against MEASURED_PEAKS.json (sustained figure: the kernel is
               timed inside a long step)
  cpu_baseline oracle port of the reference arithmetic on the host cores, bounded sample (rank 0, N=1 only)

--dump-outputs DIR writes what the last timed step of the round trip returned (rank 0's shard) as float32 .npy files:
DIR/decoded.npy [16, 2, 442368] and DIR/latent.npy [16, 64, 216], 57.5 MB together.  Weights, audio and sampler noise
come from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SAO = dict(channels=128, c_mults=[1, 2, 4, 8, 16], strides=[2, 4, 4, 8, 8], enc_latent=128, dec_latent=64,
           io_channels=2, sample_rate=44100)
CLIP_FRAMES = 216                     # 216 latent frames = 442368 samples = 10.031 s
BATCH_PER_GPU = 16
METRIC = "vae_decode_audio_sec_per_sec"
UNIT = "audio-s/s"


def sao_config():
    import helpers as H
    return H.ae_config(SAO["channels"], SAO["c_mults"], SAO["strides"], SAO["enc_latent"], SAO["dec_latent"],
                       SAO["io_channels"], SAO["sample_rate"])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"source": "measured", "hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"])}
    return {"source": "fallback", "hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def wait_first(self, timeout=8.0):
        """nvidia-smi needs up to a few seconds before its first line on an 8-GPU box: wait for it (outside any timed
        region) so that the timed region itself is covered."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        return len(self.rows)

    def stats(self, i0=0, i1=None):
        """Clocks / power / throttle reasons of the samples taken between two marks (widened by one sample on each
        side when the region was shorter than the sampling period)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        i1 = len(self.rows) if i1 is None else i1
        rows = self.rows[i0:i1]
        if len(rows) < 2:
            rows = self.rows[max(0, i0 - 1):i1 + 1]
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()


# ------------------------------------------------------------------------------------------ reference arm
def reference_decoder(device="cpu"):
    """The reference's own SAO-shape decoder (random init, seed 0) as a callable z -> waveform, plus what it is:
    kind "reference" = the UNMODIFIED reference modules imported from baseline/_ref (oracle/reference_loader.py:
    stable_audio_tools.models.autoencoders.create_autoencoder_from_config, third-party imports stubbed per SURVEY 8c);
    kind "port" = the oracle restatement (same torch kernels) when no copy of the reference travelled."""
    import torch
    import helpers as H
    from oracle import reference_loader
    torch.manual_seed(0)
    ref = reference_loader.load_reference()
    if ref is not None:
        m = ref[0].create_autoencoder_from_config(sao_config()).eval().to(device)
        for p in m.parameters():
            p.requires_grad_(False)
        return (lambda z: m.decode(z)), "reference", m
    from oracle import oobleck_oracle as O
    import kalle_audio_b200 as k
    m = k.create_autoencoder_from_config(sao_config()).eval()     # parameter container only (same init)
    dec_sd = {n: p.to(device) for n, p in H.split_sd(m.state_dict(), "decoder.").items()}
    return (lambda z: O.oobleck_decoder(dec_sd, z, SAO["strides"])), "port", None


def cpu_config0(frames=CLIP_FRAMES):
    """BASELINE configs[0] exactly: sigmaVAE (SAO-shape Oobleck) decode of ONE 10.03 s synthetic latent
    [1, 64, 216], batch 1, fp32, on the host cores (all of them).  Returns (audio_seconds, step(), threads, kind)."""
    import torch
    torch.set_grad_enabled(False)
    torch.set_num_threads(os.cpu_count() or 1)
    decode, kind, _ = reference_decoder("cpu")
    z = torch.randn(1, SAO["dec_latent"], frames, generator=torch.Generator().manual_seed(1))

    def step():
        t0 = time.perf_counter()
        y = decode(z)
        assert y.shape == (1, 2, frames * 2048)
        return time.perf_counter() - t0

    return frames * 2048 / SAO["sample_rate"], step, torch.get_num_threads(), kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    audio_s, step, threads, kind = cpu_config0()
    t_first = step()                                   # always one untimed pass (allocator, thread pool)
    frames = CLIP_FRAMES
    if t_first * (args.steps + max(args.warmup - 1, 0)) > 420.0:     # keep the whole run within a few minutes
        frames = 108
        audio_s, step, threads, kind = cpu_config0(frames)
        step()
    for _ in range(max(args.warmup - 1, 0)):
        step()
    times = [step() for _ in range(args.steps)]
    total = sum(times)
    value = audio_s * args.steps / total
    sample = (f"BASELINE configs[0]{' exactly' if frames == CLIP_FRAMES else ' at half length'}: SAO-shape decoder, 1 clip x "
              f"{frames} latent frames ({audio_s:.2f} s of 44.1 kHz stereo) per step, batch 1, fp32, torch CPU kernels on "
              f"{threads} threads, " + ("the reference's own nn.Modules (baseline/_ref)" if kind == "reference" else "oracle port")
              + "; DECODE leg only -- the CUDA arm's step is the encode+decode round trip of 16 such clips")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the CPU arm runs on rank 0's host cores only and does not grow with --gpus: compare at N=1",
    }
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(dev, steps=3):
    """The reference's own modules on the same B200 (PyTorch eager: cuDNN convs + elementwise kernels) -- the only
    existing Blackwell path, 'the number to beat' (BASELINE.md section 4.3): SAO decode of 4 clips x 10.03 s in fp32
    with TF32 off and under bf16 autocast."""
    import torch
    decode, kind, _ = reference_decoder(dev)
    B = 4
    z = torch.randn(B, SAO["dec_latent"], CLIP_FRAMES, device=dev)
    audio_s = B * CLIP_FRAMES * 2048 / SAO["sample_rate"]
    out = {"kind": kind, "sample": f"SAO decode only, {B} clips x 10.03 s, torch eager on cuda"}
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for name, ctx in (("fp32_tf32_off", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
            def step():
                if ctx is None:
                    return decode(z)
                with ctx:
                    return decode(z)
            for _ in range(2):
                step()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"value": audio_s / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    return out


def dump_outputs(out_dir, tensors):
    """name -> tensor, written as out_dir/<name>.npy in float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def workload_config(n_gpus):
    return {"workload": "BASELINE configs[1]: SAO-shape sigmaVAE encode -> sample('fix') -> decode round trip, "
                        f"{BATCH_PER_GPU} clips x 10.03 s per GPU, bf16 tensor-core mode, fp32 I/O",
            "arch": "oobleck channels=128 c_mults=[1,2,4,8,16] strides=[2,4,4,8,8] latent 128/64 stereo 44.1k",
            "clips_per_gpu": BATCH_PER_GPU, "clip_seconds": CLIP_FRAMES * 2048 / SAO["sample_rate"],
            "sharding": f"batch-sharded x{n_gpus}, no collective on the data path",
            "l2": "per-step working set (>10 GB of activations) is far larger than the 126 MB L2"}


# ------------------------------------------------------------------------------------------ CUDA arm
def run_cuda(args):
    import torch
    import torch.distributed as dist
    import kalle_audio_b200 as k
    from kalle_audio_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)

    torch.manual_seed(0)
    ae = k.create_autoencoder_from_config(sao_config()).eval().to(dev).set_precision("bf16")
    B, L = BATCH_PER_GPU, CLIP_FRAMES * 2048
    gen = torch.Generator().manual_seed(2 + rank)
    x_host = (0.1 * torch.randn(B, 2, L, generator=gen)).pin_memory()
    y_host = torch.empty(B, 2, L).pin_memory()
    x_dev = x_host.to(dev)
    audio_s_per_step = B * L / SAO["sample_rate"]

    def roundtrip(x):
        # encode -> split mean | scale -> sample('fix') in one plan call (the sampler runs in the epilogue of the
        # encoder's last conv; torch only draws the noise), then decode
        _ms, z = ae.encode_and_sample(x)
        return ae.decode(z), z

    last = {}                            # outputs of the latest step, kept only for --dump-outputs

    def step_resident():
        y, z = roundtrip(x_dev)
        if args.dump_outputs:
            last["decoded"], last["latent"] = y, z
        return y

    # end-to-end leg: the public host-buffer pipeline (kalle_audio_b200.HostPipeline) -- every step copies its input
    # from pinned host memory and its waveform back inside the timed region; the copies of consecutive steps overlap
    # the kernels (double-buffered device input, copy streams), as a serving loop over batches would run it
    pipe = k.HostPipeline(lambda xd: roundtrip(xd)[0], dev)

    def step_e2e():
        pipe.submit(x_host, y_host)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, sampler=None):
        barrier()
        i0 = sampler.mark() if sampler else 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        clocks = sampler.stats(i0, sampler.mark()) if sampler else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), clocks

    def timed_e2e(steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step_e2e()
        pipe.join()                      # the last step's device->host copy is inside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), None

    sampler = ClockSampler(local)        # started before the warm-up: nvidia-smi is slow to produce its first line
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler.wait_first()
    # roofline leg: per-step CUDA events inside the library, on the launching stream
    enc_r, dec_r = ae.encoder.runner(dev), ae.decoder.runner(dev)
    enc_r.set_profiling(True); dec_r.set_profiling(True)
    _lib.lib().kvae_launch_count(1)
    total_ms, clocks = timed(step_resident, args.steps, sampler)
    sampler.stop()
    launches = int(_lib.lib().kvae_launch_count(0))
    prof = enc_r.step_profile() + dec_r.step_profile()          # last step of the timed region
    enc_r.set_profiling(False); dec_r.set_profiling(False)

    _, z_dev = roundtrip(x_dev)
    for _ in range(2):
        ae.decode(z_dev)
    dec_ms, _ = timed(lambda: ae.decode(z_dev), args.steps)
    for _ in range(2):
        step_e2e()
    e2e_ms, _ = timed_e2e(args.steps)

    if rank == 0:
        peaks = measured_peaks()
        tc = [(ms, fl) for ms, fl, on_tc in prof if on_tc]
        tc_ms, tc_fl = sum(m for m, _ in tc), sum(f for _, f in tc)
        other_ms = sum(ms for ms, _, on_tc in prof if not on_tc)
        achieved = tc_fl / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
        # the single kernel that dominates the step: conv_ru2_kernel (fused ResidualUnit of the 128-channel stages).
        # It moves 1024 B per output row against 2*128*128*8 FLOPs (256 FLOP/B, right at the machine balance), and
        # no unit is above 60 % in ncu (profiles/r01_ncu_summary.txt); reported against the HBM roofline, with the
        # tensor figure in `tflops`.
        ru = [(prof[i][0], prof[i][1]) for i in range(len(prof) - 1)
              if prof[i + 1][0] < 0.01 and abs(prof[i][1] / max(prof[i + 1][1], 1.0) - 7.0) < 1e-6]
        ru_ms = sum(m for m, _ in ru)
        ru_rows = sum(f / (2.0 * 128 * 128 * 7) for _, f in ru)
        ru_bytes = ru_rows * 1024.0                       # bf16 operand in + fp16 skip in + fp16 stream out + bf16 operand out
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "conv_ru_traffic.json")
        if os.path.exists(tpath) and ru:
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj["dram_bytes"] / tj["rows"] * (ru_rows / len(ru))
        ru_tflops = sum(f for _, f in ru) * 8.0 / 7.0 / (ru_ms * 1e-3) / 1e12 if ru_ms > 0 else 0.0
        ru_gbs = ru_bytes / (ru_ms * 1e-3) / 1e9 if ru_ms > 0 else 0.0
        step_fl = enc_r.flops(B, L) + dec_r.flops(B, CLIP_FRAMES)
        ms_per_step = total_ms / args.steps
        value = world * audio_s_per_step * args.steps / (total_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(world),
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": world * audio_s_per_step * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": y_host.numel() * 4},
            "decode_only": {"value": world * audio_s_per_step * args.steps / (dec_ms * 1e-3), "unit": UNIT,
                            "ms_per_step": dec_ms / args.steps,
                            "tflops": dec_r.flops(B, CLIP_FRAMES) / (dec_ms / args.steps * 1e-3) / 1e12},
            # the dominant kernel: conv_ru2_kernel, the one-launch ResidualUnit of the 128-channel stages.  Dense
            # contraction => tensor roofline; `achieved` = algorithmic FLOPs of its launches (2*C*C*(7+1) per output
            # row) / their CUDA-event time.  Both measured peaks are given: `frac` against the sustained cuBLAS figure
            # (the kernel is timed inside a long, power-capped step), `frac_burst` against the burst figure BASELINE.md
            # quotes its 60 % target on.  `traffic` = ncu dram read+write bytes per launch (profiles/conv_ru_traffic.json,
            # scaled by rows); the algorithmic HBM bytes and the achieved GB/s sit beside it.
            "roofline": {
                "bound": "tensor", "kernel": "conv_ru2_kernel (one launch = one fused ResidualUnit of a 128-channel stage)",
                "achieved": ru_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": ru_tflops / peaks["bf16_tflops_sustained"],
                "peak_burst": peaks["bf16_tflops"], "frac_burst": ru_tflops / peaks["bf16_tflops"],
                "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, scaled by rows)",
                "algorithmic_bytes_per_launch": ru_bytes / len(ru) if ru else 0.0,
                "hbm_achieved_gbs": ru_gbs, "hbm_peak_gbs": peaks["hbm_gbs"], "hbm_frac": ru_gbs / peaks["hbm_gbs"],
                "launches_per_step": len(ru), "kernel_ms_per_step": ru_ms, "share_of_step": ru_ms / ms_per_step,
                "peak_source": peaks["source"] + " (MEASURED_PEAKS.json: cuBLAS bf16 sustained / burst, copy bandwidth)"},
            # the whole tcgen05 conv family (conv_umma2_kernel + conv_ru2_kernel): every tensor-core launch of the step
            "roofline_conv_family": {
                "bound": "tensor", "kernel": "conv_umma2_kernel + conv_ru2_kernel (tcgen05 conv family)",
                "achieved": achieved, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["bf16_tflops_sustained"], "frac_burst": achieved / peaks["bf16_tflops"],
                "launches_per_step": len(tc), "kernel_ms_per_step": tc_ms, "other_kernels_ms_per_step": other_ms,
                "whole_step_tflops": step_fl / (ms_per_step * 1e-3) / 1e12,
                "whole_step_frac": step_fl / (ms_per_step * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
                "whole_step_frac_burst": step_fl / (ms_per_step * 1e-3) / 1e12 / peaks["bf16_tflops"]},
        }
        line["decode_only"]["frac_burst"] = line["decode_only"]["tflops"] / peaks["bf16_tflops"]
        line["decode_only"]["frac_sustained"] = line["decode_only"]["tflops"] / peaks["bf16_tflops_sustained"]
        if world == 1 and not args.no_cpu_baseline:
            audio_s, step, threads, kind = cpu_config0()
            step()
            t = min(step() for _ in range(2))
            line["cpu_baseline"] = {"value": audio_s / t, "unit": UNIT, "cores": threads, "kind": kind,
                                    "sample": "BASELINE configs[0] exactly: SAO decode of 1 clip x 216 latent frames "
                                              f"({audio_s:.2f} s), batch 1, fp32, {threads} threads, "
                                              + ("the reference's own nn.Modules (baseline/_ref)" if kind == "reference" else "oracle port")
                                              + ", warm-up 1 + best of 2 (decode leg only)"}
        else:
            line["cpu_baseline"] = None
    # the other BASELINE configs ride on the same line (extra keys; the driver's scaling run then carries the
    # north-star's sharding config -- configs[2], strong scaling -- and the training config at every N)
    extra = {}
    if not args.main_only:
        del pipe
        ae.encoder._plans.clear(); ae.decoder._plans.clear()
        torch.cuda.empty_cache()
        legs = [("config3_o12_decode_strong", lambda: measure_o12_decode(args, dev, rank, world)),
                ("config5_train", lambda: measure_train(args, dev, rank, world, ae))]
        if world == 1:
            legs += [("config4_stream", lambda: measure_stream(args, dev)),
                     ("bigvgan_decode", lambda: measure_bigvgan(args, dev)),
                     ("mrstft_loss", lambda: measure_mrstft(args, dev)),
                     ("oobleck_discriminator", lambda: measure_discriminator(args, dev)),
                     ("gpu_eager_baseline", lambda: gpu_eager_baseline(dev))]
        for name, fn in legs:
            try:
                extra[name] = fn()
            except Exception as exc:                       # never lose the main line to an extra leg
                extra[name] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()
    if args.dump_outputs and rank == 0:  # after every timed leg: no file I/O between them
        dump_outputs(args.dump_outputs, last)
    last.clear()
    if rank == 0:
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ other BASELINE configs
O12 = dict(channels=128, c_mults=[1, 2, 4, 8, 16], strides=[2, 4, 4, 5, 8], io_channels=1, sample_rate=16000)


def _o12_decoder(latent, dev):
    import torch
    import kalle_audio_b200 as k
    torch.manual_seed(0)
    dec = k.OobleckDecoder(out_channels=1, channels=O12["channels"], latent_dim=latent, c_mults=O12["c_mults"],
                           strides=O12["strides"], use_snake=True, final_tanh=False).eval().to(dev)
    return dec.set_precision("bf16")


def _sync(dev, world):
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)


def measure_o12_decode(args, dev, rank, world):
    """BASELINE configs[2]: vae_12_5_dim1024-shape decoder (latent 512), 64 clips x 30 s in total, batch-sharded over
    the ranks (STRONG scaling: 64 / N clips per GPU, no collective on the data path), decode only."""
    import torch
    import torch.distributed as dist
    from kalle_audio_b200.sharding import shard_bounds
    torch.set_grad_enabled(False)
    latent, total_clips, T = 512, 64, 375
    dec = _o12_decoder(latent, dev)
    lo, hi = shard_bounds(total_clips, world, rank)
    z = torch.randn(hi - lo, latent, T, generator=torch.Generator().manual_seed(1 + rank)).to(dev)
    mb = args.micro_batch or (hi - lo)

    def step():
        for i in range(0, hi - lo, mb):
            dec(z[i:i + mb])

    for _ in range(max(args.warmup, 3)):
        step()
    _sync(dev, world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    _sync(dev, world)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    audio_s = total_clips * T * 1280 / O12["sample_rate"]
    flops = dec.runner(dev).flops(1, T) * total_clips
    t = float(ms.item()) / args.steps * 1e-3
    peaks = measured_peaks()
    tfl = flops / t / 1e12 / world
    return {"metric": METRIC, "value": audio_s / t, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "tflops_per_gpu": tfl, "frac_burst": tfl / peaks["bf16_tflops"], "frac_sustained": tfl / peaks["bf16_tflops_sustained"],
            "clips_per_gpu": hi - lo,
            "config": {"workload": "BASELINE configs[2]: O12 latent-512 (dim1024) decoder, 64 clips x 30 s, "
                                   f"batch-sharded {total_clips // world} per GPU, micro-batch {mb}, bf16 mode"}}


def measure_stream(args, dev):
    """BASELINE configs[3]: vae_12_5hz_dim2048-shape decoder (latent 1024), batch 1, decode_audio(chunked=True,
    chunk_size=128, overlap=32) semantics over T=375 -- per-chunk latency, first-chunk wall time, real-time factor;
    CUDA-graph replay on.  Plus the stateful incremental decoder when the library has it."""
    import torch
    import kalle_audio_b200 as k
    torch.set_grad_enabled(False)
    latent, T, chunk, overlap = 1024, 375, 128, 32
    dec = _o12_decoder(latent, dev)
    ae = k.AudioAutoencoder(None, dec, latent_dim=latent, downsampling_ratio=1280, sample_rate=16000, io_channels=1)
    dec.enable_cuda_graphs(True)
    z = torch.randn(1, latent, T, generator=torch.Generator().manual_seed(1)).to(dev)
    for _ in range(max(args.warmup, 3)):
        ae.decode_audio(z, chunked=True, overlap=overlap, chunk_size=chunk)
        dec(z[:, :, :chunk])
    torch.cuda.synchronize(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    for _ in range(args.steps):
        dec(z[:, :, :chunk])                      # one chunk, as a streaming caller would issue it
    ev[1].record()
    for _ in range(args.steps):
        ae.decode_audio(z, chunked=True, overlap=overlap, chunk_size=chunk)   # all 4 windows in one batched call
    ev[2].record()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    y = dec(z[:, :, :chunk])
    y[0, 0, :8].cpu()
    first_wall = time.perf_counter() - t0
    # streaming decoders, hop 96 frames (= chunk - overlap, the reference's hop): the stateful engine of libkvae
    # (persistent per-layer halo state, 0 % recompute, one CUDA graph per hop) and the exact-context window engine
    zz = torch.randn(1, latent, 96 * 12, generator=torch.Generator().manual_seed(5)).to(dev)
    hop_ms = {}
    for name, stateful in (("stateful", True), ("windows", False)):
        sdec = k.StreamingDecoder(dec, hop=chunk - overlap, stateful=stateful)
        for i in range(4):
            sdec.push(zz[:, :, i * 96:(i + 1) * 96])
        torch.cuda.synchronize(dev)
        es = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        es[0].record()
        for i in range(4, 12):
            sdec.push(zz[:, :, i * 96:(i + 1) * 96])
        es[1].record()
        torch.cuda.synchronize(dev)
        hop_ms[name] = es[0].elapsed_time(es[1]) / 8
        if stateful:
            lookahead = sdec.lookahead
        sdec.flush()
    stream_hop_ms = hop_ms["windows"]
    sdec = k.StreamingDecoder(dec, hop=chunk - overlap, stateful=False)
    chunk_ms = ev[0].elapsed_time(ev[1]) / args.steps
    full_ms = ev[1].elapsed_time(ev[2]) / args.steps
    audio_s = T * 1280 / 16000
    flops_chunk = dec.runner(dev).flops(1, chunk)
    peaks = measured_peaks()
    return {"metric": METRIC, "value": audio_s / (full_ms * 1e-3), "unit": UNIT, "n_gpus": 1,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": full_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "per_chunk_ms": chunk_ms,
            "per_chunk_tflops": flops_chunk / (chunk_ms * 1e-3) / 1e12,
            "per_chunk_frac_burst": flops_chunk / (chunk_ms * 1e-3) / 1e12 / peaks["bf16_tflops"],
            "first_chunk_wall_ms_incl_d2h": first_wall * 1e3,
            "real_time_factor_per_chunk": (chunk - overlap) * 1280 / 16000 / (chunk_ms * 1e-3),
            "stateful_stream": {"hop_frames": chunk - overlap, "ms_per_hop": hop_ms["stateful"], "recompute_factor": 1.0,
                                "lookahead_samples": lookahead,
                                "tflops": dec.runner(dev).flops(1, chunk - overlap) / (hop_ms["stateful"] * 1e-3) / 1e12,
                                "real_time_factor": (chunk - overlap) * 1280 / 16000 / (hop_ms["stateful"] * 1e-3),
                                "engine": "kvae_decode_stream_push: persistent per-layer halo state, one CUDA graph per hop"},
            "exact_context_stream": {"hop_frames": chunk - overlap, "window_frames": chunk - overlap + sdec.left + sdec.right,
                                     "ms_per_hop": stream_hop_ms, "recompute_factor": sdec.recompute_factor,
                                     "real_time_factor": (chunk - overlap) * 1280 / 16000 / (stream_hop_ms * 1e-3)},
            "config": {"workload": "BASELINE configs[3]: O12 latent-1024 (dim2048) decoder, batch 1, "
                                   "chunked decode chunk 128 / overlap 32 over T=375 (4 windows), "
                                   "CUDA-graph replay, bf16 mode"}}


def measure_bigvgan(args, dev):
    """SURVEY section 8(f) item 2: the reference's 12.5 Hz VAE, BigVGANFlowVAE.inference_from_latents
    (backup/flows.py:498-529), at a production-like synthetic config (the reference ships no config json): 16 kHz mono,
    ratio 1280 = 8*5*4*2*2*2, latent 512, channels 1024 -> 16, AMPBlock1 with kernels 3/7/11 and dilations 1/3/5,
    causal, snakebeta.  2 clips x 30 s, decode only."""
    import torch
    from kalle_audio_b200 import bigvgan as BV

    class AttrDict(dict):
        __getattr__ = dict.__getitem__

    h = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
                 downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
                 resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
                 upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
                 activation="snakebeta", snake_logscale=True)
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(h).eval().to(dev)
    B, T = 2, 375
    z = torch.randn(B, 512, T, device=dev)
    # algorithmic FLOPs: 2 * Cin * Cout * K per output sample of every conv / transposed conv (per input sample)
    fl, L, ch = 2.0 * 512 * 1024 * 7 * T, T, 1024
    for u, k in zip(h.upsample_rates, h.upsample_kernel_sizes):
        fl += 2.0 * ch * (ch // 2) * k * L
        L, ch = L * u, ch // 2
        fl += sum(2.0 * ch * ch * rk * L * 2 * 3 for rk in h.resblock_kernel_sizes)
    fl += 2.0 * ch * 1 * 7 * L
    out = {"config": {"workload": "BigVGANFlowVAE.inference_from_latents, synthetic 12.5 Hz config (latent 512, 1024 -> 16 "
                                  f"channels, rates 8/5/4/2/2/2, AMPBlock1 k 3/7/11), {B} clips x 30 s, decode only"},
           "gflop_per_clip": fl / 1e9}
    audio_s = B * T * 1280 / 16000
    for prec in ("bf16", "fp32"):
        m.set_precision(prec)
        for _ in range(2):
            m.inference_from_latents(z, do_sample=False)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = max(2, args.steps // 2)
        for _ in range(n):
            m.inference_from_latents(z, do_sample=False)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / n
        out[prec + "_mode"] = {"value": audio_s / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                               "tflops": B * fl / (ms * 1e-3) / 1e12}
    return out


def measure_mrstft(args, dev):
    """SURVEY section 8(f) item 4 (loss half): the spectral loss of the reference's autoencoder training wrapper
    (SumAndDifferenceSTFTLoss with the 7 resolutions 2048 .. 32 and A-weighting, training/autoencoders.py:123-129) at the
    training batch of BASELINE configs[4] (4 clips x 5.016 s stereo): value + gradient w.r.t. the decoded signal through
    kvae_mrstft_loss, next to the same loss written with torch.stft (cuFFT) + autograd on the same GPU."""
    import torch
    import kalle_audio_b200 as k
    A = dict(fft_sizes=[2048, 1024, 512, 256, 128, 64, 32], hop_sizes=[512, 256, 128, 64, 32, 16, 8],
             win_lengths=[2048, 1024, 512, 256, 128, 64, 32], perceptual_weighting=True, sample_rate=44100)
    mod = k.SumAndDifferenceSTFTLoss(**A)
    torch.manual_seed(0)
    B, T = 4, 221184
    x = 0.1 * torch.randn(B, 2, T, device=dev)
    y = (0.9 * x + 0.02 * torch.randn_like(x)).requires_grad_(True)
    taps = mod.fir_taps.to(dev).view(1, 1, -1)

    def ours():
        with torch.enable_grad():
            l = mod(x, y)
            l.backward()
        y.grad = None
        return l

    def eager():
        with torch.enable_grad():
            return eager_()

    def eager_():
        tot = 0.0
        for sx_, sy_ in ((x[:, 0] + x[:, 1], y[:, 0] + y[:, 1]), (x[:, 0] - x[:, 1], y[:, 0] - y[:, 1])):
            fx = torch.nn.functional.conv1d(sx_.unsqueeze(1), taps, padding=50).squeeze(1)
            fy = torch.nn.functional.conv1d(sy_.unsqueeze(1), taps, padding=50).squeeze(1)
            acc = 0.0
            for n, h in zip(A["fft_sizes"], A["hop_sizes"]):
                w = torch.hann_window(n, device=dev)
                a = torch.stft(fx, n, h, n, w, return_complex=True)
                b = torch.stft(fy, n, h, n, w, return_complex=True)
                am = torch.sqrt(torch.clamp(a.real ** 2 + a.imag ** 2, min=1e-8))
                bm = torch.sqrt(torch.clamp(b.real ** 2 + b.imag ** 2, min=1e-8))
                sc = (torch.norm(bm - am, p="fro", dim=[-1, -2]) / torch.norm(bm, p="fro", dim=[-1, -2])).mean()
                acc = acc + sc + torch.nn.functional.l1_loss(torch.log(am), torch.log(bm))
            tot = tot + acc / len(A["fft_sizes"])
        l = tot / 2
        l.backward()
        y.grad = None
        return l

    out = {"config": {"workload": f"SumAndDifferenceSTFTLoss (7 resolutions, A-weighting), {B} x 2 x {T} samples, value + "
                                  "gradient w.r.t. the decoded signal"}}
    for name, fn in (("kvae", ours), ("torch_eager_cufft", eager)):
        for _ in range(3):
            l = fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = max(3, args.steps // 2)
        for _ in range(n):
            l = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        out[name] = {"ms_fwd_bwd": e0.elapsed_time(e1) / n, "loss": float(l.detach())}
    # signal bytes one call has to touch at least: read input + target, write one gradient (fp32)
    out["hbm_floor_bytes"] = 3 * B * 2 * T * 4
    return out


def measure_discriminator(args, dev):
    """SURVEY section 8(f) item 4 (discriminator half): OobleckDiscriminator.loss of the reference's autoencoder training
    wrapper (models/discriminators.py:240-297, called at training/autoencoders.py:288) at the per-GPU training batch of
    BASELINE configs[4] (4 clips x 5.016 s stereo): the generator step (losses + gradient w.r.t. the decoded signal) and
    the discriminator step (losses + gradients of all 50.4 M parameters), next to the reference's own module in torch
    eager on the same GPU (cuDNN, torch's default conv settings) when a copy of the reference is reachable."""
    import torch
    import kalle_audio_b200.discriminators as D
    torch.manual_seed(0)
    ours = D.OobleckDiscriminator(in_channels=2)
    sd = {k: v.detach().clone() for k, v in ours.state_dict().items()}
    ours = ours.to(dev)
    B, T = 4, 221184
    reals = 0.1 * torch.randn(B, 2, T, device=dev)
    fakes = (0.9 * reals + 0.02 * torch.randn_like(reals)).requires_grad_(True)
    # multiply-adds the folded form executes (2 FLOP each), forward, both halves of the batch
    flops = 0.0
    for net, W0, T0 in [(n, 1, T >> i) for i, n in enumerate(ours.multi_discriminator.discriminators[0].layers)] + \
                       [(n, p, -(-T // p)) for n, p in zip(ours.multi_discriminator.discriminators[1].layers,
                                                           ours.multi_discriminator.discriminators[1].periods)]:
        W, t = W0, T0
        for cv in net.convs():
            Wo = (W + 2 * cv.padding - cv.kernel_size) // cv.stride + 1 if cv.two_d else 1
            t = (t + 2 * cv.padding - cv.kernel_size) // cv.stride + 1
            flops += 2.0 * 2 * B * t * (cv.out_channels * Wo) * (cv.in_channels * W) * cv.kernel_size
            W = Wo
    out = {"config": {"workload": f"OobleckDiscriminator.loss, {B} x 2 x {T} samples (reals + fakes = {2 * B} signals), fp32"},
           "fwd_flops_folded": flops}

    def steps(mod):
        params = [p for p in mod.parameters()]

        def gen_step():
            for p in params:
                p.requires_grad_(False)
            with torch.enable_grad():
                dis, gen, fm = mod.loss(reals, fakes)
                (gen + fm).backward()
            fakes.grad = None
            return gen

        def dis_step():
            for p in params:
                p.requires_grad_(True)
            with torch.enable_grad():
                dis, gen, fm = mod.loss(reals, fakes.detach())
                dis.backward()
            for p in params:
                p.grad = None
            return dis
        return (("generator_step", gen_step), ("discriminator_step", dis_step))

    mods = [("kvae", ours)]
    try:
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from oracle.reference_loader import load_reference_discriminators
        rd = load_reference_discriminators()
        if rd is not None and os.environ.get("KVAE_DISC_NO_REF", "0") != "1":
            ref = rd.OobleckDiscriminator(in_channels=2)
            ref.load_state_dict(sd)
            mods.append(("reference_torch_eager", ref.to(dev)))
    except Exception as exc:
        out["reference_torch_eager"] = {"error": f"{type(exc).__name__}: {exc}"}
    for name, mod in mods:
        res = {}
        for sname, fn in steps(mod):
            for _ in range(1 if args.steps < 4 else 2):
                l = fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            n = max(1 if args.steps < 4 else 2, args.steps // 4)
            for _ in range(n):
                l = fn()
            e1.record()
            t1 = time.perf_counter()           # host time to ISSUE the steps (no synchronisation inside the loop)
            torch.cuda.synchronize(dev)
            res[sname] = {"ms": e0.elapsed_time(e1) / n, "host_issue_ms": (t1 - t0) * 1e3 / n, "loss": float(l.detach())}
        out[name] = res
        del mod
        torch.cuda.empty_cache()
    if args.workload == "discriminator":
        # stand-alone runs only: the generator step captured once into a CUDA graph (every launch of the step goes to the
        # current stream through the C ABI, buffers come from torch's graph pool) and replayed -- the step without the
        # host's launch overhead
        try:
            for p in ours.parameters():
                p.requires_grad_(False)
            sf = fakes.detach().clone().requires_grad_(True)

            def once():
                with torch.enable_grad():
                    dis, gen, fm = ours.loss(reals, sf)
                    (gf,) = torch.autograd.grad(gen + fm, sf)
                return gen, gf
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    once()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                gen_g, gf_g = once()
            torch.cuda.synchronize(dev)
            for _ in range(2):
                graph.replay()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = max(2, args.steps // 2)
            for _ in range(n):
                graph.replay()
            e1.record()
            torch.cuda.synchronize(dev)
            out["kvae"]["generator_step_cuda_graph"] = {"ms": e0.elapsed_time(e1) / n, "loss": float(gen_g.detach())}
        except Exception as exc:
            out["kvae"]["generator_step_cuda_graph"] = {"error": f"{type(exc).__name__}: {exc}"}
    k = out["kvae"]
    out["kvae"]["generator_step"]["tflops_folded"] = 2 * flops / (k["generator_step"]["ms"] * 1e9)      # fwd + dgrad
    out["kvae"]["discriminator_step"]["tflops_folded"] = 3 * flops / (k["discriminator_step"]["ms"] * 1e9)  # + wgrad
    return out


def run_extra(args):
    """--workload o12_decode / stream as stand-alone lines (the default line carries them as extra keys)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.workload == "bigvgan":
        out = measure_bigvgan(args, dev)
    elif args.workload == "discriminator":
        out = measure_discriminator(args, dev)
    else:
        out = measure_o12_decode(args, dev, rank, world) if args.workload == "o12_decode" else measure_stream(args, dev)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_eager_baseline(args):
    import torch
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    print(json.dumps({"impl": "torch-eager (the reference's modules on cuda:0, cuDNN + eager elementwise)",
                      **gpu_eager_baseline(dev, max(args.steps, 1))}), flush=True)


def measure_train(args, dev, rank, world, ae=None):
    """BASELINE configs[4]: SAO encoder + decoder training step (encode -> vae_sample -> decode -> Gaussian NLL +
    KL -> backward -> gradient all-reduce -> AdamW), 4 clips x 5.016 s per GPU (8 GPUs = the config's global batch
    of 32), bf16 tensor-core mode with fp32 master weights.  Reports step time, trained audio-seconds per second,
    algorithmic TFLOP/s (3 x forward FLOPs) and the exposed all-reduce time (step with the all-reduce minus the
    same step without it)."""
    import torch
    import torch.distributed as dist
    import kalle_audio_b200 as k
    from kalle_audio_b200 import _lib, training as TR
    if ae is None:
        torch.manual_seed(0)
        ae = k.create_autoencoder_from_config(sao_config()).to(dev)
    ae.train()
    B, frames = args.micro_batch or 4, 108
    L = frames * 2048
    x = (0.1 * torch.randn(B, 2, L, generator=torch.Generator().manual_seed(2 + rank))).to(dev)
    noise = torch.randn(B, 64, frames, generator=torch.Generator().manual_seed(3 + rank)).to(dev)
    tr = TR.AutoencoderTrainer(ae, lr=1e-4, kl_weight=1e-4, log_sigma=-2.0, precision="bf16")

    def timed(steps):
        _sync(dev, world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            info = tr.training_step(x, noise)
        e1.record()
        _sync(dev, world)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, info

    losses = []
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    with torch.enable_grad():
        for _ in range(max(args.warmup, 3)):
            losses.append(float(tr.training_step(x, noise)["loss"]))
        _lib.lib().kvae_launch_count(1)
        sampler.wait_first()
        i0 = sampler.mark()
        ms, info = timed(args.steps)
        clocks = sampler.stats(i0, sampler.mark())
        sampler.stop()
        launches = int(_lib.lib().kvae_launch_count(0))
        losses.append(float(info["loss"]))
        ms_nosync = ms
        if world > 1:
            tr.sync.enabled = False            # same step without the gradient all-reduce (ranks diverge; timing only)
            ms_nosync, _ = timed(args.steps)
            tr.sync.enabled = True
        # the same step on the reference's spectral term instead of the Gaussian NLL (SumAndDifferenceSTFTLoss(reals,
        # decoded), training/autoencoders.py:163): its generator loss minus the GAN terms.  Timing only, after the
        # configs[4] measurement (the parameters keep moving, the workload does not).
        ms_spectral = None
        if world == 1:
            try:
                tr.spectral_loss = k.SumAndDifferenceSTFTLoss(
                    fft_sizes=[2048, 1024, 512, 256, 128, 64, 32], hop_sizes=[512, 256, 128, 64, 32, 16, 8],
                    win_lengths=[2048, 1024, 512, 256, 128, 64, 32], perceptual_weighting=True, sample_rate=SAO["sample_rate"])
                tr.nll_weight = 0.0
                for _ in range(2):
                    tr.training_step(x, noise)
                ms_spectral, _ = timed(max(3, args.steps // 2))
            except Exception as exc:
                ms_spectral = f"{type(exc).__name__}: {exc}"
            tr.spectral_loss, tr.nll_weight = None, 1.0
    peaks = measured_peaks()
    enc_r, dec_r = ae.encoder.runner(dev), ae.decoder.runner(dev)
    fwd = enc_r.flops(B, L) + dec_r.flops(B, frames)
    tfl = 3.0 * fwd / (ms * 1e-3) / 1e12
    audio_s = world * B * L / SAO["sample_rate"]
    return {
        "metric": "vae_train_audio_sec_per_sec", "value": audio_s / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[4]: SAO sigmaVAE training step fwd+bwd (Gaussian NLL + KL), "
                               f"{B} clips x {L / SAO['sample_rate']:.3f} s per GPU (global batch {B * world}), bf16 "
                               "tensor-core operands, fp32 master weights / gradients / AdamW, NCCL all-reduce of "
                               "the flat gradients overlapped with the encoder backward"},
        "clocks": clocks, "gpu_launches": launches,
        "tflops_per_gpu": tfl, "frac_of_sustained_bf16": tfl / peaks["bf16_tflops_sustained"],
        "frac_of_burst_bf16": tfl / peaks["bf16_tflops"],
        "allreduce_exposed_ms": ms - ms_nosync, "params": int(tr.flat_enc.numel() + tr.flat_dec.numel()),
        "loss_first_to_last": [losses[0], losses[-1]], "ms_per_step_mrstft_plus_kl": ms_spectral}


def run_train(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    out = measure_train(args, dev, rank, world)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["cuda", "reference"], default="cuda")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", choices=["roundtrip", "o12_decode", "stream", "train", "eager_baseline", "bigvgan", "discriminator"], default="roundtrip",
                    help="roundtrip = BASELINE configs[1] (the driver's line); o12_decode = configs[2]; stream = configs[3]; "
                         "train = configs[4]")
    ap.add_argument("--micro-batch", type=int, default=0)
    ap.add_argument("--main-only", action="store_true",
                    help="only the configs[1] line (skip the extra keys: configs[2] strong scaling, configs[3] streaming, "
                         "configs[4] training step, torch-eager GPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the decoded waveform and the sampled latent of the last timed "
                         "round-trip step as DIR/decoded.npy and DIR/latent.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "cuda" or args.workload != "roundtrip"):
        ap.error("--dump-outputs applies to the CUDA round trip (--impl cuda --workload roundtrip)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "train":
        run_train(args)
    elif args.workload == "eager_baseline":
        run_eager_baseline(args)
    elif args.workload != "roundtrip":
        run_extra(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
