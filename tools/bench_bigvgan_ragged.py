"""Ragged batches of BigVGANFlowVAE at bench.py's production-like config: one ``valid_len`` call against a loop of
single-clip calls, with the zero-padded call without ``valid_len`` for reference (not exact for the shorter clips).

    python tools/bench_bigvgan_ragged.py --out profiles/r06_bigvgan_ragged.json

Workloads (seeded): decode 16 utterances of 2-20 s of 12.5 Hz latents; encode 16 clips of 2-20 s of 16 kHz audio
(whole latent frames).
Per mode and precision: p50 / p90 ms per batch over --reps timed repetitions after --warmup untimed ones (CUDA events
around each batch; each batch ends with its outputs on the device), audio-s/s of the clips' own lengths at p50, peak
device memory of one batch (``torch.cuda.max_memory_allocated`` above what was allocated before it) and libkvae
launches per batch (``kvae_launch_count``).  The card's name and power limit are read with a read-only nvidia-smi query
in the same run."""
import argparse
import json
import os
import random
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from kalle_audio_b200 import _lib  # noqa: E402
from kalle_audio_b200 import bigvgan as BV  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


# bench.py measure_bigvgan: 16 kHz, ratio 1280 (12.5 Hz latents), latent 512, 1024 -> 16 channels, AMPBlock1 k 3/7/11
H = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
             downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
             resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
             upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
             activation="snakebeta", snake_logscale=True)
SR, RATIO = 16000, 1280


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100 * (len(v) - 1))))]


def timed(fn, reps, warmup, dev):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    _lib.lib().kvae_launch_count(1)
    fn()
    launches = int(_lib.lib().kvae_launch_count(0))
    torch.cuda.synchronize(dev)
    peak = torch.cuda.max_memory_allocated(dev) - base
    t = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize(dev)
        t.append(e0.elapsed_time(e1))
    return {"ms_p50": pct(t, 50), "ms_p90": pct(t, 90), "peak_mb": peak / 2 ** 20, "launches": launches}


def run(fns, audio_s, reps, warmup, dev):
    out = {}
    for mode, fn in fns.items():
        r = timed(fn, reps, warmup, dev)
        r["audio_s_per_s"] = audio_s / (r["ms_p50"] * 1e-3)
        out[mode] = r
    out["ragged_over_loop_p50"] = out["b_ragged"]["ms_p50"] / out["a_single_clip_loop"]["ms_p50"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=16)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="profiles/r06_bigvgan_ragged.json")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rng = random.Random(6)
    frames = [rng.randint(2 * SR // RATIO, 20 * SR // RATIO) for _ in range(args.clips)]      # 25 .. 250 frames
    # whole latent frames: on the tensor cores the encoder's strided convs take inputs that divide by their stride
    samples = [RATIO * rng.randint(2 * SR // RATIO, 20 * SR // RATIO) for _ in range(args.clips)]
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(H).eval().to(dev)
    z = torch.randn(args.clips, 512, max(frames), device=dev)
    x = 0.3 * torch.randn(args.clips, 1, max(samples), device=dev)
    for b in range(args.clips):                  # a padded batch as a caller builds it
        z[b, :, frames[b]:] = 0
        x[b, :, samples[b]:] = 0
    res = {"config": {"workload": "BigVGANFlowVAE ragged batches, bench.py measure_bigvgan config (latent 512, 1024 -> "
                                  "16 channels, rates 8/5/4/2/2/2, AMPBlock1 k 3/7/11, causal; encoder 12 -> 768 "
                                  f"channels, rates 2/2/4/4/4/5), {args.clips} clips of 2-20 s (seeded)",
                      "gpu": smi, "reps": args.reps, "warmup": args.warmup,
                      "decode_frames": frames, "encode_samples": samples,
                      "modes": {"a_single_clip_loop": "one call per clip on its own length (exact)",
                                "b_ragged": "one call with valid_len (exact per clip)",
                                "c_padded": "one call on the zero-padded batch without valid_len (reference only: "
                                            "not exact for clips shorter than the longest)"}},
           "decode": {}, "encode": {}}
    dec_s, enc_s = sum(frames) * RATIO / SR, sum(samples) / SR
    for prec in ("bf16", "fp32"):
        m.set_precision(prec)
        res["decode"][prec] = run({
            "a_single_clip_loop": lambda: [m.inference_from_latents(z[b:b + 1, :, :n], do_sample=False)
                                           for b, n in enumerate(frames)],
            "b_ragged": lambda: m.inference_from_latents(z, do_sample=False, valid_len=frames),
            "c_padded": lambda: m.inference_from_latents(z, do_sample=False)}, dec_s, args.reps, args.warmup, dev)
        res["encode"][prec] = run({
            "a_single_clip_loop": lambda: [m.extract_latents(x[b:b + 1, :, :n]) for b, n in enumerate(samples)],
            "b_ragged": lambda: m.extract_latents(x, valid_len=samples),
            "c_padded": lambda: m.extract_latents(x)}, enc_s, args.reps, args.warmup, dev)
        print(prec, json.dumps({w: {k: v["ms_p50"] for k, v in res[w][prec].items() if isinstance(v, dict)}
                                for w in ("decode", "encode")}), flush=True)
    res["config"]["audio_s"] = {"decode": dec_s, "encode": enc_s}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
