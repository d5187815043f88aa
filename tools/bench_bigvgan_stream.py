"""Streaming decode of BigVGANFlowVAE (BigVGANStreamingDecoder) at bench.py's production-like config: ms per push,
time to first audio, launches per push and real-time factor, next to what a caller does without it (one
``inference_from_latents`` per hop on the exact receptive-field window) and the whole-clip decode, in one process.

    python tools/bench_bigvgan_stream.py --out profiles/r03_bigvgan_stream.json

Timing: CUDA events around every push (each push ends with its output on the device; the events bracket the whole
push, host orchestration included).  The card's name and power limit are read with a read-only nvidia-smi query."""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kalle_audio_b200 as k  # noqa: E402
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
SR, FRAME_S = 16000, 0.08


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100 * (len(v) - 1))))]


def stream_run(m, z, hop, graphs, utterances, skip):
    sd = k.BigVGANStreamingDecoder(m, max_frames=16, use_cuda_graphs=graphs)
    times, first, launches = [], None, []
    for u in range(utterances):
        ev = []
        got = 0
        for i in range(0, z.shape[2], hop):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            _lib.lib().kvae_launch_count(1)
            e0.record()
            y = sd.push(z[:, :, i:i + hop])
            e1.record()
            launches.append(int(_lib.lib().kvae_launch_count(0)))
            ev.append((e0, e1))
            got += y.shape[2]
            if first is None and got > 0:
                first = i + hop
        sd.flush()
        torch.cuda.synchronize()
        times += [a.elapsed_time(b) for a, b in ev[skip:]]
    ms50, ms99 = pct(times, 50), pct(times, 99)
    res = {"hop_frames": hop, "cuda_graphs": graphs, "steady_pushes": len(times), "ms_per_push_p50": ms50,
           "ms_per_push_p99": ms99, "rtf": hop * FRAME_S / (ms50 * 1e-3), "graph_replays": sd.graph_replays,
           "graph_captures": sd.graph_captures, "first_audio_frames": first, "lookahead_samples": sd.lookahead}
    if graphs:       # a replay issues no library call: one graph launch per push, its kernels counted in the eager run
        res["graph_launches_per_push"] = 1
    else:
        res["library_kernels_per_push"] = pct(launches[skip:], 50)
    return res


def left_context_frames(m, dev):
    """Frames before a sample's own frame that it reads: the last sample a NaN in frame f reaches."""
    T, f = 64, 8
    z = torch.randn(1, 512, T, device=dev)
    z[:, :, f] = float("nan")
    y = m.inference_from_latents(z, do_sample=False)
    last = int(torch.isnan(y.flatten()).nonzero().max())
    return last // 1280 - f


def window_baseline(m, z, hop, left, right, n_hops):
    ts = []
    for j in range(n_hops):
        e = 40 + j * hop                       # far from the clip's edges
        w0, w1 = e - left, e + hop + right
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y = m.inference_from_latents(z[:, :, w0:w1], do_sample=False)
        y = y[:, :, (e - w0) * 1280:(e - w0 + hop) * 1280].contiguous()
        e1.record()
        ts.append((e0, e1))
    torch.cuda.synchronize()
    t = [a.elapsed_time(b) for a, b in ts[3:]]
    return {"hop_frames": hop, "window_frames": left + hop + right, "ms_per_hop_p50": pct(t, 50),
            "ms_per_hop_p99": pct(t, 99), "rtf": hop * FRAME_S / (pct(t, 50) * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--out", default="profiles/r03_bigvgan_stream.json")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(H).eval().to(dev)
    T = int(round(args.seconds / FRAME_S))
    z = torch.randn(1, 512, T, device=dev)
    la = k.bigvgan_stream_geometry(H)["lookahead"]
    res = {"config": {"workload": "BigVGANStreamingDecoder, bench.py measure_bigvgan config (latent 512, 1024 -> 16 "
                                  "channels, rates 8/5/4/2/2/2, AMPBlock1 k 3/7/11, causal), B = 1, "
                                  f"{args.seconds:g} s of latents", "gpu": smi, "lookahead_samples": la,
                      "lookahead_ms": 1e3 * la / SR},
           "modes": {}}
    for prec in ("bf16", "fp32"):
        m.set_precision(prec)
        r = {}
        left = left_context_frames(m, dev)
        right = math.ceil(la / 1280)
        skip = right + 12
        for hop in (1, 4):
            r[f"stream_hop{hop}_graphs"] = stream_run(m, z, hop, True, 1 if hop == 1 else 3, skip // hop + 1)
            r[f"stream_hop{hop}_eager"] = stream_run(m, z, hop, False, 1, skip // hop + 1)
            r[f"window_recompute_hop{hop}"] = window_baseline(m, z, hop, left, right, 40)
        for key in ("stream_hop1_graphs", "stream_hop4_graphs"):
            s = r[key]
            s["library_kernels_per_graph"] = r[key.replace("graphs", "eager")]["library_kernels_per_push"]
            s["first_audio_ms"] = s["first_audio_frames"] * FRAME_S * 1e3 + s["ms_per_push_p50"]
        for _ in range(2):
            m.inference_from_latents(z, do_sample=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            m.inference_from_latents(z, do_sample=False)
        e1.record()
        torch.cuda.synchronize()
        whole = e0.elapsed_time(e1) / 3
        r["whole_clip"] = {"ms": whole, "rtf": args.seconds / (whole * 1e-3)}
        r["left_context_frames"], r["right_context_frames"] = left, right
        r["hop4_stream_vs_window_speedup"] = (r["window_recompute_hop4"]["ms_per_hop_p50"] /
                                              r["stream_hop4_graphs"]["ms_per_push_p50"])
        res["modes"][prec] = r
        print(prec, json.dumps(r), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"bf16_hop4_speedup": res["modes"]["bf16"]["hop4_stream_vs_window_speedup"],
                      "fp32_hop4_speedup": res["modes"]["fp32"]["hop4_stream_vs_window_speedup"]}))


if __name__ == "__main__":
    main()
