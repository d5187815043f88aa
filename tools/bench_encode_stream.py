"""Streaming encode (StreamingEncoder / kvae_encode_stream_*): ms per push, p50 / p99, with and without CUDA-graph
replay, next to what a caller does without it, all in one process:
  (a) re-encoding the exact receptive-field window per hop (``encoder`` on left + hop + right samples),
  (b) the overlapping windows of ``AudioAutoencoder.encode_audio(chunked=True)`` (128 frames, 32 overlap) over the
      whole clip,
  (c) the whole-clip encode,
and the stream's device memory (a ``torch.cuda.mem_get_info`` delta around ``begin``) against the workspace of a
whole-clip encode of the same audio (``kvae_workspace_bytes``).

    python tools/bench_encode_stream.py --out profiles/r04_encode_stream.json

Workloads: the O12 latent-1024 encoder (16 kHz mono, 30 s) with 1-frame (1 280 samples = 80 ms) and 4-frame pushes,
and the SAO encoder (44.1 kHz stereo, 30 s) with 1-frame (2 048 samples) pushes, all at B = 1.  Timing: CUDA events
around every push (the events bracket the whole push, host orchestration included).  The card's name and power limit
are read with a read-only nvidia-smi query in the same run."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import helpers as H  # noqa: E402
import kalle_audio_b200 as k  # noqa: E402
from kalle_audio_b200 import _lib  # noqa: E402


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100 * (len(v) - 1))))]


def timed(fn, n):
    ev = []
    for i in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(i)
        e1.record()
        ev.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def stream_run(enc, x, hop, graphs, skip):
    se = k.StreamingEncoder(enc, max_samples=max(hop, 8192), use_cuda_graphs=graphs)
    se.push(x[:, :, :0])
    L = _lib.lib()
    launches = []

    def push(i):
        L.kvae_launch_count(1)
        se.push(x[:, :, i * hop:(i + 1) * hop])
        launches.append(int(L.kvae_launch_count(0)))
    n = x.shape[2] // hop
    t = []
    while len(t) < 256:                      # whole passes over the clip until >= 256 steady-state pushes
        launches.clear()
        t += timed(push, n)[skip:]
        se.flush()
    res = {"hop_samples": hop, "cuda_graphs": graphs, "steady_pushes": len(t), "ms_per_push_p50": pct(t, 50),
           "ms_per_push_p99": pct(t, 99), "lookahead_samples": se.lookahead}
    if not graphs:
        res["library_kernels_per_push"] = pct(launches[skip:], 50)
    return res


def stream_memory(enc, x, hop):
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    se = k.StreamingEncoder(enc, max_samples=max(hop, 8192), use_cuda_graphs=False)
    se.push(x[:, :, :0])
    torch.cuda.synchronize()
    used = free0 - torch.cuda.mem_get_info()[0]
    se.reset()
    return used


def window_baseline(enc, x, hop, left, right, n):
    def one(j):
        e = left + 8 * hop + j * hop
        y = enc(x[:, :, e - left:e + hop + right])
        return y
    ratio = enc._ratio
    left = -(-left // ratio) * ratio
    right = -(-right // ratio) * ratio
    t = timed(one, n)[4:]
    return {"hop_samples": hop, "window_samples": left + hop + right, "ms_per_hop_p50": pct(t, 50),
            "ms_per_hop_p99": pct(t, 99)}


def measure(name, model, x, hops, sr):
    enc = model.encoder
    strides = list(H.strides_of(name))
    ratio = enc._ratio
    left, right = k.encoder_context_samples(strides)
    r = {"model": name, "sample_rate": sr, "io_channels": x.shape[1], "seconds": x.shape[2] / sr, "ratio": ratio,
         "context_left_samples": left, "context_right_samples": right}
    for hop_frames in hops:
        hop = hop_frames * ratio
        skip = right // hop + 8
        r[f"stream_{hop_frames}f_graphs"] = stream_run(enc, x, hop, True, skip)
        r[f"stream_{hop_frames}f_eager"] = stream_run(enc, x, hop, False, skip)
        r[f"a_window_recompute_{hop_frames}f"] = window_baseline(enc, x, hop, left, right, 64)
        r[f"{hop_frames}f_stream_graphs_vs_window_speedup"] = (r[f"a_window_recompute_{hop_frames}f"]["ms_per_hop_p50"] /
                                                              r[f"stream_{hop_frames}f_graphs"]["ms_per_push_p50"])
    # (b) encode_audio(chunked=True)'s windows (128 frames, 32 overlap) over the encoder itself: encode_audio proper
    # rejects these encoders, whose output is the bottleneck's mean | scale pair (2 x latent_dim channels)
    cs, ov = 128 * ratio, 32 * ratio
    chunked = lambda i: model._chunked(enc, x, cs, cs - ov, enc._out_channels_for_plan, x.shape[2] // ratio,  # noqa: E731
                                       lambda pos: pos // ratio, ov // ratio // 2)
    for _ in range(2):
        chunked(0)
    r["b_chunked_windows_128_32_ms"] = pct(timed(chunked, 5), 50)
    for _ in range(2):
        enc(x)
    r["c_whole_clip_ms"] = pct(timed(lambda i: enc(x), 5), 50)
    r["stream_device_bytes"] = stream_memory(enc, x, hops[0] * ratio)
    runner = enc.runner(x.device)
    r["whole_clip_workspace_bytes"] = int(_lib.lib().kvae_workspace_bytes(runner.handle, x.shape[0], x.shape[2]))
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=30.0)
    ap.add_argument("--out", default="profiles/r04_encode_stream.json")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"config": {"workload": "StreamingEncoder, B = 1, bf16 mode, CUDA events per push", "gpu": smi}, "runs": []}
    g = torch.Generator().manual_seed(2)
    m = H.build("o12_d1024", 0).to(dev).set_precision("bf16")
    x = (0.1 * torch.randn(1, 1, int(args.seconds * 16000) // 1280 * 1280, generator=g)).to(dev)
    res["runs"].append(measure("o12_d1024", m, x, [1, 4], 16000))
    print(json.dumps(res["runs"][-1]), flush=True)
    del m
    m = H.build("sao", 0).to(dev).set_precision("bf16")
    x = (0.1 * torch.randn(1, 2, int(args.seconds * 44100) // 2048 * 2048, generator=g)).to(dev)
    res["runs"].append(measure("sao", m, x, [1], 44100))
    print(json.dumps(res["runs"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
