"""BigVGANStreamingEncoder at bench.py's BigVGAN config (16 kHz, ratio 1280, latent 512), B = 1:

    python tools/bench_bigvgan_encode_stream.py --out profiles/r07_bigvgan_encode_stream.json

Per precision ("bf16", "fp32"), over a seeded 60 s clip:
  * ms per push, p50 / p99 over every push of a whole stream (CUDA events around each push), at hops of 1 and 4
    latent frames (1280 / 5120 samples), with CUDA graphs (a second stream after one that captured them) and without;
  * library launches per push (``kvae_launch_count``, eager pushes; a graph-replayed push is one graph launch);
  * the exact-window re-encode a caller does without the stream: ``extract_latents`` of the context + lookahead window
    around each hop, p50 ms;
  * the whole-clip ``extract_latents``, p50 ms;
  * peak device memory above the model's for a 10 min clip: the whole-clip call against a hop-4 stream with graphs.
Every streamed result is checked with ``torch.equal`` against the whole-clip call.  The card's name and power limit are
read with a read-only nvidia-smi query in the same run."""
import argparse
import json
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


H = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
             downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
             resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
             upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
             activation="snakebeta", snake_logscale=True)
SR, RATIO = 16000, 1280


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100 * (len(v) - 1))))]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:          # noqa: BLE001  (recorded, not fatal)
        return f"not read: {e}"


def stream_once(se, x, hop, dev, timed):
    """One whole stream; per-push ms (CUDA events) and the concatenated latents."""
    outs, ev = [], []
    for i in range(0, x.shape[2], hop):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        outs.append(se.push(x[:, :, i:i + hop]))
        e1.record()
        ev.append((e0, e1))
    outs.append(se.flush())
    torch.cuda.synchronize(dev)
    return ([a.elapsed_time(b) for a, b in ev] if timed else None), torch.cat(outs, dim=2)


def call_ms(fn, reps, dev):
    fn()
    torch.cuda.synchronize(dev)
    t = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize(dev)
        t.append(e0.elapsed_time(e1))
    return pct(t, 50)


def peak_above(fn, dev):
    torch.cuda.synchronize(dev)
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    fn()
    torch.cuda.synchronize(dev)
    return (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 20


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07_bigvgan_encode_stream.json")
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--long-seconds", type=float, default=600.0)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(H).eval().to(dev)
    n = int(args.seconds * SR) // RATIO * RATIO
    x = 0.3 * torch.randn(1, 1, n, generator=torch.Generator().manual_seed(1)).to(dev)
    geo = k.bigvgan_encode_stream_geometry(H)
    res = {"card": card(), "config": "bench.py BigVGAN config (16 kHz, rates 2/2/4/4/4/5, latent 512), B = 1, "
                                     f"{n / SR:.1f} s clip", "lookahead_samples": geo["lookahead"],
           "context_samples": geo["context"]}
    L = _lib.lib()
    for prec in ("bf16", "fp32"):
        m.set_precision(prec)
        r = {}
        ref = m.extract_latents(x)
        r["whole_clip_ms_p50"] = call_ms(lambda: m.extract_latents(x), args.reps, dev)
        for hop_frames in (1, 4):
            hop = hop_frames * RATIO
            # the exact re-encode per hop: every sample a hop's frames read, rounded to whole frames
            W = -(-(geo["context"] + geo["lookahead"] + hop) // RATIO) * RATIO
            xw = x[:, :, :W].contiguous()
            r[f"hop{hop_frames}_exact_window_reencode_ms_p50"] = call_ms(lambda: m.extract_latents(xw), args.reps, dev)
            r[f"hop{hop_frames}_exact_window_samples"] = W
            for graphs in (False, True):
                se = k.BigVGANStreamingEncoder(m, max_samples=hop, use_cuda_graphs=graphs)
                stream_once(se, x, hop, dev, False)                 # warm-up; with graphs: captures
                caps = se.graph_captures
                L.kvae_launch_count(1)
                t, y = stream_once(se, x, hop, dev, True)
                launches = int(L.kvae_launch_count(0))
                assert torch.equal(y, ref), f"{prec} hop {hop_frames} graphs={graphs}: stream differs"
                tag = f"hop{hop_frames}_{'graphs' if graphs else 'eager'}"
                r[tag] = {"push_ms_p50": pct(t, 50), "push_ms_p99": pct(t, 99), "pushes": len(t),
                          "library_launches_per_push": launches / (len(t) + 1),
                          "graph_captures_second_stream": se.graph_captures - caps}
        # 10 min clip: peak memory above the model's, whole clip against a hop-4 stream with graphs
        nl = int(args.long_seconds * SR) // RATIO * RATIO
        xl = 0.3 * torch.randn(1, 1, nl, generator=torch.Generator().manual_seed(2)).to(dev)
        r["long_clip_s"] = nl / SR
        r["long_whole_clip_peak_mib"] = peak_above(lambda: m.extract_latents(xl), dev)
        se = k.BigVGANStreamingEncoder(m, max_samples=4 * RATIO)
        r["long_stream_hop4_peak_mib"] = peak_above(lambda: stream_once(se, xl, 4 * RATIO, dev, False), dev)
        del xl
        res[prec] = r
        print(prec, json.dumps(r, indent=1), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
