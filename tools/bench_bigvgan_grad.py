"""Forward + backward of BigVGANFlowVAE's decoder (decode_with_grad) at bench.py's BigVGAN config (latent 512,
1024 -> 16 channels, rates 8/5/4/2/2/2, AMPBlock1 k 3/7/11, causal, snakebeta): B = 4 segments of 2 s and 8 s, under
"bf16" and "fp32", with every parameter trainable and with a frozen decoder (latent gradient only).

Per case: p50 / p10 / p90 of the step (CUDA events around each step, after warm-up), peak memory, and a per-kernel-class
split from torch.profiler (a separate run; the forward is profiled on its own and subtracted from the step, which splits
the tensor-core conv kernel's time into forward and data gradient).  Baseline: the same step by torch eager autograd
through oracle/bigvgan_oracle.py in fp32 on the same GPU.  Writes one JSON file (--out).

    python tools/bench_bigvgan_grad.py --out profiles/r08_bigvgan_grad.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from kalle_audio_b200 import bigvgan as BV  # noqa: E402
from oracle import bigvgan_oracle as BO  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


H = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
             downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
             resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
             upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
             activation="snakebeta", snake_logscale=True)
FRAME_RATE = 12.5

# kernel name -> class of the split
CLASSES = [("tc_conv", ("conv_umma2_kernel",)), ("tc_wgrad", ("wgrad_umma_kernel",)),
           ("cuda_core_conv", ("conv_direct_kernel",)), ("cuda_core_wgrad", ("wgrad_direct_kernel",)),
           ("aa_act_fwd", ("aa_act_kernel",)), ("aa_act_bwd", ("aa_act_bwd",)),
           ("layout_and_packing", ("cf_to_cl", "pack_weights", "split_pack", "weight_norm_fold"))]


def _class(name):
    for c, keys in CLASSES:
        if any(k in name for k in keys):
            return c
    return "elementwise_and_other"


def _gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def _time(step, warmup, steps):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms = []
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    q = statistics.quantiles(ms, n=10)
    return {"p50_ms": statistics.median(ms), "p10_ms": q[0], "p90_ms": q[-1], "steps": steps,
            "peak_mem_mib": torch.cuda.max_memory_allocated() / 2 ** 20}


def _split(fn, reps=3):
    """ms per call by kernel class (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out, names = {}, {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        c = _class(e.name)
        us = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
        out[c] = out.get(c, 0.0) + us / 1e3 / reps
        names.setdefault(c, set()).add(e.name.split("(")[0][:80])
    return out, {c: sorted(v) for c, v in names.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bigvgan_grad.json")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--seconds", type=float, nargs="+", default=[2.0, 8.0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-eager", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bigvgan_grad: needs a GPU")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(H).to(dev)
    res = {"gpu": _gpu_info(), "config": "bench.py BigVGAN h, decode_with_grad, loss (y * r).sum()", "batch": args.batch,
           "cases": []}
    for sec in args.seconds:
        T = int(round(sec * FRAME_RATE))
        g = torch.Generator(device=dev).manual_seed(1)
        x = torch.randn(args.batch, 2 * H.latent_dim, T, device=dev, generator=g)
        noise = torch.randn(args.batch, H.latent_dim, T, device=dev, generator=g)
        r = torch.randn(args.batch, 1, m.wav_length(T), device=dev, generator=g)

        def step():
            xg = x.requires_grad_(True)
            xg.grad = None
            for p in m.parameters():
                p.grad = None
            (m.decode_with_grad(xg, noise=noise) * r).sum().backward()

        def fwd():
            with torch.no_grad():
                m.decode_with_grad(x, noise=noise)

        for prec in ("bf16", "fp32"):
            m.set_precision(prec)
            for frozen in (False, True):
                m.requires_grad_(not frozen)
                case = {"seconds": sec, "frames": T, "precision": prec, "frozen": frozen}
                case.update(_time(step, args.warmup, args.steps))
                full, names = _split(step)
                fw, _ = _split(fwd)
                case["split_ms"] = {"step": full, "forward": fw,
                                    "backward": {c: full.get(c, 0.0) - fw.get(c, 0.0) for c in full}}
                case["kernels"] = names
                res["cases"].append(case)
                print(json.dumps({k: v for k, v in case.items() if k != "kernels"}), flush=True)
        m.requires_grad_(True)
        if not args.no_eager:
            sd = {n: p.detach().clone().requires_grad_(n.startswith(("conv_", "ups", "resblocks", "activation_post")))
                  for n, p in m.state_dict().items()}
            xe = x.clone().requires_grad_(True)

            def eager():
                xe.grad = None
                for t in sd.values():
                    t.grad = None
                with torch.device(dev):
                    (BO.inference_from_latents(sd, dict(H), xe, noise) * r).sum().backward()

            case = {"seconds": sec, "frames": T, "precision": "torch eager fp32 (oracle)", "frozen": False}
            case.update(_time(eager, 2, max(5, args.steps // 2)))
            res["cases"].append(case)
            print(json.dumps(case), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
