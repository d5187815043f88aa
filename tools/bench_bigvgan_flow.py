"""BigVGANFlowVAE's flow (ResidualCouplingBlock(512, 64, 5, 1, 4), bench.py's BigVGAN config) on its own: the forward
without grad, and forward + backward with every flow parameter trainable and with a frozen flow (input gradient only),
under set_precision None / "fp32" / "bf16", at B x T = 4 x 100 and 16 x 375 latent frames (8 s and 30 s clips at
12.5 Hz), fp32 input, all-ones mask.

Per case: p50 / p10 / p90 (CUDA events around each call, after warm-up; the working set stays in L2, which is how the
flow runs inside a training step), and the kernels per call from torch.profiler (a separate run), in total and per
coupling layer, with their names.  Baseline: the same forward + backward by torch eager autograd through the float64
restatement tests/flow_oracle.py run in fp32 on the same GPU (TF32 off).  Writes one JSON file (--out).

    python tools/bench_bigvgan_flow.py --out profiles/r10_bigvgan_flow.json
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

from kalle_audio_b200 import bigvgan as BV  # noqa: E402
import flow_oracle as FO  # noqa: E402

C, HIDDEN, N_FLOWS = 512, 64, 4
SIZES = [(4, 100), (16, 375)]


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


def _kernels(fn, reps=3):
    """Kernels per call and their names (torch.profiler, CUDA activities; memcpy / memset listed apart)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    kern, copies, names = 0, 0, {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name.split("(")[0][:80]
        if "memcpy" in name.lower() or "memset" in name.lower():
            copies += 1
        else:
            kern += 1
        names[name] = names.get(name, 0) + 1
    return {"kernels_per_call": kern / reps, "kernels_per_coupling_layer": kern / reps / N_FLOWS,
            "copies_and_memsets_per_call": copies / reps,
            "names_per_call": {n: c / reps for n, c in sorted(names.items())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bigvgan_flow.json")
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--no-eager", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bigvgan_flow: needs a GPU")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    flow = BV.ResidualCouplingBlock(C, HIDDEN, 5, 1, N_FLOWS)
    gen = torch.Generator().manual_seed(1)
    for n, p in flow.named_parameters():
        if ".post." in n:
            p.data = 0.3 * torch.randn(p.shape, generator=gen)
    flow = flow.to(dev)
    res = {"gpu": _gpu_info(), "config": f"ResidualCouplingBlock({C}, {HIDDEN}, 5, 1, {N_FLOWS}), fp32 input, "
           "all-ones mask, loss (flow(x, mask) * r).sum()", "cases": []}
    for B, T in SIZES:
        g = torch.Generator(device=dev).manual_seed(2)
        x = torch.randn(B, C, T, device=dev, generator=g)
        r = torch.randn(B, C, T, device=dev, generator=g)
        mask = torch.ones(B, 1, T, device=dev)

        def fwd():
            with torch.no_grad():
                flow(x, mask)

        def step():
            xg = x.detach().requires_grad_(True)
            for p in flow.parameters():
                p.grad = None
            (flow(xg, mask) * r).sum().backward()

        for prec in (None, "fp32", "bf16"):
            for m in flow.modules():
                if isinstance(m, BV._WNConvBase):
                    m.tc_precision = prec
            for mode in ("forward_no_grad", "fwd_bwd_trainable", "fwd_bwd_frozen"):
                flow.requires_grad_(mode != "fwd_bwd_frozen")
                fn = fwd if mode == "forward_no_grad" else step
                case = {"B": B, "frames": T, "precision": prec, "mode": mode}
                case.update(_time(fn, args.warmup, args.steps))
                case.update(_kernels(fn))
                res["cases"].append(case)
                print(json.dumps({k: v for k, v in case.items() if k != "names_per_call"}), flush=True)
        flow.requires_grad_(True)
        if not args.no_eager:
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
            sd = {"flow." + n: p.detach().clone().requires_grad_(True) for n, p in flow.state_dict().items()}
            hh = {"flow_hidden_channels": HIDDEN}

            def eager_fwd():
                with torch.no_grad():
                    FO.flow(sd, hh, x, mask)

            def eager():
                xe = x.detach().requires_grad_(True)
                for t in sd.values():
                    t.grad = None
                (FO.flow(sd, hh, xe, mask) * r).sum().backward()

            for mode, fn in (("forward_no_grad", eager_fwd), ("fwd_bwd_trainable", eager)):
                case = {"B": B, "frames": T, "precision": "torch eager fp32 (oracle)", "mode": mode}
                case.update(_time(fn, args.warmup, args.steps))
                case.update(_kernels(fn))
                res["cases"].append(case)
                print(json.dumps({k: v for k, v in case.items() if k != "names_per_call"}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
