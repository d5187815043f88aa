"""Forward + backward of BigVGANFlowVAE's encoder (encode_with_grad) at bench.py's BigVGAN config (downsample channels
12 .. 768, rates 2/2/4/4/4/5, latent 512 x 2): B = 4 clips of 2 s and 8 s at 16 kHz, under "bf16" and "fp32".

Cases per clip length:
  * encoder forward + backward, loss (latents * r).sum(), every parameter trainable and with a frozen encoder (audio
    gradient only), per precision;
  * the whole autoencoder: encode_with_grad -> decode_with_grad (Gaussian sample) -> MultiResolutionSTFTLoss against
    the input, backward to every encoder and decoder parameter, per precision;
  * baseline: torch eager autograd through oracle/bigvgan_oracle.extract_latents in fp32 on the same GPU.
Per case: p50 / p10 / p90 of the step (CUDA events around each step, after warm-up) and peak memory; the encoder cases
also get a per-kernel-class split from torch.profiler in a separate run (the forward profiled on its own and
subtracted).  Writes one JSON file (--out).

    python tools/bench_bigvgan_encode_grad.py --out profiles/r09_bigvgan_encode_grad.json
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_bigvgan_grad import H, _gpu_info, _split, _time  # noqa: E402  (also puts the repository on sys.path)

from kalle_audio_b200 import bigvgan as BV  # noqa: E402
from kalle_audio_b200.losses import MultiResolutionSTFTLoss  # noqa: E402
from oracle import bigvgan_oracle as BO  # noqa: E402

SAMPLE_RATE = 16000


def _with_split(step, fwd, case):
    full, names = _split(step)
    fw, _ = _split(fwd)
    case["split_ms"] = {"step": full, "forward": fw, "backward": {c: full.get(c, 0.0) - fw.get(c, 0.0) for c in full}}
    case["kernels"] = names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bigvgan_encode_grad.json")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--seconds", type=float, nargs="+", default=[2.0, 8.0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bigvgan_encode_grad: needs a GPU")
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(H).to(dev)
    enc_params = [p for n, p in m.named_parameters() if n.startswith("audio_encoder.")]
    loss_fn = MultiResolutionSTFTLoss()
    res = {"gpu": _gpu_info(), "config": "bench.py BigVGAN h, encode_with_grad, loss (latents * r).sum(); round trip: "
           "+ decode_with_grad + MultiResolutionSTFTLoss", "batch": args.batch, "sample_rate": SAMPLE_RATE, "cases": []}

    def record(case, timing_fn, warmup=None, steps=None):
        case.update(_time(timing_fn, args.warmup if warmup is None else warmup, steps or args.steps))
        res["cases"].append(case)
        print(json.dumps({k: v for k, v in case.items() if k != "kernels"}), flush=True)

    for sec in args.seconds:
        L = int(round(sec * SAMPLE_RATE))
        g = torch.Generator(device=dev).manual_seed(1)
        x = 0.3 * torch.randn(args.batch, 1, L, device=dev, generator=g)
        F_ = m.latent_length(L)
        r = torch.randn(args.batch, 2 * H.latent_dim, F_, device=dev, generator=g)
        noise = torch.randn(args.batch, H.latent_dim, F_, device=dev, generator=g)
        xg = x.clone().requires_grad_(True)

        def zero():
            xg.grad = None
            for p in m.parameters():
                p.grad = None

        def enc_step():
            zero()
            (m.encode_with_grad(xg) * r).sum().backward()

        def enc_fwd():
            with torch.no_grad():
                m.encode_with_grad(x)

        def round_trip():
            zero()
            y = m.decode_with_grad(m.encode_with_grad(x), noise=noise)
            loss_fn(y, x[:, :, :y.shape[2]]).backward()

        base = {"seconds": sec, "samples": L, "frames": F_}
        for prec in ("bf16", "fp32"):
            m.set_precision(prec)
            for frozen in (False, True):
                m.requires_grad_(False)
                for p in ([] if frozen else enc_params):
                    p.requires_grad_(True)
                case = dict(base, what="encoder fwd+bwd", precision=prec, frozen=frozen)
                _with_split(enc_step, enc_fwd, case)
                record(case, enc_step)
            m.requires_grad_(True)
            record(dict(base, what="round trip (encode, decode, MR-STFT loss) fwd+bwd", precision=prec, frozen=False),
                   round_trip)
        sd = {n: p.detach().clone().requires_grad_(True) for n, p in m.state_dict().items()
              if n.startswith("audio_encoder.")}
        xe = x.clone().requires_grad_(True)

        def eager():
            xe.grad = None
            for t in sd.values():
                t.grad = None
            with torch.device(dev):
                (BO.extract_latents(sd, dict(H), xe) * r).sum().backward()

        record(dict(base, what="encoder fwd+bwd, torch eager autograd through the fp32 oracle",
                    precision="torch eager fp32 (oracle)", frozen=False), eager, 2, max(5, args.steps // 2))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
