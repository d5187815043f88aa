"""Development aid: SAO decode + encode at B=8 with the library KVAE_LIB names (and the kept switches of tools/README.md):
per-step CUDA-event profile summed by kernel class, plus the parity numbers against the golden anchor.  One line per run."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch

import helpers as H
import kalle_audio_b200 as k

torch.set_grad_enabled(False)
dev = torch.device("cuda:0")
tag = sys.argv[1] if len(sys.argv) > 1 else "run"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 8
g = H.golden("sao_full")
m = H.build("sao", 0).to(dev).set_precision("bf16")
z = torch.randn(1, 64, 216, generator=torch.Generator().manual_seed(1)).to(dev)
y = m.decode(z)
idx = H.t(g["dec_idx"]).long().to(dev)
err = float((y[:, :, idx].cpu() - H.t(g["dec_out_at_idx"])).abs().max())
x = (0.1 * torch.randn(1, 2, 442368, generator=torch.Generator().manual_seed(2))).to(dev)
err_e = float((m.encode(x).cpu() - H.t(g["enc_out"])).abs().max())


def prof(runner, fn):
    runner.set_profiling(True)
    best = None
    for _ in range(6):
        fn()
        torch.cuda.synchronize()
        p = runner.step_profile()
        if best is None or sum(q[0] for q in p) < sum(q[0] for q in best):
            best = p
    runner.set_profiling(False)
    return best


zb = torch.randn(B, 64, 216, device=dev)
pd = prof(m.decoder.runner(dev), lambda: m.decode(zb))
xb = 0.1 * torch.randn(B, 2, 442368, device=dev)
pe = prof(m.encoder.runner(dev), lambda: m.encode(xb))
tot_d, tot_e = sum(q[0] for q in pd), sum(q[0] for q in pe)
fl = sum(q[1] for q in pd)
# fused ResidualUnits show up as a long step followed by a ~0.003 ms placeholder step
ru_d = sum(pd[i][0] for i in range(len(pd) - 1) if pd[i + 1][0] < 0.01)
ru_e = sum(pe[i][0] for i in range(len(pe) - 1) if pe[i + 1][0] < 0.01)
print(f"AB {tag}: decode B={B} {tot_d:.3f} ms ({fl / tot_d / 1e9:.0f} TFLOP/s, fused RU {ru_d:.3f} ms)  encode {tot_e:.3f} ms "
      f"(fused RU {ru_e:.3f} ms)  parity dec {err:.2e} enc {err_e:.2e}", flush=True)
if os.environ.get("AB_STEPS"):
    for i, (ms, f, tc) in enumerate(pd):
        print(f"   dec step {i:2d} {ms:7.3f} ms {f / max(ms, 1e-9) / 1e9:8.1f} TFLOP/s")
