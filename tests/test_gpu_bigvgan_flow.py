"""BigVGANFlowVAE's flow (ResidualCouplingBlock on the flow.cuh kernels and the layer-level conv) against float64
autograd through tests/flow_oracle.py on the module's own parameters, with ``post`` randomised (a zero ``post`` makes
the flow an identity):

  * forward and reverse outputs, and the gradients of x and of every flow parameter, at the golden config (hidden 8:
    CUDA cores) and the bench config (hidden 64: tensor cores from 64 frames on), B in {1, 3}, T on both sides of 64,
    all-ones and per-clip prefix masks, fp32 and bf16 inputs, under every precision;
  * the no-grad output is torch.equal to the grad-mode output; masked frames come out 0 with zero gradient;
  * reverse(forward(z)) recovers z; a frozen flow runs no weight-gradient kernel and gives the same input gradient;
  * bad calls raise; encode_with_grad -> sample -> flow -> a KL-shaped term plus an MR-STFT loss on
    decode_with_grad(z, do_sample=False) reaches every encoder, flow and decoder parameter."""
import os
import sys

import pytest
import torch

import flow_oracle as FO
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.losses import MultiResolutionSTFTLoss

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402

pytestmark = pytest.mark.gpu

CONFIGS = {"golden": (BIGVGAN_H["latent_dim"], BIGVGAN_H["flow_hidden_channels"]), "bench": (512, 64)}
PRECISIONS = (None, "fp32", "bf16")
# test_gpu_bigvgan_grad.GRAD_BOUND for fp32 inputs; bf16 storage alone rounds at 2^-9
GRAD_BOUND = {None: 1e-5, "fp32": 2.0 ** -14, "bf16": 2.5e-2}
BF16_BOUND = 2.5e-2
# (B, T, per-clip valid lengths or None for an all-ones mask): T on both sides of TC_MIN_ROWS = 64
SHAPES = [(1, 40, None), (3, 80, None), (3, 40, (40, 27, 9)), (3, 96, (96, 70, 33)), (1, 80, (61,))]
WGRAD_KERNELS = ("wgrad_umma_kernel", "wgrad_direct_kernel", "weight_norm_bwd", "bias_grad_cf_kernel")


@pytest.fixture(autouse=True)
def _grad_mode():
    """Other test modules turn grad mode off when they are imported; these tests need it on."""
    with torch.enable_grad():
        yield


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _randomise_post(flow, seed):
    gen = torch.Generator().manual_seed(seed)
    for n, p in flow.named_parameters():
        if ".post." in n:
            p.data = 0.3 * torch.randn(p.shape, generator=gen).to(p)


def _flow(tag, dev, seed=0):
    C, H = CONFIGS[tag]
    torch.manual_seed(seed)
    f = BV.ResidualCouplingBlock(C, H, 5, 1, 4)
    _randomise_post(f, seed + 1)
    return f.to(dev)


def _set_precision(flow, prec):
    for m in flow.modules():
        if isinstance(m, BV._WNConvBase):
            m.tc_precision = prec
    return flow


def _mask(B, T, lens, dev):
    mask = torch.zeros(B, 1, T, device=dev)
    for b in range(B):
        mask[b, :, :T if lens is None else lens[b]] = 1
    return mask


def _rel(a, ref):
    a, ref = a.double(), ref.double()
    return float((a - ref).norm() / ref.norm().clamp_min(1e-300))


def _oracle(flow, x, mask, r, reverse, H):
    sd = {"flow." + n: p.detach().double().clone().requires_grad_(True) for n, p in flow.state_dict().items()}
    xd = x.detach().double().clone().requires_grad_(True)
    y = FO.flow(sd, {"flow_hidden_channels": H}, xd, mask.double(), reverse=reverse)
    (y * r.double()).sum().backward()
    return y.detach(), xd.grad, {n[5:]: t.grad for n, t in sd.items()}


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_flow_vs_oracle(dev, tag, dtype, prec):
    C, H = CONFIGS[tag]
    f = _set_precision(_flow(tag, dev), prec)
    bound = GRAD_BOUND[prec] if dtype == torch.float32 else BF16_BOUND
    gen = torch.Generator(device=dev).manual_seed(7)
    fails, worst = [], {}
    for B, T, lens in SHAPES:
        mask = _mask(B, T, lens, dev)
        for reverse in (False, True):
            x = torch.randn(B, C, T, device=dev, generator=gen).to(dtype)
            r = torch.randn(B, C, T, device=dev, generator=gen)
            yo, gxo, gpo = _oracle(f, x, mask, r, reverse, H)
            with torch.no_grad():
                y0 = f(x, mask, reverse=reverse)
            xg = x.clone().requires_grad_(True)
            f.zero_grad(set_to_none=True)
            y = f(xg, mask, reverse=reverse)
            assert y.dtype == dtype
            assert torch.equal(y, y0), (B, T, lens, reverse)                 # no-grad = grad-mode output
            (y.float() * r).sum().backward()
            dead = mask.expand(B, C, T) == 0
            assert not y[dead].any() and not xg.grad[dead].any()            # masked frames: 0, no gradient
            errs = {"out": _rel(y, yo), "x": _rel(xg.grad, gxo)}
            for n, p in f.named_parameters():
                errs[n] = _rel(p.grad, gpo[n])
            for k, e in errs.items():
                key = k if k in ("out", "x") else k.split(".", 2)[-1]
                worst[key] = max(worst.get(key, 0.0), e)
                if not e <= bound:
                    fails.append(f"B {B} T {T} lens {lens} reverse {reverse} {k}: {e:.2e} > {bound:.1e}")
    print(f"{tag} {dtype} {prec}: worst out {worst['out']:.2e} x {worst['x']:.2e} params "
          f"{max(v for k, v in worst.items() if k not in ('out', 'x')):.2e}")
    assert not fails, "\n".join(fails[:40])


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_round_trip(dev, tag, prec):
    C, _ = CONFIGS[tag]
    f = _set_precision(_flow(tag, dev, seed=2), prec)
    gen = torch.Generator(device=dev).manual_seed(3)
    with torch.no_grad():
        for B, T, lens in SHAPES:
            mask = _mask(B, T, lens, dev)
            z = torch.randn(B, C, T, device=dev, generator=gen)
            zp = f(z, mask)
            assert _rel(zp, z * mask) > 1e-2                                 # not an identity
            back = f(zp, mask, reverse=True)
            assert _rel(back, z * mask) <= GRAD_BOUND[prec], (B, T, lens)


def _kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


@pytest.mark.parametrize("prec", PRECISIONS)
def test_frozen_flow_runs_no_weight_gradient(dev, prec):
    C, _ = CONFIGS["bench"]
    f = _set_precision(_flow("bench", dev, seed=4), prec)
    gen = torch.Generator(device=dev).manual_seed(4)
    x = torch.randn(2, C, 80, device=dev, generator=gen)
    mask = _mask(2, 80, (80, 50), dev)
    r = torch.randn(2, C, 80, device=dev, generator=gen)

    def step():
        xg = x.clone().requires_grad_(True)
        (f(xg, mask) * r).sum().backward()
        return xg.grad

    g_full = step()
    names_full = _kernels_of(step)
    f.requires_grad_(False)
    g_frozen = step()
    names_frozen = _kernels_of(step)
    assert torch.equal(g_full, g_frozen)
    assert any("wgrad" in n for n in names_full), sorted(names_full)
    bad = sorted(n for n in names_frozen if any(k in n for k in WGRAD_KERNELS))
    assert not bad, bad


def test_bad_calls_raise(dev):
    f = _flow("golden", dev)
    C = CONFIGS["golden"][0]
    x = torch.randn(2, C, 30, device=dev)
    mask = torch.ones(2, 1, 30, device=dev)
    with pytest.raises(NotImplementedError):
        f(x, mask, g=torch.zeros(2, 4, 1, device=dev))
    for bad in (torch.ones(2, 30, device=dev), torch.ones(2, 2, 30, device=dev), torch.ones(1, 1, 30, device=dev),
                torch.ones(2, 1, 29, device=dev)):
        with pytest.raises(ValueError):
            f(x, bad)
    with pytest.raises(ValueError):
        f(torch.randn(2, C + 2, 30, device=dev), mask)


def test_model_flow_follows_set_precision(dev):
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(BV_H()).to(dev).set_precision("bf16")
    convs = [x for n, x in m.named_modules() if n.startswith("flow.") and isinstance(x, BV._WNConvBase)]
    assert len(convs) == 4 * (2 + 8) and all(c.tc_precision == "bf16" for c in convs)
    m.set_precision(None)
    assert all(c.tc_precision is None for c in convs)


class _Attr(dict):
    __getattr__ = dict.__getitem__


def BV_H(**kw):
    return _Attr(BIGVGAN_H, causal=True, **kw)


def test_training_objective_reaches_every_parameter(dev):
    """encode_with_grad -> Gaussian sample -> flow -> the KL term of VITS's kl_loss against a standard normal prior,
    plus the MR-STFT loss of decode_with_grad(z, do_sample=False): finite, nonzero gradients on every encoder, flow and
    decoder parameter."""
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(BV_H()).to(dev)
    _randomise_post(m.flow, 11)
    gen = torch.Generator(device=dev).manual_seed(9)
    D = m.h.latent_dim
    x = 0.3 * torch.randn(2, 1, 8 * 512, device=dev, generator=gen)
    lat = m.encode_with_grad(x)
    T = lat.shape[2]
    mask = _mask(2, T, (T, T - 100), dev)
    logs_q = lat[:, D:]
    z = BV._GaussSampleFn.apply(lat, torch.randn(2, D, T, device=dev, generator=gen), D)
    z_p = m.flow(z, mask)
    kl = ((-logs_q - 0.5 + 0.5 * z_p * z_p) * mask).sum() / mask.sum()
    y = m.decode_with_grad(z, do_sample=False)
    (kl + MultiResolutionSTFTLoss()(y, x[:, :, :y.shape[2]])).backward()
    bad = [n for n, p in m.named_parameters()
           if p.grad is None or not bool(torch.isfinite(p.grad).all()) or float(p.grad.abs().max()) == 0.0]
    assert not bad, bad
