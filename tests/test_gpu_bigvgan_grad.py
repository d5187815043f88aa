"""Gradients through BigVGANFlowVAE's decoder (decode_with_grad) against float64 autograd through
oracle/bigvgan_oracle.py on the module's own parameters:

  * kvae_aa_act_bwd (the fused anti-aliased activation backward) across its 1024-output tiles, Snake and SnakeBeta,
    logscale on and off, fp32 and bf16 input, with bit-identical d alpha / d beta from call to call;
  * the conv backward (kvae_conv1d_win_bwd) of every conv geometry of the bench decoder on each engine it runs on, at
    the 64-row threshold and the M-tile edges;
  * the whole decoder: forward equal to inference_from_latents, gradients of the latents and of every parameter, a
    frozen decoder that runs no weight-gradient kernel, and the MR-STFT loss backpropagated through the bench model."""
import pytest
import torch
import torch.nn.functional as F

import helpers as H
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.layers import TC_MIN_ROWS
from kalle_audio_b200.losses import MultiResolutionSTFTLoss
from oracle import bigvgan_oracle as BO

import os
import sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402

pytestmark = pytest.mark.gpu


class AttrDict(dict):
    __getattr__ = dict.__getitem__


BENCH = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
                 downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
                 resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
                 upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
                 activation="snakebeta", snake_logscale=True)
# wide enough for the tensor cores (256 / 128 / 64 channels), small enough for float64 autograd per case
WIDE = AttrDict(BIGVGAN_H, upsample_initial_channel=256)
PRECISIONS = (None, "fp32", "bf16")
# per tensor relative L2: fp32 sums (None); under "fp32" the data gradients of the wide convs run on the bf16x3 split,
# whose error against the exact conv is bounded by 2^-14 A per element (test_gpu_bigvgan_reference.BOUND_EXACT; measured
# 2.5e-5 .. 3.7e-5 here), above the 1e-5 of the Oobleck training step; bf16 operands under "bf16"
GRAD_BOUND = {None: 1e-5, "fp32": 2.0 ** -14, "bf16": 2.5e-2}


@pytest.fixture(autouse=True)
def _grad_mode():
    """Other test modules turn grad mode off when they are imported; these tests need it on."""
    with torch.enable_grad():
        yield


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _model(h, dev, seed=0):
    torch.manual_seed(seed)
    m = BV.BigVGANFlowVAE(AttrDict(h)).eval()
    for n, p in m.named_parameters():               # snake parameters away from their init
        if n.endswith(("alpha", "beta")):
            p.data = 0.2 * torch.randn_like(p) if m.h.snake_logscale else 1.0 + 0.3 * torch.rand_like(p)
    return m.to(dev)


def _rel(a, ref):
    a, ref = a.double(), ref.double()
    return float((a - ref).norm() / ref.norm().clamp_min(1e-300))


class _F64:
    """float64 default dtype on a device: the oracle's alias-free filters follow it."""

    def __init__(self, dev):
        self.dev = dev

    def __enter__(self):
        self.prev = torch.get_default_dtype()
        torch.set_default_dtype(torch.float64)
        self.ctx = torch.device(self.dev)
        self.ctx.__enter__()

    def __exit__(self, *a):
        self.ctx.__exit__(*a)
        torch.set_default_dtype(self.prev)


# ------------------------------------------------------------------------------------------------- a. activation
def _act_case(dev, snake, logscale, dtype, C, B, T, gen):
    act = BV._make_act(AttrDict(activation=snake, snake_logscale=logscale), C).to(dev)
    for p in act.act.parameters():
        p.data = (0.3 * torch.randn(C, device=dev, generator=gen) if logscale else
                  1.0 + 0.3 * torch.rand(C, device=dev, generator=gen))
    x = torch.randn(B, C, T, device=dev, generator=gen).to(dtype).requires_grad_(True)
    gy = torch.randn(B, C, T, device=dev, generator=gen).to(dtype)
    params = [act.act.alpha] + ([act.act.beta] if snake == "snakebeta" else [])
    grads = []
    for _ in range(2):                              # two backward calls: the parameter gradients repeat bit for bit
        y = act(x)
        grads.append(torch.autograd.grad(y, [x] + params, gy))
    with _F64(dev):
        xd = x.detach().double().requires_grad_(True)
        sd = {"a.act.alpha": act.act.alpha.detach().double().requires_grad_(True)}
        if snake == "snakebeta":
            sd["a.act.beta"] = act.act.beta.detach().double().requires_grad_(True)
        yd = BO.aa_activation(sd, "a", xd, logscale)
        refs = torch.autograd.grad(yd, [xd] + list(sd.values()), gy.double())
    return grads, refs


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("logscale", [True, False], ids=["log", "lin"])
@pytest.mark.parametrize("snake", ["snake", "snakebeta"])
def test_aa_act_bwd_vs_float64(dev, snake, logscale, dtype):
    """gx within 1e-5 relative L2 for fp32 input (bf16: the bf16 rounding of the stored gradient), d alpha / d beta
    within 1e-5; T covers one row below the halo and the 1024-output tile edges."""
    gen = torch.Generator(device=dev).manual_seed(1)
    gx_bound = 1e-5 if dtype == torch.float32 else 8e-3
    worst, fails = {}, []
    for C in (6, 96):
        for B in (1, 3):
            for T in (1, 5, 11, 1023, 1024, 1025, 3000):
                grads, refs = _act_case(dev, snake, logscale, dtype, C, B, T, gen)
                case = f"C={C} B={B} T={T}"
                for i, name in enumerate(["gx", "dalpha", "dbeta"][:len(refs)]):
                    e = _rel(grads[0][i], refs[i])
                    worst[name] = max(worst.get(name, 0.0), e)
                    if e > (gx_bound if i == 0 else 1e-5):
                        fails.append(f"{case}: {name} rel L2 {e:.2e}")
                for i in range(1, len(refs)):
                    if not torch.equal(grads[0][i], grads[1][i]):
                        fails.append(f"{case}: parameter gradient {i} differs between two calls")
    H.report(f"aa_act_bwd {snake} {'log' if logscale else 'lin'} {dtype}: worst rel L2",
             ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    assert not fails, "\n".join(fails[:30])


# ------------------------------------------------------------------------------------------------- b. conv layers
def _q_rows(m, T):
    K, s, d, p = m.kernel_size[0], m.stride[0], m.dilation[0], m.padding[0]
    if m.transposed:
        keep = T * s if getattr(m, "_drop", 0) else (T - 1) * s - 2 * p + K
        return -(-keep // s)
    return T if getattr(m, "causal", False) and K > 1 else T + 2 * p - d * (K - 1)


def _lengths(m):
    """the 64-row threshold and inputs whose output rows per stride phase are 127 / 128 / 129 (M-tile edges)"""
    out = [TC_MIN_ROWS]
    for tq in (127, 128, 129):
        out.append(next(T for T in range(TC_MIN_ROWS, 4 * tq) if _q_rows(m, T) == tq))
    return out


def _conv_layer64(m, x, v, g, bias):
    w = v * (g / v.flatten(1).norm(dim=1).view(-1, 1, 1))
    K, s, d, p = m.kernel_size[0], m.stride[0], m.dilation[0], m.padding[0]
    if m.transposed:
        y = F.conv_transpose1d(x, w, bias, stride=s, padding=p)
        return y[:, :, :-m._drop] if m._drop else y
    y = F.conv1d(x, w, bias, padding=p, dilation=d)
    return y[:, :, :x.shape[2]] if m.causal and K > 1 else y


# per tensor relative L2 against float64, from each engine's rounding: fp32 sums (engine 0, and the CUDA-core weight
# gradient of engine 2), the bf16x3 split (engine 2's data gradient: 2^-14, test_gpu_bigvgan_reference.BOUND_EXACT),
# bf16 operands (engine 1: about 2^-9 per product, measured 2.4e-3 .. 3.7e-3)
CONV_BOUND = {0: {"gx": 1e-5, "w": 1e-5}, 2: {"gx": 2.0 ** -14, "w": 1e-5}, 1: {"gx": 1e-2, "w": 1e-2}}


@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
def test_conv_backward_per_engine(dev, causal):
    model = _model(dict(BENCH, causal=causal), dev)
    ops, _ = BV._program(model.h)
    mods = {}
    for op in ops:
        if op.kind in ("conv", "convT"):
            m = BV._module(model, op.module)
            key = (m.transposed, m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0], m.dilation[0])
            mods.setdefault(key, (op.module, m))
    gen = torch.Generator(device=dev).manual_seed(2)
    worst, fails = {}, []
    for tag, m in mods.values():
        m.tc_precision = "fp32"
        precs = PRECISIONS if m.tc_layer() else (None,)
        for T in _lengths(m):
            x = torch.randn(2, m.in_channels, T, device=dev, generator=gen)
            with _F64(dev):
                xd = x.double().requires_grad_(True)
                vd, gd = m.weight_v.detach().double().requires_grad_(True), m.weight_g.detach().double().requires_grad_(True)
                bd = m.bias.detach().double().requires_grad_(True)
                yd = _conv_layer64(m, xd, vd, gd, bd)
                r = torch.randn(yd.shape, device=dev, generator=gen, dtype=torch.float64)
                refs = torch.autograd.grad(yd, [xd, gd, vd, bd], r)
            for prec in precs:
                m.tc_precision = prec
                e_id = 0 if prec is None or T < TC_MIN_ROWS else (1 if prec == "bf16" else 2)
                xg = x.clone().requires_grad_(True)
                with torch.enable_grad():
                    y = m(xg)
                    got = torch.autograd.grad(y, [xg, m.weight_g, m.weight_v, m.bias], r.float())
                for name, a, ref in zip(("gx", "dg", "dv", "dbias"), got, refs):
                    e = _rel(a, ref)
                    kind = "gx" if name == "gx" else "w"
                    worst[(e_id, name)] = max(worst.get((e_id, name), 0.0), e)
                    if e > CONV_BOUND[e_id][kind]:
                        fails.append(f"{tag} T={T} engine {e_id}: {name} rel L2 {e:.2e}")
        m.tc_precision = "fp32"
    H.report(f"BigVGAN conv backward {'causal' if causal else 'noncausal'}: worst rel L2",
             ", ".join(f"e{e} {n} {v:.2e}" for (e, n), v in sorted(worst.items())))
    assert not fails, "\n".join(fails[:40])


# ------------------------------------------------------------------------------------------------- c. whole decoder
def _decoder_params(m):
    return [(n, p) for n, p in m.named_parameters() if not n.startswith(("flow.", "audio_encoder."))]


def _oracle_grads(m, x, noise, r):
    with _F64(x.device):
        sd = {n: p.detach().double() for n, p in m.state_dict().items()}
        leaves = {n: sd[n].requires_grad_(True) for n, _ in _decoder_params(m)}
        xd = x.detach().double().requires_grad_(True)
        y = BO.inference_from_latents(sd, dict(m.h), xd, noise.double())
        gs = torch.autograd.grad((y * r.double()).sum(), [xd] + list(leaves.values()))
    return gs[0], dict(zip(leaves, gs[1:]))


@pytest.mark.parametrize("activation", ["snake", "snakebeta"])
@pytest.mark.parametrize("resblock", ["1", "2"])
@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
def test_decode_with_grad_vs_oracle(dev, causal, resblock, activation):
    h = dict(WIDE, causal=causal, resblock=resblock, activation=activation)
    m = _model(h, dev)
    gen = torch.Generator(device=dev).manual_seed(3)
    x = torch.randn(2, 2 * h["latent_dim"], 70, device=dev, generator=gen)
    noise = torch.randn(2, h["latent_dim"], 70, device=dev, generator=gen)
    r = None
    fails, worst = [], {}
    for prec in PRECISIONS:
        m.set_precision(prec)
        ref_y = m.inference_from_latents(x, noise=noise)
        xg = x.clone().requires_grad_(True)
        for p in m.parameters():
            p.grad = None
        y = m.decode_with_grad(xg, noise=noise)
        if not torch.equal(y.detach(), ref_y):
            fails.append(f"{prec}: decode_with_grad output differs from inference_from_latents")
        if r is None:
            r = torch.randn(y.shape, device=dev, generator=gen)
            ref_gx, ref_gp = _oracle_grads(m, x, noise, r)
        (y * r).sum().backward()
        for name, got, ref in [("latents", xg.grad, ref_gx)] + [(n, p.grad, ref_gp[n]) for n, p in _decoder_params(m)]:
            if got is None:
                fails.append(f"{prec}: {name} has no gradient")
                continue
            e = _rel(got, ref)
            worst[prec] = max(worst.get(prec, 0.0), e)
            if e > GRAD_BOUND[prec]:
                fails.append(f"{prec}: {name} rel L2 {e:.2e}")
    H.report(f"decode_with_grad {'causal' if causal else 'noncausal'} resblock {resblock} {activation}: worst rel L2",
             ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    assert not fails, "\n".join(fails[:40])


WGRAD_KERNELS = ("wgrad_umma_kernel", "wgrad_direct_kernel", "weight_norm_bwd", "bias_grad_cf_kernel",
                 "aa_act_bwd_params_kernel")


def _kernels_of_backward(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type.name == "CUDA"}


@pytest.mark.parametrize("prec", PRECISIONS)
def test_frozen_decoder_runs_no_weight_gradient(dev, prec):
    m = _model(dict(WIDE, causal=True), dev).set_precision(prec)
    gen = torch.Generator(device=dev).manual_seed(4)
    x = torch.randn(1, 2 * WIDE["latent_dim"], 70, device=dev, generator=gen)
    noise = torch.randn(1, WIDE["latent_dim"], 70, device=dev, generator=gen)
    r = torch.randn(1, 1, m.wav_length(70), device=dev, generator=gen)

    def step():
        xg = x.clone().requires_grad_(True)
        (m.decode_with_grad(xg, noise=noise) * r).sum().backward()
        return xg.grad

    g_full = step()
    names_full = _kernels_of_backward(step)
    m.requires_grad_(False)
    g_frozen = step()
    names_frozen = _kernels_of_backward(step)
    assert torch.equal(g_full, g_frozen)
    assert any("wgrad" in n for n in names_full), sorted(names_full)
    bad = sorted(n for n in names_frozen if any(k in n for k in WGRAD_KERNELS))
    assert not bad, bad


def test_mrstft_loss_reaches_every_decoder_parameter(dev):
    """The MR-STFT loss on decode_with_grad's output backpropagates to every decoder parameter of the bench-geometry
    model under "bf16", with finite, nonzero gradients."""
    m = _model(BENCH, dev).set_precision("bf16")
    gen = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn(1, 2 * BENCH["latent_dim"], 12, device=dev, generator=gen)
    target = 0.1 * torch.randn(1, 1, m.wav_length(12), device=dev, generator=gen)
    loss_fn = MultiResolutionSTFTLoss()
    y = m.decode_with_grad(x, noise=torch.zeros(1, BENCH["latent_dim"], 12, device=dev))
    loss_fn(y, target).backward()
    bad = [n for n, p in _decoder_params(m)
           if p.grad is None or not bool(torch.isfinite(p.grad).all()) or float(p.grad.abs().max()) == 0.0]
    assert not bad, bad


def test_inference_only_paths_refuse_gradients(dev):
    m = _model(dict(WIDE, causal=True), dev)
    x = torch.randn(1, 2 * WIDE["latent_dim"], 8, device=dev, requires_grad=True)
    with pytest.raises(NotImplementedError):
        m.decode_with_grad(x, valid_len=[8])
    from kalle_audio_b200.bigvgan_stream import BigVGANStreamingDecoder
    sd = BigVGANStreamingDecoder(m)
    with pytest.raises(ValueError, match="inference-only"):
        sd.push(x)
