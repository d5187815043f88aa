"""Gradients through BigVGANFlowVAE's encoder (encode_with_grad) against float64 autograd through
oracle/bigvgan_oracle.py on the module's own parameters:

  * the conv backward (kvae_conv1d_win_bwd) of every conv geometry of the bench encoder on each engine it runs on, the
    strided downsampling convs included, at B = 1 and 3, at the 64-row threshold and at data-gradient outputs on the
    M-tile edges with every T mod s;
  * the whole encoder: forward equal to extract_latents (fp32 and bf16 audio, clips that are not whole frames),
    gradients of the audio and of every encoder parameter;
  * a frozen encoder runs no weight-gradient kernel, and the bench encoder's strided layers run their backward on the
    tensor cores under "bf16";
  * the whole autoencoder, decode_with_grad(encode_with_grad(x)), against float64 autograd and under the MR-STFT loss.

LeakyReLU's derivative jumps at 0 (slope 1 or 0.2 / 0.01), so the gradient is not a continuous function of the
forward activations: an element whose pre-activation lies within the forward's rounding error of 0 takes the other
slope, and k such elements out of N give a relative L2 error of about sqrt(k / N), far above the engine's rounding
error (against plain float64 autograd: up to 1.7e-2 under "fp32" and 0.12 under "bf16"; 1e-2 under None at the bench
config, where torch's own fp32 autograd is off by 1.8e-3).  The whole-encoder references therefore run the oracle in
float64 with each LeakyReLU's slope taken where the library's forward put it (``_masked_oracle``), which leaves the
rounding of the backward itself to GRAD_BOUND; the error against the plain oracle is reported."""
import contextlib

import pytest
import torch
import torch.nn.functional as F

import helpers as H
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.layers import TC_MIN_ROWS
from kalle_audio_b200.losses import MultiResolutionSTFTLoss
from oracle import bigvgan_oracle as BO
from test_gpu_bigvgan_grad import (BENCH, CONV_BOUND, GRAD_BOUND, PRECISIONS, WGRAD_KERNELS, WIDE, AttrDict, _F64,
                                   _decoder_params, _kernels_of_backward, _model, _rel)

pytestmark = pytest.mark.gpu

# the strided s 4 and s 5 convs (64 -> 128, 128 -> 192) on the tensor cores from 512 samples on; decoder as WIDE
SMALL = AttrDict(WIDE, causal=True, downsample_channels=[12, 64, 128, 192], downsample_rates=[2, 4, 5])


@pytest.fixture(autouse=True)
def _grad_mode():
    """Other test modules turn grad mode off when they are imported; these tests need it on."""
    with torch.enable_grad():
        yield


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _encoder_params(m):
    return [(n, p) for n, p in m.named_parameters() if n.startswith("audio_encoder.")]


# ------------------------------------------------------------------------------------------------- a. conv layers
def _encoder_layers(model):
    mods = {}
    for op in BV._encoder_program(model.h)[0]:
        if op.kind == "conv":
            m = BV._module(model, op.module)
            mods.setdefault((m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0], m.dilation[0]), (op.module, m))
    return list(mods.values())


def _sweep_lengths(m):
    """the 64-row threshold, and inputs whose data gradient (T rows, in ceil(T / s) stride groups on the tensor cores)
    has 127 / 128 / 129 groups, with every T mod s"""
    s = m.stride[0]
    return sorted({TC_MIN_ROWS} | {tq * s - r for tq in (127, 128, 129) for r in range(s)})


def test_encoder_conv_backward_per_engine(dev):
    model = _model(BENCH, dev)
    gen = torch.Generator(device=dev).manual_seed(2)
    worst, fails, n_strided_tc = {}, [], 0
    for tag, m in _encoder_layers(model):
        m.tc_precision = "fp32"
        precs = PRECISIONS if m.tc_layer() else (None,)
        n_strided_tc += int(m.tc_layer() and m.stride[0] > 1)
        K, s, d, p = m.kernel_size[0], m.stride[0], m.dilation[0], m.padding[0]
        for B in (1, 3):
            for T in _sweep_lengths(m):
                x = torch.randn(B, m.in_channels, T, device=dev, generator=gen)
                with _F64(dev):
                    xd = x.double().requires_grad_(True)
                    vd, gd = m.weight_v.detach().double().requires_grad_(True), m.weight_g.detach().double().requires_grad_(True)
                    bd = m.bias.detach().double().requires_grad_(True)
                    wd = vd * (gd / vd.flatten(1).norm(dim=1).view(-1, 1, 1))
                    yd = F.conv1d(xd, wd, bd, stride=s, padding=p, dilation=d)
                    r = torch.randn(yd.shape, device=dev, generator=gen, dtype=torch.float64)
                    refs = torch.autograd.grad(yd, [xd, gd, vd, bd], r)
                for prec in precs:
                    m.tc_precision = prec
                    e_id = 0 if prec is None or T < TC_MIN_ROWS else (1 if prec == "bf16" else 2)
                    xg = x.clone().requires_grad_(True)
                    y = m(xg)
                    got = torch.autograd.grad(y, [xg, m.weight_g, m.weight_v, m.bias], r.float())
                    for name, a, ref in zip(("gx", "dg", "dv", "dbias"), got, refs):
                        e = _rel(a, ref)
                        worst[(e_id, name)] = max(worst.get((e_id, name), 0.0), e)
                        if e > CONV_BOUND[e_id]["gx" if name == "gx" else "w"]:
                            fails.append(f"{tag} B={B} T={T} engine {e_id}: {name} rel L2 {e:.2e}")
        m.tc_precision = "fp32"
    H.report("BigVGAN encoder conv backward: worst rel L2",
             ", ".join(f"e{e} {n} {v:.2e}" for (e, n), v in sorted(worst.items())))
    assert n_strided_tc == 2                         # 192 -> 384 (s 4) and 384 -> 768 (s 5)
    assert not fails, "\n".join(fails[:40])


# ------------------------------------------------------------------------------------------------- b. whole encoder
def _kink_masks(m, run):
    """(pre-activation > 0) of every LeakyReLU of the encoder, in execution order, as the library's forward ``run()``
    computes them"""
    masks, hooks = [], []
    for mod in m.audio_encoder.modules():
        if isinstance(mod, BV.LeakyReLU):
            hooks.append(mod.register_forward_pre_hook(lambda _, inp: masks.append(inp[0].detach() > 0)))
    try:
        with torch.no_grad():
            run()
    finally:
        for h in hooks:
            h.remove()
    return masks


class _MaskedF:
    """torch.nn.functional for the oracle, each leaky_relu's slope chosen by the next mask"""

    def __init__(self, masks):
        self.masks = iter(masks)

    def __getattr__(self, name):
        return getattr(F, name)

    def leaky_relu(self, x, slope):
        return torch.where(next(self.masks), x, slope * x)


@contextlib.contextmanager
def _masked_oracle(masks):
    """bigvgan_oracle's encoder with the library's LeakyReLU slopes"""
    prev, BO.F = BO.F, _MaskedF(masks)
    try:
        yield
    finally:
        BO.F = prev


def _encoder_oracle(m, x, r, masks=None):
    """the gradients of sum(latents * r) w.r.t. the audio and every encoder parameter by float64 autograd through the
    oracle (with the library's LeakyReLU slopes when ``masks`` is given)"""
    with _F64(x.device), (_masked_oracle(masks) if masks is not None else contextlib.nullcontext()):
        sd = {n: p.detach().double() for n, p in m.state_dict().items() if n.startswith("audio_encoder.")}
        leaves = {n: sd[n].requires_grad_(True) for n, _ in _encoder_params(m)}
        xd = x.detach().double().requires_grad_(True)
        y = BO.extract_latents(sd, dict(m.h), xd)
        gs = torch.autograd.grad((y * r.double()).sum(), [xd] + list(leaves.values()))
    return gs[0], dict(zip(leaves, gs[1:]))


ENCODE_CASES = {"small_2813": (SMALL, 2, 2813), "small_2800": (SMALL, 2, 2800), "bench_113000": (BENCH, 1, 113000),
                "bench_102400": (BENCH, 1, 102400)}


@pytest.mark.parametrize("case", list(ENCODE_CASES))
def test_encode_with_grad_vs_oracle(dev, case):
    h, B, L = ENCODE_CASES[case]
    m = _model(h, dev, seed=3)
    gen = torch.Generator(device=dev).manual_seed(4)
    x = 0.3 * torch.randn(B, 1, L, device=dev, generator=gen)
    r = torch.randn(B, 2 * h["latent_dim"], m.latent_length(L), device=dev, generator=gen)
    plain_gx, plain_gp = _encoder_oracle(m, x, r)
    fails, worst, plain = [], {}, {}
    for prec in PRECISIONS:
        m.set_precision(prec)
        ref_gx, ref_gp = _encoder_oracle(m, x, r, _kink_masks(m, lambda: m.extract_latents(x)))
        for dt in (torch.float32, torch.bfloat16):
            xa = x.to(dt)
            ref_y = m.extract_latents(xa)
            xg = xa.clone().requires_grad_(True)
            for p in m.parameters():
                p.grad = None
            y = m.encode_with_grad(xg)
            if not torch.equal(y.detach(), ref_y):
                fails.append(f"{prec} {dt}: encode_with_grad output differs from extract_latents")
            (y.float() * r).sum().backward()
            named = [("audio", xg.grad, ref_gx)] + [(n, p.grad, ref_gp[n]) for n, p in _encoder_params(m)]
            if dt == torch.bfloat16:                # bf16 audio: bf16 activations throughout; gradients reach everything
                fails += [f"{prec} bf16: {n} gradient missing or not finite" for n, g, _ in named
                          if g is None or not bool(torch.isfinite(g).all())]
                continue
            for name, got, ref in named:
                if got is None:
                    fails.append(f"{prec}: {name} has no gradient")
                    continue
                e = _rel(got, ref)
                worst[prec] = max(worst.get(prec, 0.0), e)
                plain[prec] = max(plain.get(prec, 0.0), _rel(got, plain_gx if name == "audio" else plain_gp[name]))
                if e > GRAD_BOUND[prec]:
                    fails.append(f"{prec}: {name} rel L2 {e:.2e}")
    H.report(f"encode_with_grad {case}: worst rel L2 (library's LeakyReLU slopes)",
             ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    H.report(f"encode_with_grad {case}: worst rel L2 (plain float64 oracle)",
             ", ".join(f"{k} {v:.2e}" for k, v in plain.items()))
    assert not fails, "\n".join(fails[:40])


# ------------------------------------------------------------------------------------------------- c. kernels
@pytest.mark.parametrize("prec", PRECISIONS)
def test_frozen_encoder_runs_no_weight_gradient(dev, prec):
    m = _model(SMALL, dev).set_precision(prec)
    gen = torch.Generator(device=dev).manual_seed(5)
    x = 0.3 * torch.randn(1, 1, 2813, device=dev, generator=gen)
    r = torch.randn(1, 2 * SMALL["latent_dim"], m.latent_length(2813), device=dev, generator=gen)

    def step():
        xg = x.clone().requires_grad_(True)
        (m.encode_with_grad(xg) * r).sum().backward()
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


def test_strided_layers_backward_on_tensor_cores(dev):
    """Under "bf16" the bench encoder's 192 -> 384 and 384 -> 768 downsampling convs run their data gradient on
    conv_umma2_kernel and their weight gradient on wgrad_umma_kernel, nothing on the CUDA-core conv kernels."""
    m = _model(BENCH, dev).set_precision("bf16")
    gen = torch.Generator(device=dev).manual_seed(6)
    seen = 0
    for tag, layer in _encoder_layers(m):
        if layer.stride[0] == 1 or not layer.tc_layer():
            continue
        seen += 1
        T = 130 * layer.stride[0] + 1
        xg = torch.randn(2, layer.in_channels, T, device=dev, generator=gen).requires_grad_(True)
        y = layer(xg)
        r = torch.randn(y.shape, device=dev, generator=gen)
        names = _kernels_of_backward(lambda: y.backward(r))
        assert any("conv_umma2_kernel" in n for n in names), (tag, sorted(names))
        assert any("wgrad_umma_kernel" in n for n in names), (tag, sorted(names))
        bad = sorted(n for n in names if "conv_direct_kernel" in n or "wgrad_direct_kernel" in n)
        assert not bad, (tag, bad)
    assert seen == 2


# ------------------------------------------------------------------------------------------------- d. round trip
def test_round_trip_vs_oracle(dev):
    m = _model(SMALL, dev, seed=7)
    gen = torch.Generator(device=dev).manual_seed(8)
    L = 2813
    x = 0.3 * torch.randn(2, 1, L, device=dev, generator=gen)
    F_ = m.latent_length(L)
    noise = torch.randn(2, SMALL["latent_dim"], F_, device=dev, generator=gen)
    r = torch.randn(2, 1, m.wav_length(F_), device=dev, generator=gen)
    params = _encoder_params(m) + _decoder_params(m)

    def reference(masks):
        with _F64(dev), _masked_oracle(masks):
            sd = {n: p.detach().double() for n, p in m.state_dict().items()}
            leaves = {n: sd[n].requires_grad_(True) for n, _ in params}
            xd = x.double().requires_grad_(True)
            yd = BO.inference_from_latents(sd, dict(m.h), BO.extract_latents(sd, dict(m.h), xd), noise.double())
            gs = torch.autograd.grad((yd * r.double()).sum(), [xd] + list(leaves.values()))
        return dict(zip(["audio"] + list(leaves), gs))

    fails, worst = [], {}
    for prec in PRECISIONS:
        m.set_precision(prec)
        ref = reference(_kink_masks(m, lambda: m.extract_latents(x)))
        for p in m.parameters():
            p.grad = None
        xg = x.clone().requires_grad_(True)
        y = m.decode_with_grad(m.encode_with_grad(xg), noise=noise)
        (y * r).sum().backward()
        for name, got in [("audio", xg.grad)] + [(n, p.grad) for n, p in params]:
            if got is None:
                fails.append(f"{prec}: {name} has no gradient")
                continue
            e = _rel(got, ref[name])
            worst[prec] = max(worst.get(prec, 0.0), e)
            if e > GRAD_BOUND[prec]:
                fails.append(f"{prec}: {name} rel L2 {e:.2e}")
    H.report("encode_with_grad -> decode_with_grad round trip: worst rel L2",
             ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))
    assert not fails, "\n".join(fails[:40])


def test_mrstft_round_trip_reaches_every_parameter(dev):
    """The MR-STFT loss of the bench autoencoder's reconstruction under "bf16" backpropagates to every encoder and
    decoder parameter, with finite, nonzero gradients."""
    m = _model(BENCH, dev).set_precision("bf16")
    gen = torch.Generator(device=dev).manual_seed(9)
    L = 1280 * 20                                     # the 384 -> 768 conv gets 80 input rows: on the tensor cores
    x = 0.3 * torch.randn(1, 1, L, device=dev, generator=gen)
    lat = m.encode_with_grad(x)
    y = m.decode_with_grad(lat, noise=torch.randn(1, BENCH["latent_dim"], lat.shape[2], device=dev, generator=gen))
    MultiResolutionSTFTLoss()(y, x[:, :, :y.shape[2]]).backward()
    bad = [n for n, p in _encoder_params(m) + _decoder_params(m)
           if p.grad is None or not bool(torch.isfinite(p.grad).all()) or float(p.grad.abs().max()) == 0.0]
    assert not bad, bad


def test_encoder_inference_only_paths_refuse_gradients(dev):
    m = _model(SMALL, dev)
    x = torch.randn(1, 1, 800, device=dev, requires_grad=True)
    with pytest.raises(NotImplementedError):
        m.encode_with_grad(x, valid_len=[800])
    from kalle_audio_b200.bigvgan_stream import BigVGANStreamingEncoder
    with pytest.raises(ValueError, match="inference-only"):
        BigVGANStreamingEncoder(m).push(x)
