"""GPU parity of the training step (BASELINE config 5, SURVEY.md section 8 row 12): loss and every parameter
gradient from kvae_forward_train / kvae_backward (through the drop-in modules' autograd nodes) against
  * gradients recorded from autograd through the REFERENCE's modules (tests/golden/train_*.npz), and
  * torch autograd through the CPU oracle on the same seeded inputs.
Tolerances: fp32 mode <= 1e-4 of each gradient's max magnitude (fp32 summation order differs: atomics);
bf16 mode (bf16 tensor-core operands in forward, dgrad and saved activations) relative L2 error <= 5e-2 per
parameter tensor -- BASELINE.json states no gradient tolerance, so it is stated here."""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as H
import kalle_audio_b200 as k
from kalle_audio_b200 import _lib, training as TR
from oracle import oobleck_oracle as O

pytestmark = pytest.mark.gpu

REL_F32 = 1e-4
REL_BF16 = 5e-2


@pytest.fixture(autouse=True)
def _grad_mode():
    """Other test modules switch autograd off globally at import; the training tests need it on."""
    with torch.enable_grad():
        yield


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def rel_l2(a, b):
    a, b = a.detach().double().cpu().reshape(-1), torch.as_tensor(b).double().reshape(-1)
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


# --------------------------------------------------------------------------- layer-level kernels
def test_snake_bwd_kernel(dev):
    torch.manual_seed(0)
    rows, Cc = 777, 37
    x = torch.randn(rows, Cc, requires_grad=True)
    al = (0.4 * torch.randn(Cc)).requires_grad_(True)
    be = (0.4 * torch.randn(Cc)).requires_grad_(True)
    gy = torch.randn(rows, Cc)
    y = O.snake_beta(x.t().unsqueeze(0), al, be)      # [1, C, rows]
    y.backward(gy.t().unsqueeze(0))
    xd, gd = x.detach().to(dev), gy.to(dev)
    ald, bed = al.detach().to(dev), be.detach().to(dev)
    gx = torch.empty_like(xd)
    da, db = torch.empty(Cc, device=dev), torch.empty(Cc, device=dev)
    scratch = torch.empty(2 * Cc, device=dev)
    _lib.check(_lib.lib().kvae_snake_bwd(xd.data_ptr(), gd.data_ptr(), gx.data_ptr(), ald.data_ptr(), bed.data_ptr(), 1, da.data_ptr(), db.data_ptr(), rows, Cc,
                                         scratch.data_ptr(), _lib.stream_ptr(dev)))
    assert float((gx.cpu() - x.grad).abs().max()) <= 1e-5
    assert float((da.cpu() - al.grad).abs().max()) <= 1e-4 * float(al.grad.abs().max())
    assert float((db.cpu() - be.grad).abs().max()) <= 1e-4 * float(be.grad.abs().max())


@pytest.mark.parametrize("shape", [(16, 8, 7), (5, 3, 1), (256, 128, 16)])
def test_weight_norm_bwd_kernel(dev, shape):
    torch.manual_seed(1)
    v = torch.randn(shape, requires_grad=True)
    g = (1.0 + 0.3 * torch.randn(shape[0], 1, 1)).requires_grad_(True)
    dw = torch.randn(shape)
    O.weight_norm_fold(v, g).backward(dw)
    vd, gd, dwd = v.detach().to(dev), g.detach().to(dev), dw.to(dev)
    dv, dg = torch.empty_like(vd), torch.empty(shape[0], device=dev)
    _lib.check(_lib.lib().kvae_weight_norm_bwd(vd.data_ptr(), gd.data_ptr(), dwd.data_ptr(), dv.data_ptr(), dg.data_ptr(),
                                               shape[0], shape[1] * shape[2], _lib.stream_ptr(dev)))
    assert float((dv.cpu() - v.grad).abs().max()) <= 1e-5 * max(1.0, float(v.grad.abs().max()))
    assert float((dg.cpu() - g.grad.reshape(-1)).abs().max()) <= 1e-5 * max(1.0, float(g.grad.abs().max()))


def test_vae_sample_and_nll_autograd_nodes(dev):
    torch.manual_seed(2)
    mean = torch.randn(3, 16, 50, requires_grad=True)
    scale = torch.randn(3, 16, 50, requires_grad=True)
    noise = torch.randn(3, 16, 50)
    target = torch.randn(3, 16, 50)
    z, kl = O.vae_sample(mean, scale, noise)
    ref = O.gaussian_nll(target, z, -0.5) + 0.3 * kl
    ref.backward()
    md, sd = mean.detach().to(dev).requires_grad_(True), scale.detach().to(dev).requires_grad_(True)
    zz, kk = TR.vae_sample_with_grad(md, sd, noise.to(dev))
    loss = TR.gaussian_nll(target.to(dev), zz, -0.5) + 0.3 * kk
    loss.backward()
    assert torch.equal(zz.detach().cpu(), z.detach())          # sample path stays bit-exact
    assert abs(float(loss.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach()))
    assert float((md.grad.cpu() - mean.grad).abs().max()) <= 1e-5 * float(mean.grad.abs().max())
    assert float((sd.grad.cpu() - scale.grad).abs().max()) <= 1e-5 * float(scale.grad.abs().max())


def test_flat_adamw_matches_torch(dev):
    torch.manual_seed(3)
    p0 = torch.randn(10001)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref], lr=3e-3, betas=(0.8, 0.99), eps=1e-8, weight_decay=1e-2)
    flat = p0.clone().to(dev)
    mine = TR.FlatAdamW([flat], lr=3e-3, betas=(0.8, 0.99), eps=1e-8, weight_decay=1e-2)
    for i in range(4):
        g = torch.randn(10001)
        ref.grad = g.clone() * 0.5
        opt.step()
        mine.step([g.to(dev)], grad_scale=0.5)
    assert float((flat.cpu() - ref.detach()).abs().max()) <= 2e-6


# --------------------------------------------------------------------------- stand-alone leaf modules under autograd
def test_snake_beta_module_backward(dev):
    torch.manual_seed(4)
    m = k.SnakeBeta(19).to(dev)
    with torch.no_grad():
        m.alpha.copy_(0.4 * torch.randn(19)); m.beta.copy_(0.4 * torch.randn(19))
    x = torch.randn(2, 19, 333, requires_grad=True)
    al, be = m.alpha.detach().cpu().requires_grad_(True), m.beta.detach().cpu().requires_grad_(True)
    w = torch.randn(2, 19, 333)
    (O.snake_beta(x, al, be) * w).sum().backward()
    xd = x.detach().to(dev).requires_grad_(True)
    (m(xd) * w.to(dev)).sum().backward()
    assert float((xd.grad.cpu() - x.grad).abs().max()) <= 1e-5
    assert float((m.alpha.grad.cpu() - al.grad).abs().max()) <= 1e-4 * float(al.grad.abs().max())
    assert float((m.beta.grad.cpu() - be.grad).abs().max()) <= 1e-4 * float(be.grad.abs().max())


@pytest.mark.parametrize("transposed,cin,cout,K,stride,dil,pad,T", [
    (0, 5, 7, 7, 1, 1, 3, 50), (0, 16, 16, 7, 1, 9, 27, 300), (0, 8, 16, 8, 4, 1, 2, 64), (0, 8, 4, 10, 5, 1, 3, 45),
    (0, 6, 6, 1, 1, 1, 0, 33), (0, 2, 32, 7, 1, 1, 3, 200), (1, 8, 4, 4, 2, 1, 1, 33), (1, 6, 3, 11, 5, 1, 3, 11),
    (1, 16, 8, 8, 4, 1, 2, 20),
    # 'same' with an even kernel (one more zero row on the right); padding past d (K - 1) on each kind of layer
    (0, 6, 5, 8, 1, 1, "same", 40), (0, 5, 7, 3, 1, 2, 6, 50), (0, 8, 4, 4, 2, 1, 5, 45), (1, 6, 4, 4, 2, 1, 4, 40)])
def test_wnconv_modules_backward(dev, transposed, cin, cout, K, stride, dil, pad, T):
    torch.manual_seed(5)
    if transposed:
        m = k.WNConvTranspose1d(cin, cout, K, stride=stride, padding=pad)
    else:
        m = k.WNConv1d(cin, cout, K, stride=stride, dilation=dil, padding=pad)
    with torch.no_grad():
        m.weight_g.mul_(1.0 + 0.2 * torch.randn_like(m.weight_g))
    sd = {"c." + n: p.detach().clone().requires_grad_(True) for n, p in m.state_dict().items()}
    x = torch.randn(2, cin, T, requires_grad=True)
    ref = (O._wn_conv_transpose1d(sd, "c", x, stride=stride, padding=pad) if transposed
           else O._wn_conv1d(sd, "c", x, stride=stride, padding=pad, dilation=dil))
    w = torch.randn_like(ref)
    (ref * w).sum().backward()
    m = m.to(dev)
    xd = x.detach().to(dev).requires_grad_(True)
    (m(xd) * w.to(dev)).sum().backward()
    tol = lambda r: 2e-5 * max(1.0, float(r.abs().max()))
    assert float((xd.grad.cpu() - x.grad).abs().max()) <= tol(x.grad)
    for n, p in m.named_parameters():
        r = sd["c." + n].grad
        assert p.grad is not None and float((p.grad.cpu() - r).abs().max()) <= tol(r), n


def test_residual_unit_standalone_backward(dev):
    """A block of the module tree used on its own (leaf kernels chained by torch autograd)."""
    torch.manual_seed(6)
    ru = k.ResidualUnit(12, 12, dilation=3, use_snake=True)
    H.randomize_snake(ru, 3)
    sd = {"r." + n: p.detach().clone().requires_grad_(True) for n, p in ru.state_dict().items()}
    x = torch.randn(2, 12, 90, requires_grad=True)
    w = torch.randn(2, 12, 90)
    (O.residual_unit(sd, "r", x, 3) * w).sum().backward()
    ru = ru.to(dev)
    xd = x.detach().to(dev).requires_grad_(True)
    (ru(xd) * w.to(dev)).sum().backward()
    assert float((xd.grad.cpu() - x.grad).abs().max()) <= 2e-5 * max(1.0, float(x.grad.abs().max()))
    for n, p in ru.named_parameters():
        r = sd["r." + n].grad
        assert float((p.grad.cpu() - r).abs().max()) <= 1e-4 * max(1.0, float(r.abs().max())), n


# --------------------------------------------------------------------------- whole training step
def _loss_and_grads(m, x, noise, kl_weight, log_sigma, precision):
    m.encoder.set_precision(precision)
    m.decoder.set_precision(precision)
    for p in m.parameters():
        p.grad = None
    enc = m.encoder(x)
    mean, scale = enc.chunk(2, dim=1)
    z, kl = TR.vae_sample_with_grad(mean, scale, noise)
    dec = m.decoder(z)
    nll = TR.gaussian_nll(x, dec, log_sigma)
    loss = nll + kl_weight * kl
    loss.backward()
    return loss.detach(), kl.detach(), dec.detach(), {n: p.grad for n, p in m.named_parameters()}


def test_training_grads_tiny_fp32_vs_reference_autograd(dev):
    g = H.golden("train_tiny")
    m = H.build("tiny", 0, snake_seed=7).to(dev).train()
    sd = {kk[3:]: H.t(g[kk]) for kk in g.files if kk.startswith("sd.")}
    m.load_state_dict(sd)
    loss, kl, dec, grads = _loss_and_grads(m, H.t(g["x"]).to(dev), H.t(g["noise"]).to(dev), float(g["kl_weight"]),
                                           float(g["log_sigma"]), "fp32")
    assert abs(float(loss) - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    assert abs(float(kl) - float(g["kl"])) <= 1e-5 * abs(float(g["kl"]))
    assert float((dec.cpu() - H.t(g["decoded"])).abs().max()) <= 1e-5
    worst = 0.0
    for n, gr in grads.items():
        ref = H.t(g["g." + n])
        assert gr is not None and gr.shape == ref.shape, n
        err = float((gr.cpu() - ref).abs().max()) / max(float(ref.abs().max()), 1e-12)
        worst = max(worst, err)
        assert err <= REL_F32, (n, err)
    print(f"tiny fp32: worst gradient error relative to its max = {worst:.2e}")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_training_grads_mid_vs_reference_autograd(dev, precision):
    g = H.golden("train_mid")
    m = H.build("mid", 0, snake_seed=7)
    H.check_checksums(m.state_dict(), g)
    m = m.to(dev).train()
    loss, kl, dec, grads = _loss_and_grads(m, H.t(g["x"]).to(dev), H.t(g["noise"]).to(dev), float(g["kl_weight"]),
                                           float(g["log_sigma"]), precision)
    tol = REL_F32 * 10 if precision == "fp32" else REL_BF16
    assert abs(float(loss) - float(g["loss"])) <= (1e-5 if precision == "fp32" else 2e-3) * abs(float(g["loss"]))
    worst = 0.0
    for i, n in enumerate(str(s) for s in g["g_keys"]):
        gr = grads[n]
        samp = gr.reshape(-1)[::max(1, gr.numel() // 256)][:256]
        ref = H.t(g[f"g_sample{i}"])
        e = rel_l2(samp, ref)
        worst = max(worst, e)
        assert e <= tol, (n, e)
        rn = float(g["g_norm"][i])
        assert abs(float(gr.double().norm()) - rn) <= tol * rn, n
    print(f"mid {precision}: worst per-parameter relative L2 gradient error = {worst:.2e}")


def test_decoder_input_gradient_and_frozen_parameters(dev):
    """Only the input requires grad (frozen decoder): the latent gradient must still match autograd."""
    g = H.golden("tiny_ae")
    m = H.build("tiny", 0, snake_seed=7).to(dev)
    sd = {kk[3:]: H.t(g[kk]) for kk in g.files if kk.startswith("sd.")}
    m.load_state_dict(sd)
    for p in m.parameters():
        p.requires_grad_(False)
    z = H.t(g["z"]).clone().requires_grad_(True)
    w = torch.randn(2, 2, 13 * 40, generator=torch.Generator().manual_seed(5))
    dsd = {kk[len("decoder."):]: v for kk, v in sd.items() if kk.startswith("decoder.")}
    (O.oobleck_decoder(dsd, z, H.strides_of("tiny")) * w).sum().backward()
    zd = H.t(g["z"]).to(dev).requires_grad_(True)
    (m.decoder.set_precision("fp32")(zd) * w.to(dev)).sum().backward()
    assert float((zd.grad.cpu() - z.grad).abs().max()) <= 1e-4 * float(z.grad.abs().max())


def test_training_grads_sao_shape_bf16_vs_oracle_autograd(dev):
    """The graded architecture (C = 128 ... 2048, tensor-core forward and data gradients) on a short clip,
    against torch autograd through the oracle on the host CPU."""
    m = H.build("sao", 0).to(dev).train()
    H.randomize_snake(m, 7)
    x = 0.1 * torch.randn(1, 2, 2048 * 6, generator=torch.Generator().manual_seed(2))
    noise = torch.randn(1, 64, 6, generator=torch.Generator().manual_seed(3))
    sd = {kk: v.detach().cpu().clone().requires_grad_(True) for kk, v in m.state_dict().items()}
    ref_loss, _, _, _ = O.training_loss(sd, x, noise, H.strides_of("sao"), 1e-2, -1.0)
    ref_loss.backward()
    loss, kl, dec, grads = _loss_and_grads(m, x.to(dev), noise.to(dev), 1e-2, -1.0, "bf16")
    assert abs(float(loss) - float(ref_loss)) <= 2e-3 * abs(float(ref_loss))
    worst, worst_name = 0.0, ""
    for n, gr in grads.items():
        ref = sd[n].grad
        e = rel_l2(gr, ref)
        if e > worst:
            worst, worst_name = e, n
        assert e <= REL_BF16, (n, e)
    print(f"SAO bf16: worst per-parameter relative L2 gradient error = {worst:.2e} ({worst_name})")


def test_trainer_step_updates_and_reduces_loss(dev):
    m = H.build("mid", 0, snake_seed=7).to(dev).train()
    x = 0.1 * torch.randn(4, 2, 40 * 32, generator=torch.Generator().manual_seed(9)).to(dev)
    noise = torch.randn(4, 64, 32, generator=torch.Generator().manual_seed(10)).to(dev)
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    tr = TR.AutoencoderTrainer(m, lr=2e-4, kl_weight=1e-4, log_sigma=-2.0, precision="bf16")
    assert list(before.keys()) == [n for n, _ in m.named_parameters()]
    losses = [float(tr.training_step(x, noise)["loss"]) for _ in range(6)]
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    changed = sum(int(not torch.equal(before[n], p.detach())) for n, p in m.named_parameters())
    assert changed == len(before)
    # parameters stay views of the flat master buffers, and inference sees the updated weights
    assert next(m.encoder.parameters()).data_ptr() == tr.flat_enc.data_ptr()
    with torch.no_grad():
        y1 = m.decode(noise)
    m2 = H.build("mid", 0, snake_seed=7).to(dev)
    m2.load_state_dict(m.state_dict())
    m2.encoder.set_precision("bf16"); m2.decoder.set_precision("bf16")
    with torch.no_grad():
        y2 = m2.decode(noise)
    assert float((y1 - y2).abs().max()) <= 1e-6


def test_other_precision_runner_sees_every_optimizer_step(dev):
    """A second runner of the same module (fp32-mode validation between bf16 training steps) must re-pack after EVERY
    optimizer step: kvae_adamw_step writes through the flat buffer, which does not bump the parameter views' version
    counters, so the trainer bumps an explicit weights epoch that every runner's fingerprint includes."""
    m = H.build("mid", 0, snake_seed=7).to(dev).train()
    x = 0.1 * torch.randn(2, 2, 40 * 16, generator=torch.Generator().manual_seed(9)).to(dev)
    noise = torch.randn(2, 64, 16, generator=torch.Generator().manual_seed(10)).to(dev)
    tr = TR.AutoencoderTrainer(m, lr=5e-3, kl_weight=1e-4, log_sigma=-2.0, precision="bf16")

    def fresh_eval():
        m2 = H.build("mid", 0, snake_seed=7).to(dev)
        m2.load_state_dict(m.state_dict())
        with torch.no_grad():
            return m2.set_precision("fp32").decode(noise)

    outs = []
    for _ in range(3):
        m.set_precision("bf16")
        tr.training_step(x, noise)
        m.set_precision("fp32")
        with torch.no_grad():
            y = m.decode(noise)          # the fp32 runner: created at the first pass, must not serve stale weights later
        assert float((y - fresh_eval()).abs().max()) <= 1e-6
        outs.append(y)
    assert float((outs[1] - outs[0]).abs().max()) > 1e-5 and float((outs[2] - outs[1]).abs().max()) > 1e-5
    assert all(p.grad is None for p in m.parameters())      # trainer mode: the flat gradient buffer is the product
    # .to() rebuilds the plan cache; the trainer's flat buffers and hook are re-attached to the new runners
    m.set_precision("bf16")
    m.encoder._plans.clear(); m.decoder._plans.clear()
    assert np.isfinite(float(tr.training_step(x, noise)["loss"]))


def test_training_step_config5_shape_properties(dev):
    """BASELINE configs[4] per-GPU shape (4 clips x 5.016 s, bf16 mode): finite loss and gradients, the backward is
    linear in the incoming gradient, and two runs agree (the only non-determinism is the order of fp32 atomics)."""
    m = H.build("sao", 0).to(dev).train()
    m.encoder.set_precision("bf16"); m.decoder.set_precision("bf16")
    x = (0.1 * torch.randn(4, 2, 108 * 2048, generator=torch.Generator().manual_seed(2))).to(dev)
    noise = torch.randn(4, 64, 108, generator=torch.Generator().manual_seed(3)).to(dev)

    def grads(scale):
        for p in m.parameters():
            p.grad = None
        enc = m.encoder(x)
        mean, sc = enc.chunk(2, dim=1)
        zz, kl = TR.vae_sample_with_grad(mean, sc, noise)
        loss = (TR.gaussian_nll(x, m.decoder(zz), -2.0) + 1e-4 * kl) * scale
        loss.backward()
        return float(loss.detach()), torch.cat([p.grad.reshape(-1) for p in m.parameters()])

    l1, g1 = grads(1.0)
    l2, g2 = grads(1.0)
    l3, g3 = grads(2.0)
    assert np.isfinite(l1) and bool(torch.isfinite(g1).all())
    assert l1 == l2
    n = float(g1.norm())
    assert float((g1 - g2).norm()) <= 1e-4 * n                      # atomics order only
    assert float((g3 - 2.0 * g1).norm()) <= 2e-4 * 2.0 * n          # linear in the incoming gradient


def test_trainer_with_the_spectral_loss(dev):
    """AutoencoderTrainer with the reference's spectral term (SumAndDifferenceSTFTLoss(reals, decoded), the way
    training/autoencoders.py:163 wires it) instead of the Gaussian NLL: the loss the decoder is trained on in the
    reference minus its GAN terms.  A fixed batch must be fitted better step by step."""
    torch.manual_seed(0)
    ae = H.build("mid", 0).to(dev)
    sd = k.SumAndDifferenceSTFTLoss(fft_sizes=[512, 256, 128, 64, 32], hop_sizes=[128, 64, 32, 16, 8],
                                    win_lengths=[512, 256, 128, 64, 32], perceptual_weighting=True, sample_rate=16000)
    tr = k.AutoencoderTrainer(ae, lr=2e-4, precision="bf16", data_parallel=False, spectral_loss=sd, nll_weight=0.0)
    x = 0.1 * torch.randn(2, 2, 40 * 64, device=dev)
    noise = torch.randn(2, 64, 64, device=dev)
    losses = []
    for _ in range(6):
        info = tr.training_step(x, noise)          # (enables autograd itself)
        assert "mrstft" in info and torch.isfinite(info["loss"])
        losses.append(float(info["mrstft"]))
    assert losses[-1] < losses[0], losses


def test_trainer_with_the_discriminator(dev):
    """AutoencoderTrainer with the reference's GAN terms (training/autoencoders.py:287-337): even steps train the
    autoencoder on spectral + adversarial + feature-matching + KL, odd steps train the OobleckDiscriminator on the hinge
    loss; each step moves only its own parameters, and the logged GAN terms are the discriminator's own loss() on the
    step's decoded signal."""
    from kalle_audio_b200.discriminators import OobleckDiscriminator
    torch.manual_seed(0)
    ae = H.build("mid", 0).to(dev)
    disc = OobleckDiscriminator(in_channels=2).to(dev)
    sd = k.SumAndDifferenceSTFTLoss(fft_sizes=[512, 256, 128, 64, 32], hop_sizes=[128, 64, 32, 16, 8],
                                    win_lengths=[512, 256, 128, 64, 32], perceptual_weighting=True, sample_rate=16000)
    tr = k.AutoencoderTrainer(ae, lr=2e-4, precision="bf16", data_parallel=False, spectral_loss=sd, nll_weight=0.0,
                              discriminator=disc, adversarial_weight=0.1, feature_matching_weight=5.0)
    x = 0.1 * torch.randn(2, 2, 40 * 64, device=dev)
    noise = torch.randn(2, 64, 64, device=dev)
    ae0 = torch.cat([tr.flat_enc, tr.flat_dec]).clone()
    d0 = tr.flat_disc.clone()
    info = tr.training_step(x, noise)                      # step 0: generator
    assert {"mrstft", "loss_adv", "feature_matching_distance", "kl"} <= set(info)
    assert torch.isfinite(info["loss"])
    assert not torch.equal(torch.cat([tr.flat_enc, tr.flat_dec]), ae0) and torch.equal(tr.flat_disc, d0)
    with torch.no_grad():
        dis, adv, fm = disc.loss(x, info["decoded"].float())
    assert abs(float(adv) - float(info["loss_adv"])) <= 1e-5 + 1e-4 * abs(float(adv))
    assert abs(float(fm) - float(info["feature_matching_distance"])) <= 1e-4 * float(fm)
    want = float(info["mrstft"]) + 0.1 * float(adv) + 5.0 * float(fm) + tr.kl_weight * float(info["kl"])
    assert abs(float(info["loss"]) - want) <= 1e-4 * abs(want)
    ae1 = torch.cat([tr.flat_enc, tr.flat_dec]).clone()
    info = tr.training_step(x, noise)                      # step 1: discriminator
    assert "mrstft" not in info and torch.isfinite(info["loss_dis"])
    assert torch.equal(torch.cat([tr.flat_enc, tr.flat_dec]), ae1) and not torch.equal(tr.flat_disc, d0)
    first = float(info["loss_dis"])
    for _ in range(3):                                     # discriminator steps on a fixed batch lower its hinge loss
        info = tr.discriminator_step(x, noise)
    assert float(info["loss_dis"]) < first, (first, float(info["loss_dis"]))
    info = tr.training_step(x, noise)                      # step 2: generator again, with the updated discriminator
    assert "mrstft" in info and torch.isfinite(info["loss"])
