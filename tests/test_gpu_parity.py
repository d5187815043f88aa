"""GPU parity: the CUDA path (through the Python drop-in modules and the C ABI) against the CPU oracle and
the golden outputs of the reference's own modules.  Tolerances are BASELINE.json's: max-abs <= 1e-5 in fp32
mode, <= 1e-3 in bf16 mode (both against the fp32 reference); latent sampling bit-exact."""
import numpy as np
import pytest
import torch

import helpers as H
import kalle_audio_b200 as k
from oracle import oobleck_oracle as O

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

TOL_F32 = 1e-5
TOL_BF16 = 1e-3


def bf16_tol(ref):
    """BASELINE.json's 1e-3 max-abs budget is quoted for the random-init SAO / O12 models, whose waveform
    abs-max is ~0.125.  Other fixtures (perturbed SnakeBeta parameters, fewer stages, encoder latents) have
    larger outputs, so the budget scales with the reference's magnitude: 1e-3 * max(1, absmax / 0.125)."""
    a = float(np.abs(np.asarray(ref.detach().cpu() if torch.is_tensor(ref) else ref)).max())
    return TOL_BF16 * max(1.0, a / 0.125)


def _sd_from_golden(g, prefix="sd."):
    return {kk[len(prefix):]: H.t(g[kk]) for kk in g.files if kk.startswith(prefix)}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def maxerr(a, b):
    return float((a.detach().float().cpu() - H.t(b).float()).abs().max())


# --------------------------------------------------------------------------- leaves
def test_snake_beta_module(dev):
    torch.manual_seed(0)
    m = k.SnakeBeta(37).to(dev)
    with torch.no_grad():
        m.alpha.copy_(0.4 * torch.randn(37)); m.beta.copy_(0.4 * torch.randn(37))
    x = torch.randn(3, 37, 1001)
    ref = O.snake_beta(x, m.alpha.cpu(), m.beta.cpu())
    assert maxerr(m(x.to(dev)), ref) <= 2e-6
    yb = m(x.to(dev).bfloat16())
    assert yb.dtype == torch.bfloat16 and maxerr(yb, O.snake_beta(x.bfloat16().float(), m.alpha.cpu(), m.beta.cpu())) <= 4e-2
    assert k.SnakeBeta(4).to(dev)(torch.zeros(2, 4, 0, device=dev)).shape == (2, 4, 0)    # empty input
    f = k.snake_beta(x.to(dev), torch.exp(m.alpha).view(1, -1, 1), torch.exp(m.beta).view(1, -1, 1))
    assert maxerr(f, ref) <= 2e-6


@pytest.mark.parametrize("cin,cout,K,stride,dil,pad,T", [
    (5, 7, 7, 1, 1, 3, 50), (16, 16, 7, 1, 9, 27, 300), (8, 16, 8, 4, 1, 2, 64), (8, 4, 10, 5, 1, 3, 45),
    (128, 2, 7, 1, 1, 3, 777), (2, 128, 7, 1, 1, 3, 500), (6, 6, 1, 1, 1, 0, 33), (4, 4, 7, 1, 3, 9, 5), (3, 5, 3, 2, 1, 1, 17)])
def test_wnconv1d_module(dev, cin, cout, K, stride, dil, pad, T):
    torch.manual_seed(1)
    m = k.WNConv1d(cin, cout, K, stride=stride, dilation=dil, padding=pad)
    with torch.no_grad():
        m.weight_g.mul_(1.0 + 0.2 * torch.randn_like(m.weight_g))
    x = torch.randn(2, cin, T)
    sd = {"c." + n: p for n, p in m.state_dict().items()}
    ref = O._wn_conv1d(sd, "c", x, stride=stride, padding=pad, dilation=dil)
    y = m.to(dev)(x.to(dev))
    assert y.shape == ref.shape
    assert maxerr(y, ref) <= 2e-5 * max(1.0, float(ref.abs().max()))
    assert maxerr(m.weight, O.weight_norm_fold(sd["c.weight_v"], sd["c.weight_g"])) <= 1e-6


@pytest.mark.parametrize("cin,cout,stride,T", [(8, 4, 2, 33), (16, 8, 4, 20), (6, 3, 5, 11), (8, 8, 8, 9), (128, 64, 4, 50)])
def test_wnconvtranspose1d_module(dev, cin, cout, stride, T):
    torch.manual_seed(2)
    K, pad = 2 * stride + stride % 2, (stride + 1) // 2
    m = k.WNConvTranspose1d(cin, cout, K, stride=stride, padding=pad)
    with torch.no_grad():
        m.weight_g.mul_(1.0 + 0.2 * torch.randn_like(m.weight_g))
    x = torch.randn(2, cin, T)
    sd = {"c." + n: p for n, p in m.state_dict().items()}
    ref = O._wn_conv_transpose1d(sd, "c", x, stride=stride, padding=pad)
    y = m.to(dev)(x.to(dev))
    assert y.shape == ref.shape == (2, cout, T * stride)
    assert maxerr(y, ref) <= 2e-5 * max(1.0, float(ref.abs().max()))


def test_standalone_blocks_chain_leaf_kernels(dev):
    torch.manual_seed(3)
    ru = k.ResidualUnit(8, 8, dilation=3, use_snake=True)
    db = k.DecoderBlock(16, 8, stride=4, use_snake=True)
    eb = k.EncoderBlock(8, 16, stride=5, use_snake=True)
    x = torch.randn(2, 8, 100)
    ref = O.residual_unit({"r." + n: p for n, p in ru.state_dict().items()}, "r", x, 3)
    assert maxerr(ru.to(dev)(x.to(dev)), ref) <= 2e-5
    x16 = torch.randn(2, 16, 25)
    assert maxerr(db.to(dev)(x16.to(dev)),
                  O.decoder_block({"d." + n: p.cpu() for n, p in db.state_dict().items()}, "d", x16, 4)) <= 5e-5
    assert maxerr(eb.to(dev)(x.to(dev)),
                  O.encoder_block({"e." + n: p.cpu() for n, p in eb.state_dict().items()}, "e", x, 5)) <= 5e-5


# --------------------------------------------------------------------------- fused plans, small models
def test_tiny_model_fp32_mode_matches_reference(dev):
    g = H.golden("tiny_ae")
    m = H.build("tiny", 0, snake_seed=7)
    m.load_state_dict(_sd_from_golden(g))
    m.to(dev)
    y = m.decode(H.t(g["z"]).to(dev))
    e = m.encode(H.t(g["x"]).to(dev))
    assert y.dtype == torch.float32 and y.shape == g["dec_out"].shape and e.shape == g["enc_out"].shape
    assert maxerr(y, g["dec_out"]) <= TOL_F32
    assert maxerr(e, g["enc_out"]) <= TOL_F32


def test_mid_model_tensor_core_path(dev):
    """C = 64/128/256 three-stage model: every inner conv runs on tcgen05 in bf16 mode."""
    g = H.golden("mid_ae")
    m = H.build("mid", 0, snake_seed=7)
    H.check_checksums(m.state_dict(), g)
    m.to(dev)
    z, x = H.t(g["z"]).to(dev), H.t(g["x"]).to(dev)
    y32, e32 = m.decode(z), m.encode(x)
    assert maxerr(y32, g["dec_out"]) <= TOL_F32 and maxerr(e32, g["enc_out"]) <= TOL_F32
    m.set_precision("bf16")
    y16, e16 = m.decode(z), m.encode(x)
    assert y16.dtype == torch.float32
    assert maxerr(y16, g["dec_out"]) <= bf16_tol(g["dec_out"])
    assert maxerr(e16, g["enc_out"]) <= bf16_tol(g["enc_out"])
    assert maxerr(y16, g["dec_out"]) > 0.0      # it really is the reduced-precision path
    mb = H.build("mid", 0, snake_seed=7).to(dev).bfloat16()
    yb = mb.decode(z.bfloat16())
    assert yb.dtype == torch.bfloat16 and maxerr(yb, g["dec_out"]) <= bf16_tol(g["dec_out"]) + 2e-3  # + bf16 output rounding


@pytest.mark.parametrize("B,T", [(1, 1), (1, 7), (3, 33), (2, 130), (5, 64)])
def test_ragged_shapes_mid_decoder(dev, B, T):
    m = H.build("mid", 0, snake_seed=7)
    sd = H.split_sd(m.state_dict(), "decoder.")
    z = torch.randn(B, 64, T, generator=torch.Generator().manual_seed(B * 100 + T))
    ref = O.oobleck_decoder(sd, z, H.strides_of("mid"))
    m.to(dev).set_precision("bf16")
    assert maxerr(m.decode(z.to(dev)), ref) <= bf16_tol(ref)
    m.set_precision("fp32")
    assert maxerr(m.decode(z.to(dev)), ref) <= TOL_F32


def test_weight_update_is_picked_up(dev):
    m = H.build("mid", 0).to(dev).set_precision("bf16")
    z = torch.randn(1, 64, 8, device=dev)
    y0 = m.decode(z)
    with torch.no_grad():
        m.decoder.layers[0].weight_g.mul_(1.5)
    y1 = m.decode(z)
    assert float((y1 - y0).abs().max()) > 1e-4
    ref = O.oobleck_decoder(H.split_sd({n: p.cpu() for n, p in m.state_dict().items()}, "decoder."), z.cpu(),
                            H.strides_of("mid"))
    assert maxerr(y1, ref) <= bf16_tol(ref)


def test_errors(dev):
    m = H.build("tiny", 0).to(dev)
    with pytest.raises(ValueError):
        m.encode(torch.randn(1, 2, 81, device=dev))          # not a multiple of the ratio
    with pytest.raises(ValueError):
        m.decode(torch.randn(0, 4, 8, device=dev))
    with pytest.raises(k.KvaeError):
        m.decode(torch.randn(1, 4, 8))                        # CPU tensor
    with pytest.raises(NotImplementedError):                  # final_tanh has no backward
        dt = k.OobleckDecoder(out_channels=2, channels=8, latent_dim=4, c_mults=[1, 2], strides=[2, 4], use_snake=True,
                              final_tanh=True).to(dev)
        with torch.enable_grad():
            dt(torch.randn(1, 4, 8, device=dev))


# --------------------------------------------------------------------------- full-size models
def test_sao_full_size_decode_and_encode(dev):
    """BASELINE configs 1/2 shapes: z [1,64,216] -> [1,2,442368] and back.  EVERY one of the 884 736 output samples is
    compared with the oracle run on this box (the oracle itself is pinned to the reference at the golden points,
    tests/test_oracle_golden.py), plus the reference's recorded points directly."""
    g = H.golden("sao_full")
    m = H.build("sao", 0)
    H.check_checksums(m.state_dict(), g)
    sd = {n: p.clone() for n, p in m.state_dict().items()}
    zc = torch.randn(1, 64, 216, generator=torch.Generator().manual_seed(1))
    xc = 0.1 * torch.randn(1, 2, 442368, generator=torch.Generator().manual_seed(2))
    ref = O.oobleck_decoder(H.split_sd(sd, "decoder."), zc, H.strides_of("sao"))
    m.to(dev).set_precision("bf16")
    y = m.decode(zc.to(dev))
    assert y.shape == (1, 2, 442368)
    idx = H.t(g["dec_idx"]).long()
    assert maxerr(ref[:, :, idx], g["dec_out_at_idx"]) <= 5e-6          # the checker agrees with the reference here
    err = maxerr(y, ref)
    H.report("SAO decode bf16, all 884736 samples (budget 1e-3, abs max %.3f)" % float(g["dec_abs_max"]), err)
    assert err <= TOL_BF16
    assert maxerr(y[:, :, idx.to(dev)], g["dec_out_at_idx"]) <= TOL_BF16
    assert abs(float((y.double() ** 2).sum()) - float(g["dec_sq_sum"])) <= 2e-2 * float(g["dec_sq_sum"])
    e = m.encode(xc.to(dev))
    erre = maxerr(e, g["enc_out"])
    H.report("SAO encode bf16, all latents (abs max %.3f)" % float(np.abs(g["enc_out"]).max()), erre)
    assert erre <= bf16_tol(g["enc_out"])
    m.set_precision("fp32")
    err32 = maxerr(m.decode(zc.to(dev)), ref)
    H.report("SAO decode fp32 mode, all samples (budget 1e-5)", err32)
    assert err32 <= TOL_F32


@pytest.mark.parametrize("B,T", [(1, 6), (2, 24)])
def test_sao_fp32_mode_short_clip(dev, B, T):
    """fp32 mode on the graded architecture: tensor cores through the bf16x3 operand split, <= 1e-5."""
    m = H.build("sao", 0)
    H.randomize_snake(m, 3)
    sd = m.state_dict()
    z = torch.randn(B, 64, T, generator=torch.Generator().manual_seed(5))
    x = 0.1 * torch.randn(B, 2, 2048 * T, generator=torch.Generator().manual_seed(6))
    ref = O.oobleck_decoder(H.split_sd(sd, "decoder."), z, H.strides_of("sao"))
    ref_e = O.oobleck_encoder(H.split_sd(sd, "encoder."), x, H.strides_of("sao"))
    m.to(dev)
    err, err_e = maxerr(m.decode(z.to(dev)), ref), maxerr(m.encode(x.to(dev)), ref_e)
    print(f"SAO fp32 mode B={B} T={T}: decode err {err:.2e}, encode err {err_e:.2e} (latent abs max {float(ref_e.abs().max()):.2f})")
    assert err <= TOL_F32
    # BASELINE.json states the fp32-mode budget for the waveform only; the encoder's latents come out of much larger
    # intermediate activations, where the 16-17 significant bits of the bf16 (hi | lo) operands leave ~2e-5
    assert err_e <= 5e-5 * max(1.0, float(ref_e.abs().max()))


@pytest.mark.parametrize("name,D", [("o12_d256", 256), ("o12_d512", 512), ("o12_d1024", 1024)])
def test_o12_short_clip_decode_encode(dev, name, D):
    """The three 12.5 Hz widths ("dim512" / "dim1024" / "dim2048") against the reference's recorded outputs: absolute
    1e-3 on the waveform in bf16 mode, 1e-5 in fp32 mode."""
    g = H.golden(name)
    m = H.build(name, 0)
    H.check_checksums(m.state_dict(), g)
    m.to(dev).set_precision("bf16")
    z = torch.randn(1, D, 16, generator=torch.Generator().manual_seed(1)).to(dev)
    x = (0.1 * torch.randn(1, 1, 1280 * 16, generator=torch.Generator().manual_seed(2))).to(dev)
    y = m.decode(z)
    err = maxerr(y, g["dec_out"])
    H.report(f"O12 latent {D} decode bf16 T=16", err)
    assert y.shape == (1, 1, 20480) and err <= TOL_BF16
    e = m.encode(x)
    assert e.shape == (1, 2 * D, 16)
    erre = maxerr(e, g["enc_out"])
    H.report(f"O12 latent {D} encode bf16 T=16 (abs max {float(np.abs(g['enc_out']).max()):.3f})", erre)
    assert erre <= bf16_tol(g["enc_out"])
    m.set_precision("fp32")
    err32 = maxerr(m.decode(z), g["dec_out"])
    H.report(f"O12 latent {D} decode fp32 mode T=16", err32)
    assert err32 <= TOL_F32


def test_config3_o12_latent512_full_length_vs_oracle(dev):
    """BASELINE config 3 at its own clip length: [2,512,375] -> [2,1,480000]; every sample against the oracle run on
    this box, clip 0 also against the reference's recorded points (tests/golden/o12_full.npz)."""
    g = H.golden("o12_full")
    m = H.build("o12_d512", 0)
    sd = H.split_sd({n: p.clone() for n, p in m.state_dict().items()}, "decoder.")
    z = torch.cat([torch.randn(1, 512, 375, generator=torch.Generator().manual_seed(1)),
                   torch.randn(1, 512, 375, generator=torch.Generator().manual_seed(5))])
    ref = O.oobleck_decoder(sd, z, H.strides_of("o12_d512"))
    idx = H.t(g["idx"]).long()
    assert maxerr(ref[:1, :, idx], g["d512_at_idx"]) <= 5e-6
    m.to(dev).set_precision("bf16")
    y = m.decode(z.to(dev))
    assert y.shape == (2, 1, 480000)
    err = maxerr(y, ref)
    H.report("config 3 (O12 latent 512, T=375) decode bf16, all 2 x 480000 samples (budget 1e-3, abs max %.3f)"
             % float(g["d512_abs_max"]), err)
    assert err <= TOL_BF16
    assert maxerr(y[:1, :, idx.to(dev)], g["d512_at_idx"]) <= TOL_BF16
    m.set_precision("fp32")
    err32 = maxerr(m.decode(z[:1].to(dev)), ref[:1])
    H.report("config 3 decode fp32 mode, all samples (budget 1e-5)", err32)
    assert err32 <= TOL_F32


def test_batch_items_are_independent(dev):
    """Batch sharding relies on it: decoding a batch == decoding each clip alone (bit-identical)."""
    m = H.build("mid", 0).to(dev).set_precision("bf16")
    z = torch.randn(4, 64, 40, device=dev)
    y = m.decode(z)
    for i in range(4):
        assert torch.equal(y[i:i + 1], m.decode(z[i:i + 1]))


# --------------------------------------------------------------------------- chunked / pretransform
def test_chunked_decode_encode_match_reference(dev):
    g = H.golden("chunked")
    tiny = H.golden("tiny_ae")
    m = H.build("tiny", 0)
    m.load_state_dict(_sd_from_golden(tiny))
    m.to(dev)
    z = H.t(g["z"]).to(dev)
    y = m.decode_audio(z, chunked=True, overlap=32, chunk_size=128)
    assert y.dtype == torch.float32 and maxerr(y, g["dec_chunked"]) <= TOL_F32
    assert maxerr(m.decode_audio(z, chunked=True, overlap=16, chunk_size=64), g["dec_chunked_64_16"]) <= TOL_F32
    assert maxerr(m.decode_audio(z), g["dec_full"]) <= TOL_F32
    with pytest.raises(UnboundLocalError):
        m.decode_audio(z[:, :, :100], chunked=True)
    ms = H.build("tiny_sym", 5)
    ms.load_state_dict({kk[len("sym_sd."):]: H.t(g[kk]) for kk in g.files if kk.startswith("sym_sd.")})
    ms.to(dev)
    e = ms.encode_audio(H.t(g["x"]).to(dev), chunked=True, overlap=32, chunk_size=128)
    assert maxerr(e, g["enc_chunked"]) <= TOL_F32
    with pytest.raises(RuntimeError):
        m.encode_audio(H.t(g["x"]).to(dev), chunked=True)      # encoder emits 2*latent_dim: reference errors too


def test_pretransform_scale_and_iterate_batch(dev):
    tiny = H.golden("tiny_ae")
    cfg = H.CONFIGS["tiny"]
    pt = k.create_pretransform_from_config({"type": "autoencoder", "config": cfg["model"], "scale": 2.0,
                                            "iterate_batch": True}, 16000)
    pt.load_state_dict(_sd_from_golden(tiny))
    pt.to(dev)
    y = pt.decode(H.t(tiny["z"]).to(dev) / 2.0)
    assert maxerr(y, tiny["dec_out"]) <= TOL_F32
    e = pt.encode(H.t(tiny["x"]).to(dev))
    assert maxerr(e * 2.0, tiny["enc_out"]) <= TOL_F32


# --------------------------------------------------------------------------- latent sampling (bit exact)
def test_sampling_bit_exact_vs_reference(dev):
    g = H.golden("sampling")
    mean, scale, noise = (H.t(g[n]).to(dev) for n in ("mean", "scale", "noise"))
    lat, kl = k.vae_sample(mean, scale, noise)
    assert torch.equal(lat.cpu(), H.t(g["vae_latents"]))
    assert abs(float(kl) - float(g["vae_kl"])) <= 1e-5 * abs(float(g["vae_kl"]))
    assert torch.equal(k.sample(mean, "fix", noise=noise).cpu(), H.t(g["fix"]))
    gau = k.sample(mean, "gaussian", noise=H.t(g["noise_g"]).to(dev), std_noise=H.t(g["std_noise"]).to(dev))
    assert torch.equal(gau.cpu(), H.t(g["gaussian"]))
    assert k.sample(mean, "anything else") is mean
    fb = k.sample(mean.bfloat16(), "fix", noise=H.t(g["noise_bf"]).to(dev).bfloat16())
    assert fb.dtype == torch.bfloat16 and torch.equal(fb.float().cpu(), H.t(g["fix_bf"]))
    # LM layout [B, T, D] (model_sigmaVAE.py:68) and RNG-stream parity with torch.randn_like
    mt = mean.transpose(1, 2).contiguous()
    torch.manual_seed(3)
    a = k.sample(mt, "fix")
    torch.manual_seed(3)
    b = mt + torch.tensor(0.5).to(dev) * torch.randn_like(mt)
    assert torch.equal(a, b)
    torch.manual_seed(4)
    a = k.sample(mt, "gaussian")
    torch.manual_seed(4)
    s = torch.randn(mt.size(0), device=dev, dtype=mt.dtype) * (torch.tensor(0.5) / 0.8).to(dev)
    b = mt + s.view(-1, 1, 1) * torch.randn_like(mt)
    assert torch.equal(a, b)


def test_encode_sample_decode_roundtrip_config2_shape(dev):
    """BASELINE config 2 data flow at reduced batch: encode -> chunk(2) -> sample('fix') -> decode."""
    m = H.build("sao", 0).to(dev).set_precision("bf16")
    x = 0.1 * torch.randn(2, 2, 2048 * 12, device=dev)
    enc = m.encode(x)
    mean, _ = enc.chunk(2, dim=1)
    zl = k.sample(mean.contiguous(), "fix")
    y = m.decode(zl)
    assert enc.shape == (2, 128, 12) and y.shape == x.shape and bool(torch.isfinite(y).all())
    sd = {n: p.cpu() for n, p in m.state_dict().items()}
    ref = O.oobleck_decoder(H.split_sd(sd, "decoder."), zl.cpu(), H.strides_of("sao"))
    assert maxerr(y, ref) <= TOL_BF16


def test_cuda_graph_replay_matches_eager(dev):
    m = H.build("mid", 0, snake_seed=7).to(dev).set_precision("bf16")
    z1 = torch.randn(1, 64, 32, device=dev)
    z2 = torch.randn(1, 64, 32, device=dev)
    y1, y2 = m.decode(z1), m.decode(z2)
    m.decoder.enable_cuda_graphs(True)
    g1 = m.decode(z1)
    g2 = m.decode(z2)          # replay with new input
    g1b = m.decode(z1)
    assert torch.equal(g1, y1) and torch.equal(g2, y2) and torch.equal(g1b, y1)
    z3 = torch.randn(2, 64, 17, device=dev)        # a second shape gets its own graph
    assert torch.equal(m.decode(z3), m.decoder.enable_cuda_graphs(False)(z3))


def test_o12_full_length_batch_decode_properties(dev):
    """BASELINE config 3 shape at reduced batch: [4,512,375] -> [4,1,480000]; size-independent properties:
    batch independence (bit-identical to per-clip decode) and time locality (receptive field +-10 frames:
    frames far from a perturbation are unchanged)."""
    m = H.build("o12_d512", 0).to(dev).set_precision("bf16")
    z = torch.randn(4, 512, 375, device=dev)
    y = m.decode(z)
    assert y.shape == (4, 1, 480000) and bool(torch.isfinite(y).all())
    assert torch.equal(y[2:3], m.decode(z[2:3]))
    z2 = z.clone()
    z2[:, :, 200] += 1.0
    y2 = m.decode(z2)
    d = (y2 - y).abs().amax(dim=(0, 1))
    assert float(d[: 1280 * 185].max()) == 0.0 and float(d[1280 * 215:].max()) == 0.0
    assert float(d[1280 * 195: 1280 * 206].max()) > 0.0


def test_fused_residual_unit_matches_two_kernel_path(dev):
    """The one-kernel ResidualUnit (conv_ru.cuh, 128-channel stages) against the k7 + k1 two-kernel path of the
    same library (KVAE_NO_RU_FUSION=1) and against the oracle, incl. multi-tile persistence (T*40 rows)."""
    import os
    m = H.build("mid", 0, snake_seed=7)
    sd = H.split_sd(m.state_dict(), "decoder.")
    z = torch.randn(3, 64, 211, generator=torch.Generator().manual_seed(4))
    ref = O.oobleck_decoder(sd, z, H.strides_of("mid"))
    m.to(dev).set_precision("bf16")
    y_fused = m.decode(z.to(dev))
    os.environ["KVAE_NO_RU_FUSION"] = "1"
    try:
        m2 = H.build("mid", 0, snake_seed=7).to(dev).set_precision("bf16")
        y_split = m2.decode(z.to(dev))
    finally:
        del os.environ["KVAE_NO_RU_FUSION"]
    assert maxerr(y_fused, ref) <= bf16_tol(ref) and maxerr(y_split, ref) <= bf16_tol(ref)
    # same arithmetic in both forms (bf16 operands, fp32 accumulation, same rounding points)
    assert float((y_fused - y_split).abs().max()) <= 2e-5 * float(ref.abs().max())


def test_pipelined_residual_unit_bit_identical_across_grids(dev):
    """conv_ru2_kernel (two TMEM accumulators, GEMM2 of tile i inside GEMM1 of tile i+1) carries state from tile to
    tile of a CTA: the waveform must be bit-identical whatever the number of tiles per CTA.  KVAE_RU_GRID=5 and 7 force
    ~20 and ~14 of the 99 tiles per CTA through the cross-tile pipeline."""
    import os
    z = torch.randn(3, 64, 211, generator=torch.Generator().manual_seed(4)).to(dev)
    outs = {}
    for name, env in (("ru2", {}), ("ru2_grid5", {"KVAE_RU_GRID": "5"}), ("ru2_grid7", {"KVAE_RU_GRID": "7"})):
        os.environ.update(env)
        try:
            m = H.build("mid", 0, snake_seed=7).to(dev).set_precision("bf16")
            outs[name] = m.decode(z)
            torch.cuda.synchronize()
        finally:
            for key in env:
                del os.environ[key]
    assert bool(torch.isfinite(outs["ru2"]).all())
    for name in ("ru2_grid5", "ru2_grid7"):
        assert torch.equal(outs["ru2"], outs[name]), name


def test_host_pipeline_equals_direct_calls(dev):
    """kalle_audio_b200.HostPipeline (pinned host buffers, copy streams, double-buffered device input): five
    batches in flight give exactly the tensors of five synchronous host -> device -> decode -> host calls."""
    m = H.build("mid", 0, snake_seed=7).to(dev).set_precision("bf16")
    zs = [torch.randn(2, 64, 50 + 3 * i, generator=torch.Generator().manual_seed(20 + i)).pin_memory() for i in range(5)]
    direct = [m.decode(z.to(dev)).cpu() for z in zs]
    outs = [torch.empty_like(d).pin_memory() for d in direct]
    pipe = k.HostPipeline(m.decode, dev)
    for z, o in zip(zs, outs):
        pipe.submit(z, o)
    pipe.synchronize()
    for d, o in zip(direct, outs):
        assert torch.equal(d, o)
    # one output buffer reused by consecutive submissions of one shape: the last submission wins
    same = [zs[0], (zs[0] * 0.5).pin_memory(), (zs[0] * 0.25).pin_memory()]
    y = torch.empty_like(direct[0]).pin_memory()
    for z in same:
        pipe.submit(z, y)
    pipe.join()
    torch.cuda.synchronize()
    assert torch.equal(y, m.decode(same[-1].to(dev)).cpu())
    with pytest.raises(ValueError):
        pipe.submit(zs[0].to(dev), y)


def test_config4_chunked_decode_o12_latent1024_vs_oracle(dev):
    """BASELINE config 4: O12 latent-1024 decoder, decode_audio(chunked=True, chunk 128, overlap 32) over T=375
    (4 windows) against the oracle's restatement of the reference's chunk/overlap stitching
    (stable_audio_tools/models/autoencoders.py:514-560) run on this box, against the reference's recorded points,
    and against the unchunked decode (overlap/2 = 16 frames > receptive field 10 frames)."""
    g = H.golden("o12_full")
    m = H.build("o12_d1024", 0)
    sd = H.split_sd({n: p.clone() for n, p in m.state_dict().items()}, "decoder.")
    st = H.strides_of("o12_d1024")
    zc = torch.randn(1, 1024, 375, generator=torch.Generator().manual_seed(1))
    ref = O.decode_audio_chunked(lambda zz: O.oobleck_decoder(sd, zz, st), zc, 1280, 1, overlap=32, chunk_size=128)
    idx = H.t(g["idx"]).long()
    assert maxerr(ref[:, :, idx], g["d1024_chunked_at_idx"]) <= 5e-6
    m.to(dev).set_precision("bf16")
    z = zc.to(dev)
    full = m.decode_audio(z)
    chunked = m.decode_audio(z, chunked=True, overlap=32, chunk_size=128)
    assert full.shape == chunked.shape == (1, 1, 480000)
    err = maxerr(chunked, ref)
    H.report("config 4 (O12 latent 1024, T=375, chunked 128/32) decode bf16, all 480000 samples (budget 1e-3, abs max %.3f)"
             % float(g["d1024_abs_max"]), err)
    assert err <= TOL_BF16
    assert maxerr(chunked[:, :, idx.to(dev)], g["d1024_chunked_at_idx"]) <= TOL_BF16
    assert maxerr(full[:, :, idx.to(dev)], g["d1024_at_idx"]) <= TOL_BF16
    # identical arithmetic per output row away from window edges -> differences only from fp32 summation order: none
    assert float((full - chunked).abs().max()) <= 1e-6
    m.decoder.enable_cuda_graphs(True)
    assert torch.equal(m.decode_audio(z, chunked=True, overlap=32, chunk_size=128), chunked)
    m.decoder.enable_cuda_graphs(False)
    m.set_precision("fp32")
    err32 = maxerr(m.decode_audio(z, chunked=True, overlap=32, chunk_size=128), ref)
    H.report("config 4 chunked decode fp32 mode, all samples (budget 1e-5)", err32)
    assert err32 <= TOL_F32


def test_pcm16_tail_bit_exact(dev):
    """infer_0828_sigma.py:298: output.to(float32).div(max|output|).clamp(-1, 1).mul(32767).to(int16)."""
    torch.manual_seed(11)
    for x in (0.3 * torch.randn(2, 2, 50001), torch.randn(1, 1, 7).bfloat16(), 1e-3 * torch.randn(3, 1, 4096)):
        ref = x.to(torch.float32).div(torch.max(torch.abs(x.to(torch.float32)))).clamp(-1, 1).mul(32767).to(torch.int16)
        got = k.to_pcm16(x.to(dev))
        assert got.dtype == torch.int16 and torch.equal(got.cpu(), ref)


@pytest.mark.parametrize("precision,hop", [("fp32", 7), ("bf16", 16), ("fp32", 96)])
def test_streaming_decoder_equals_full_decode(dev, precision, hop):
    """StreamingDecoder (exact receptive-field context) against one decode of the whole sequence, ragged pushes."""
    m = H.build("tiny", 0, snake_seed=7).to(dev)
    m.decoder.set_precision(precision)
    z = torch.randn(2, 4, 211, generator=torch.Generator().manual_seed(4)).to(dev)
    full = m.decoder(z)
    sd = k.StreamingDecoder(m.decoder, hop=hop, use_cuda_graphs=(hop == 16))
    assert (sd.left, sd.right) == (15, 15)
    pieces, pos = [], 0
    for n in [1, 0, 5, 40, 3, 97, 20, 45]:
        pieces.append(sd.push(z[:, :, pos:pos + n]))
        pos += n
    assert pos == 211
    emitted = sum(p.shape[2] for p in pieces)
    assert emitted % (hop * 40) == 0 and emitted <= (211 - sd.right) * 40      # only final frames were emitted
    pieces.append(sd.flush())
    y = torch.cat(pieces, dim=2)
    assert y.shape == full.shape
    tol = 2e-6 if precision == "fp32" else 1e-6      # same inputs, same per-output summation order
    assert float((y - full).abs().max()) <= tol * max(1.0, float(full.abs().max()))


def test_fp16_stream_saturates_instead_of_overflowing(dev):
    """Inference plans keep the residual stream in fp16; activations beyond +-65504 must saturate, not become inf/NaN."""
    m = H.build("sao", 0).to(dev).set_precision("bf16")
    with torch.no_grad():
        for name, p in m.decoder.named_parameters():
            if name.endswith("layers.1.bias") and p.numel() == 128:      # biases of the 128-channel stages
                p.fill_(3.0e5)
    z = torch.randn(1, 64, 4, generator=torch.Generator().manual_seed(1)).to(dev)
    y = m.decode(z)
    assert bool(torch.isfinite(y).all())


def test_full_size_properties_sao_bench_shape(dev):
    """BASELINE configs[1] at its full size (16 clips x 10.03 s, bf16 mode), checked through size-independent
    properties: batch items are independent (what batch sharding relies on), the decoder is time-invariant away
    from the clip edges (what chunked / streaming decode relies on), and the encode -> decode round trip of a
    batch equals the round trip of one of its clips alone."""
    m = H.build("sao", 0).to(dev).set_precision("bf16")
    z = torch.randn(16, 64, 216, generator=torch.Generator().manual_seed(1)).to(dev)
    y = m.decode(z)
    assert y.shape == (16, 2, 442368) and bool(torch.isfinite(y).all())
    y3 = m.decode(z[3:4])
    assert float((y[3:4] - y3).abs().max()) == 0.0                     # same tiles, same summation order
    # time invariance: drop 8 latent frames on the left; 10 frames = the receptive field (StreamingDecoder)
    ys = m.decode(z[:2, :, 8:])
    lo, hi = (8 + 10) * 2048, (216 - 10) * 2048
    d = float((y[:2, :, lo:hi] - ys[:, :, lo - 8 * 2048:hi - 8 * 2048]).abs().max())
    assert d <= 2e-6 * max(1.0, float(y.abs().max())), d
    x = (0.1 * torch.randn(16, 2, 442368, generator=torch.Generator().manual_seed(2))).to(dev)
    e = m.encode(x)
    assert e.shape == (16, 128, 216)
    assert float((e[5:6] - m.encode(x[5:6])).abs().max()) == 0.0
    # golden anchor at this size: clip 0 of the batch is the fixture's input (same seed), sampled points
    g = H.golden("sao_full")
    z[0] = torch.randn(1, 64, 216, generator=torch.Generator().manual_seed(1))[0].to(dev)
    idx = H.t(g["dec_idx"]).long().to(dev)
    err = maxerr(m.decode(z)[:1][:, :, idx], g["dec_out_at_idx"])
    H.report("configs[1] shape (16 x 216 frames): clip 0 at the reference's recorded points", err)
    assert err <= TOL_BF16


def test_nearest_upsample_decoder_vs_reference(dev):
    """use_nearest_upsample=True (autoencoders.py:87-96; part of the preserved constructor signature): same state_dict
    keys as the reference, outputs against its recorded decode -- tiny model (CUDA-core path, fp32), C=64 model
    (tcgen05 path in bf16 and fp32 mode, with final_tanh) -- and the stand-alone block against the oracle."""
    g = H.golden("nearest")
    torch.manual_seed(0)
    d = k.OobleckDecoder(out_channels=2, channels=8, latent_dim=4, c_mults=[1, 2, 4], strides=[2, 4, 5], use_snake=True,
                         use_nearest_upsample=True, final_tanh=False).eval()
    sd = {kk[len("tiny_sd."):]: H.t(g[kk]) for kk in g.files if kk.startswith("tiny_sd.")}
    assert list(d.state_dict().keys()) == list(sd.keys())
    d.load_state_dict(sd)
    d.to(dev)
    y = d(H.t(g["tiny_z"]).to(dev))
    assert y.shape == g["tiny_out"].shape and maxerr(y, g["tiny_out"]) <= TOL_F32
    blk = d.layers[1]                                    # stand-alone DecoderBlock: Upsample + 'same' conv leaf kernels
    xb = torch.randn(2, 32, 9, generator=torch.Generator().manual_seed(3))
    ref = O.decoder_block({"b." + n: p.cpu() for n, p in blk.state_dict().items()}, "b", xb, 5, use_nearest_upsample=True)
    assert maxerr(blk(xb.to(dev)), ref) <= 5e-5
    torch.manual_seed(0)
    d = k.OobleckDecoder(out_channels=2, channels=64, latent_dim=64, c_mults=[1, 2, 4], strides=[2, 4, 5], use_snake=True,
                         use_nearest_upsample=True, final_tanh=True).eval()
    H.randomize_snake(d, 7)
    H.check_checksums(d.state_dict(), g)
    d.to(dev)
    z = H.t(g["mid_z"]).to(dev)
    e32 = maxerr(d.set_precision("fp32")(z), g["mid_out"])
    e16 = maxerr(d.set_precision("bf16")(z), g["mid_out"])
    H.report("nearest-upsample decoder (C=64, tcgen05): fp32 mode / bf16 mode", f"{e32:.3e} / {e16:.3e}")
    # This random-init fixture keeps its activations at ~2.4 through all three stages (output abs-max 0.83 after tanh;
    # the SAO waveform is 0.125): a CPU emulation of nothing but bf16 rounding of the conv operands gives 1.45e-2 on it
    # (same emulation on the ConvTranspose fixture: 2.2e-3), so the budgets scale with the fixture as in bf16_tol
    assert e32 <= TOL_F32 * max(1.0, float(np.abs(g["mid_out"]).max()) / 0.125) and e16 <= 2e-2
    with pytest.raises(NotImplementedError):
        with torch.enable_grad():
            d(z.clone().requires_grad_(True))


def _small_128_decoder(dev, latent=64):
    torch.manual_seed(0)
    d = k.OobleckDecoder(out_channels=2, channels=128, latent_dim=latent, c_mults=[1, 2], strides=[2, 4], use_snake=True,
                         final_tanh=False).eval()
    H.randomize_snake(d, 7)
    return d.to(dev)


@pytest.mark.parametrize("precision,graphs", [("bf16", False), ("bf16", True), ("fp32", False)])
def test_stateful_streaming_equals_unchunked_bit_for_bit(dev, precision, graphs):
    """kvae_decode_stream_*: persistent per-layer halo state, 0 % recompute.  Ragged pushes (incl. pushes shorter than a
    layer's halo and an empty one) through a 128/256-channel decoder (fused ResidualUnits at C=128, separate k7/k1 at
    C=256, transposed convs, tensor-core tail): the concatenation equals ONE decode of the whole sequence exactly, and
    the decode equals the oracle."""
    d = _small_128_decoder(dev).set_precision(precision)
    z = torch.randn(2, 64, 211, generator=torch.Generator().manual_seed(4)).to(dev)
    full = d(z)
    sd = k.StreamingDecoder(d, hop=16, use_cuda_graphs=graphs, stateful=True, max_frames=64)
    for rep in range(2):                                   # a second stream on the same object starts from clean state
        pieces, pos = [], 0
        for n in [1, 0, 5, 40, 3, 97, 20, 45]:
            pieces.append(sd.push(z[:, :, pos:pos + n]))
            pos += n
        assert sd.stateful and sd.recompute_factor == 1.0 and pos == 211
        emitted = sum(p.shape[2] for p in pieces)
        assert emitted == 211 * 8 - sd.lookahead and sd.lookahead > 0
        pieces.append(sd.flush())
        y = torch.cat(pieces, dim=2)
        assert y.shape == full.shape
        assert torch.equal(y, full), float((y - full).abs().max())
    ref = O.oobleck_decoder({n: p.cpu() for n, p in d.state_dict().items()}, z.cpu(), [2, 4])
    # (a fixture with perturbed SnakeBeta parameters, not a BASELINE config: budgets scale with its magnitude, see bf16_tol)
    assert maxerr(full, ref) <= (TOL_F32 * max(1.0, float(ref.abs().max()) / 0.125) if precision == "fp32" else bf16_tol(ref))
    # constant-hop steady state (what a CUDA graph replays)
    sd2 = k.StreamingDecoder(d, hop=32, use_cuda_graphs=graphs, stateful=True, max_frames=32)
    out = [sd2.push(z[:, :, i:i + 32]) for i in range(0, 192, 32)] + [sd2.push(z[:, :, 192:])]
    out.append(sd2.flush())
    assert torch.equal(torch.cat(out, dim=2), full)


def test_config4_stateful_stream_o12_latent1024(dev):
    """BASELINE config 4's model (O12 latent 1024, batch 1) streamed in 96-frame hops with CUDA-graph replay: equals
    the unchunked decode bit for bit (which test_config4_chunked_decode_... pins against the oracle and the reference)."""
    m = H.build("o12_d1024", 0).to(dev).set_precision("bf16")
    z = torch.randn(1, 1024, 375, generator=torch.Generator().manual_seed(1)).to(dev)
    full = m.decoder(z)
    sd = k.StreamingDecoder(m.decoder, hop=96, use_cuda_graphs=True, stateful=True)
    out = [sd.push(z[:, :, i:i + 96]) for i in range(0, 375, 96)]
    # the decoder's receptive field is 10 latent frames (SURVEY section 5); transposed convs emit whole input rows, +<1 frame
    assert 10 * 1280 <= sd.lookahead <= 11 * 1280
    out.append(sd.flush())
    y = torch.cat(out, dim=2)
    assert y.shape == full.shape == (1, 1, 480000)
    assert torch.equal(y, full), float((y - full).abs().max())
    g = H.golden("o12_full")
    idx = H.t(g["idx"]).long().to(dev)
    err = maxerr(y[:, :, idx], g["d1024_at_idx"])
    H.report("config 4 stateful stream (96-frame hops, 0 % recompute) at the reference's recorded points", err)
    assert err <= TOL_BF16
    with pytest.raises(k.KvaeError):
        k.StreamingDecoder(H.build("tiny", 0).to(dev).decoder, stateful=True).push(torch.randn(1, 4, 8, device=dev))
