"""CPU tests of the host-side mirror of the reference interface (no GPU needed)."""
import copy

import pytest
import torch

import helpers as H
import kalle_audio_b200 as k
from kalle_audio_b200.autoencoders import _chunk_starts


def test_state_dict_keys_and_shapes_sao():
    m = H.build("sao", 0)
    sd = m.state_dict()
    assert sd["decoder.layers.0.weight_g"].shape == (2048, 1, 1)
    assert sd["decoder.layers.1.layers.1.weight_v"].shape == (2048, 1024, 16)   # first ConvTranspose1d: [Cin,Cout,K]
    assert sd["decoder.layers.1.layers.1.weight_g"].shape == (2048, 1, 1)       # norm over in-channels
    assert "decoder.layers.7.bias" not in sd and "decoder.layers.7.weight_v" in sd  # final conv bias=False
    assert sd["encoder.layers.7.weight_v"].shape == (128, 2048, 3)
    n_dec = sum(v.numel() for kk, v in sd.items() if kk.startswith("decoder."))
    n_enc = sum(v.numel() for kk, v in sd.items() if kk.startswith("encoder."))
    assert 77e6 < n_dec < 79e6 and 77e6 < n_enc < 79e6                           # SURVEY: 78.0 M + 78.1 M
    convs = [mm for mm in m.decoder.modules() if isinstance(mm, (k.WNConv1d, k.WNConvTranspose1d))]
    snakes = [mm for mm in m.decoder.modules() if isinstance(mm, k.SnakeBeta)]
    assert len(convs) == 37 and len(snakes) == 36                                # SURVEY section 2


def test_weight_g_is_norm_of_v_at_init():
    torch.manual_seed(0)
    c = k.WNConv1d(8, 16, 7, padding=3)
    assert torch.allclose(c.weight_g.flatten(), c.weight_v.flatten(1).norm(dim=1), atol=1e-6)
    ct = k.WNConvTranspose1d(8, 16, 4, stride=2, padding=1)
    assert ct.weight_g.shape == (8, 1, 1) and ct.weight_v.shape == (8, 16, 4)


def test_load_state_dict_roundtrip_and_strict_keys():
    a, b = H.build("tiny", 0), H.build("tiny", 1)
    assert not torch.equal(a.decoder.layers[0].weight_v, b.decoder.layers[0].weight_v)
    missing, unexpected = b.load_state_dict(a.state_dict(), strict=True)
    assert not missing and not unexpected
    assert torch.equal(a.decoder.layers[0].weight_v, b.decoder.layers[0].weight_v)


def test_cpu_tensors_fail_loudly():
    m = H.build("tiny", 0)
    with pytest.raises(k.KvaeError, match="no CPU path"):
        m.decode(torch.randn(1, 4, 8))
    with pytest.raises(k.KvaeError):
        m.encode(torch.randn(1, 2, 80))
    with pytest.raises(k.KvaeError):
        k.SnakeBeta(4)(torch.randn(1, 4, 8))
    with pytest.raises(k.KvaeError):
        k.sample(torch.randn(2, 3, 4))
    assert k.sample(torch.randn(2, 3), "none").shape == (2, 3)      # pass-through branch needs no device


def test_unsupported_variants_raise():
    with pytest.raises(NotImplementedError):
        k.OobleckDecoder(use_snake=False)
    # use_nearest_upsample=True is built (autoencoders.py:87-96): same module tree / keys as the reference
    d = k.OobleckDecoder(out_channels=2, channels=8, latent_dim=4, c_mults=[1, 2], strides=[2, 5], use_snake=True,
                         use_nearest_upsample=True)
    assert "layers.1.layers.1.1.weight_v" in d.state_dict() and "layers.1.layers.1.1.bias" not in d.state_dict()
    assert d.state_dict()["layers.1.layers.1.1.weight_v"].shape == (8, 16, 10)        # k = 2 * stride, 'same' padding
    with pytest.raises(NotImplementedError):
        k.OobleckEncoder(use_snake=True, antialias_activation=True)
    with pytest.raises(NotImplementedError):
        k.create_model_from_config({"model_type": "diffusion_cond"})
    with pytest.raises(NotImplementedError):
        k.create_bottleneck_from_config({"type": "rvq"})


def test_factories_and_pretransform_wiring():
    cfg = H.CONFIGS["tiny"]
    ae = k.create_model_from_config(cfg)
    assert isinstance(ae, k.AudioAutoencoder) and isinstance(ae.bottleneck, k.VAEBottleneck)
    assert ae.downsampling_ratio == 40 and ae.latent_dim == 4 and ae.io_channels == 2 and ae.min_length == 40
    pt = k.create_pretransform_from_config({"type": "autoencoder", "config": cfg["model"], "scale": 2.0,
                                            "iterate_batch": True}, 16000)
    assert pt.scale == 2.0 and pt.iterate_batch and not pt.enable_grad
    assert all(not p.requires_grad for p in pt.parameters())
    assert pt.encoded_channels == 4 and pt.downsampling_ratio == 40
    x, info = ae.bottleneck.encode(torch.ones(1, 8, 3), return_info=True)
    assert info == {} and torch.equal(x, torch.ones(1, 8, 3)) and torch.equal(ae.bottleneck.decode(x), x)


def test_chunk_window_starts_follow_reference_loop():
    assert _chunk_starts(300, 128, 96) == [0, 96, 172]
    assert _chunk_starts(128, 128, 96) == [0]
    assert _chunk_starts(375, 128, 96) == [0, 96, 192, 247]       # BASELINE config 4: 4 chunks over T=375
    assert _chunk_starts(320, 128, 96) == [0, 96, 192]
    with pytest.raises(UnboundLocalError):
        _chunk_starts(100, 128, 96)


def test_preprocess_audio_list_pads_to_ratio_and_fixes_channels():
    ae = H.build("tiny", 0)
    out = ae.preprocess_audio_list_for_encoder([torch.randn(1, 90), torch.randn(2, 61), torch.randn(70)], 16000)
    assert out.shape == (3, 2, 120)
    assert torch.equal(out[0, 0], out[0, 1]) and float(out[0, :, 90:].abs().sum()) == 0.0
    assert ae.preprocess_audio_for_encoder(torch.randn(1, 2, 80), 16000).shape == (1, 2, 80)


def test_deepcopy_and_remove_weight_norm_keys():
    m = H.build("tiny", 0)
    m2 = copy.deepcopy(m)
    assert list(m2.state_dict().keys()) == list(m.state_dict().keys())
    c = k.WNConv1d(4, 4, 3, padding=1)
    assert c.has_weight_norm and set(dict(c.named_parameters())) == {"bias", "weight_g", "weight_v"}


def test_precision_selection():
    m = H.build("tiny", 0)
    assert m.decoder._resolve_precision() == k._lib.KVAE_PREC_F32
    m.set_precision("bf16")
    assert m.decoder._resolve_precision() == k._lib.KVAE_PREC_BF16 and m.encoder._resolve_precision() == k._lib.KVAE_PREC_BF16
    m.set_precision(None)
    m.bfloat16()
    assert m.decoder._resolve_precision() == k._lib.KVAE_PREC_BF16
    with pytest.raises(ValueError):
        m.set_precision("fp8")


def test_decoder_context_frames_is_the_exact_receptive_field():
    """streaming.decoder_context_frames against a brute-force probe of the oracle decoder: perturb one latent
    frame and see which output frames move."""
    import torch
    import helpers as H
    from oracle import oobleck_oracle as O
    from kalle_audio_b200.streaming import decoder_context_frames
    assert decoder_context_frames([2, 4, 4, 8, 8]) == (10, 10)       # SAO; SURVEY.md Appendix C measured +-10
    assert decoder_context_frames([2, 4, 4, 5, 8]) == (10, 10)       # 12.5 Hz models
    g = H.golden("tiny_ae")
    sd = {k[len("sd.decoder."):]: H.t(g[k]) for k in g.files if k.startswith("sd.decoder.")}
    strides = H.strides_of("tiny")
    left, right = decoder_context_frames(strides)
    with torch.no_grad():
        z = torch.randn(1, 4, 64, generator=torch.Generator().manual_seed(0))
        y = O.oobleck_decoder(sd, z, strides)
        z2 = z.clone()
        z2[:, :, 32] += 1.0
        moved = ((O.oobleck_decoder(sd, z2, strides) - y).abs().amax((0, 1)) > 0).nonzero().flatten()
    ratio = 40
    # frame 32 is right context of frames down to 32 - right and left context of frames up to 32 + left
    assert int(moved.min()) // ratio == 32 - right and int(moved.max()) // ratio == 32 + left


def test_host_pipeline_has_no_cpu_path():
    with pytest.raises(ValueError, match="no CPU path"):
        k.HostPipeline(lambda x: x, torch.device("cpu"))


def test_bench_clock_sampler_windows():
    """bench.py's ClockSampler: statistics of the samples between two marks; a region shorter than the sampling
    period is widened by one sample on each side; throttle reasons are collected from the window only."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(H.__file__), "..", "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    s.proc = object()                       # pretend nvidia-smi is running

    def row(mhz, watts, power_cap=False, thermal=False):
        return ["0", str(mhz), "1965", str(watts), "0x0", "Not Active", "Active" if thermal else "Not Active",
                "Not Active", "Active" if power_cap else "Not Active"]
    s.rows = [row(1965, 200), row(1500, 990, power_cap=True), row(1600, 1000, power_cap=True), row(1965, 300),
              row(900, 250, thermal=True)]
    st = s.stats(1, 3)
    assert st["samples"] == 2 and st["sm_mhz"] == 1550.0 and st["power_w_max"] == 1000.0
    assert st["reasons"] == ["sw_power_cap"] and st["sm_max_mhz"] == 1965.0
    st = s.stats(2, 2)                       # empty window -> neighbours on both sides
    assert st["samples"] == 2 and st["sm_mhz"] == 1550.0
    st = s.stats(4, 5)                       # a single sample -> widened to rows 3..4
    assert st["samples"] == 2 and st["reasons"] == ["hw_thermal_slowdown"]
    assert s.mark() == 5
    s.proc = None
    assert s.stats()["reasons"] == ["nvidia-smi unavailable"]


def test_layer_model_flops_match_survey():
    """tools/layer_model.py (the work model behind DESIGN section 7) reproduces the algorithmic FLOP counts SURVEY.md
    section 8(d) measured on the reference modules: SAO decode 1089.145 G per 216-frame clip, O12 latent-512 decode
    1255.219 G per 375-frame clip."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("layer_model", os.path.join(os.path.dirname(H.__file__), "..", "tools",
                                                                               "layer_model.py"))
    lm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(lm)
    for arch, want in (("sao", 1089.145), ("o12", 1255.219)):
        total = sum(lm.model(l)["gflop"] for l in lm.decoder_layers(lm.ARCH[arch], 1))
        assert abs(total - want) < 2e-3 * want, (arch, total)


def test_library_environment_switches_are_the_kept_set():
    """The native library reads exactly these environment switches: KVAE_NO_RU_FUSION (the two-kernel reference of
    the fused ResidualUnit), KVAE_RU_GRID (many tiles per CTA) and KVAE_FAST_EPI / KVAE_WAVE_IN_CC / KVAE_TAIL_RAW (the
    kernel variants test_gpu_variants.py compares).  A new switch has to be added here on purpose."""
    import os
    import re
    csrc = os.path.join(os.path.dirname(k.__file__), "csrc")
    names, other = set(), []
    for fn in sorted(os.listdir(csrc)):
        with open(os.path.join(csrc, fn)) as f:
            src = f.read()
        for arg in re.findall(r"\b(?:getenv|env_flag)\(([^)]*)\)", src):
            lit = re.fullmatch(r'\s*"([^"]+)"\s*', arg)
            if lit:
                names.add(lit.group(1))
            elif arg.strip() not in ("name", "const char* name"):   # env_flag's own definition
                other.append((fn, arg))
    assert not other, other
    assert names == {"KVAE_NO_RU_FUSION", "KVAE_RU_GRID", "KVAE_FAST_EPI", "KVAE_WAVE_IN_CC", "KVAE_TAIL_RAW"}
