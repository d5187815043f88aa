"""Stateful streaming encode (StreamingEncoder / kvae_encode_stream_*): the concatenated pushes equal the whole-clip
encode bit for bit, whatever the push sizes, in both precision modes and with CUDA-graph replay."""
import math

import numpy as np
import pytest
import torch

import helpers as H
import kalle_audio_b200 as k

pytestmark = pytest.mark.gpu

RAGGED = [0, 1, 3, 7, 300, 2048, 513]     # shorter than the head's halo and than a stride, then longer pushes


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def out_length(L, strides):
    """The reference's floor arithmetic: each strided conv maps L rows to floor((L + 2p - 2s) / s) + 1."""
    for s in strides:
        p = math.ceil(s / 2)
        L = (L + 2 * p - 2 * s) // s + 1
    return L


def small_encoder(dev, precision):
    """Fused ResidualUnits at C = 128, separate k7 / k1 convs at C = 256, an odd stride, both head kernels."""
    torch.manual_seed(0)
    enc = k.OobleckEncoder(in_channels=2, channels=128, latent_dim=128, c_mults=[1, 2], strides=[2, 5], use_snake=True)
    H.randomize_snake(enc, 5)
    return enc.to(dev).eval().set_precision(precision)


def run_stream(se, x, sizes, right, ratio):
    """Pushes x in pieces of `sizes` (the rest in one piece), checks the emission bound after each, then flushes."""
    outs, n, emitted = [], 0, 0
    for m in sizes + [x.shape[2] - sum(sizes)]:
        y = se.push(x[:, :, n:n + m])
        n += m
        emitted += y.shape[2]
        bound = max(0, (n - right) // ratio)
        assert bound - 1 <= emitted <= bound, (n, emitted, bound)
        outs.append(y)
    outs.append(se.flush())
    return torch.cat(outs, dim=2)


@pytest.mark.parametrize("precision,graphs", [("bf16", False), ("bf16", True), ("fp32", True)])
def test_small_encoder_stream_equals_whole_encode(dev, precision, graphs):
    enc = small_encoder(dev, precision)
    strides, ratio = [2, 5], 10
    _, right = k.encoder_context_samples(strides)
    se = k.StreamingEncoder(enc, max_samples=4096, use_cuda_graphs=graphs)
    with torch.no_grad():
        x = 0.1 * torch.randn(2, 2, 10000, generator=torch.Generator().manual_seed(1)).to(dev)
        full = enc(x)
        got = run_stream(se, x, RAGGED, right, ratio)
        assert got.dtype == full.dtype and got.shape == full.shape
        assert torch.equal(got, full), float((got - full).abs().max())
        assert right <= se.lookahead <= right + ratio
        # the same object streams again after flush
        assert torch.equal(run_stream(se, x, RAGGED, right, ratio), full)
        # a constant hop in multiples of the ratio (the steady state that replays one graph per push)
        hop = 20 * ratio
        got = torch.cat([se.push(x[:, :, i:i + hop]) for i in range(0, x.shape[2], hop)] + [se.flush()], dim=2)
        assert torch.equal(got, full)
        # a length that is not a multiple of the ratio: the reference's floor arithmetic, as the ragged batch path
        for L in (9997, 10003):
            xl = 0.1 * torch.randn(2, 2, L, generator=torch.Generator().manual_seed(L)).to(dev)
            Lp = -(-L // ratio) * ratio
            padded = torch.nn.functional.pad(xl, (0, Lp - L))
            ref = enc(padded, valid_len=[L, L])[:, :, :out_length(L, strides)]
            got = run_stream(se, xl, RAGGED, right, ratio)
            assert got.shape == ref.shape, (L, got.shape, ref.shape)
            assert torch.equal(got, ref), (L, float((got - ref).abs().max()))


def test_o12_latent1024_stream_30s(dev):
    """The 12.5 Hz model with latent 1024 at its own length (30 s at 16 kHz) in 4-frame pushes with graph replay."""
    m = H.build("o12_d1024", 0).to(dev).set_precision("bf16")
    strides = list(H.strides_of("o12_d1024"))
    ratio = int(np.prod(strides))
    _, right = k.encoder_context_samples(strides)
    x = 0.1 * torch.randn(1, 1, 480000, generator=torch.Generator().manual_seed(2)).to(dev)
    with torch.no_grad():
        full = m.encoder(x)
        se = k.StreamingEncoder(m.encoder, use_cuda_graphs=True)
        hop = 4 * ratio
        got = torch.cat([se.push(x[:, :, i:i + hop]) for i in range(0, x.shape[2], hop)] + [se.flush()], dim=2)
    assert got.shape == full.shape and full.shape[2] == 375
    assert torch.equal(got, full), float((got - full).abs().max())
    assert right <= se.lookahead <= right + ratio


def test_sao_stream_full_clip(dev):
    """The SAO encoder on the 10 s stereo clip of test_sao_full_size_decode_and_encode: bit for bit the whole encode,
    and within that test's tolerance of the reference's recorded latents."""
    g = H.golden("sao_full")
    m = H.build("sao", 0)
    xc = 0.1 * torch.randn(1, 2, 442368, generator=torch.Generator().manual_seed(2))
    m.to(dev).set_precision("bf16")
    with torch.no_grad():
        x = xc.to(dev)
        full = m.encoder(x)
        se = k.StreamingEncoder(m.encoder, use_cuda_graphs=True)
        hop = 4 * 2048
        got = torch.cat([se.push(x[:, :, i:i + hop]) for i in range(0, x.shape[2], hop)] + [se.flush()], dim=2)
        assert torch.equal(got, full), float((got - full).abs().max())
        e = got if m.bottleneck is None else m.bottleneck.encode(got)
    ref = H.t(g["enc_out"]).float()
    err = float((e.float().cpu() - ref).abs().max())
    tol = 1e-3 * max(1.0, float(ref.abs().max()) / 0.125)
    H.report("SAO streaming encode bf16 (8192-sample pushes) vs the reference's latents", err)
    assert err <= tol


def test_stream_errors(dev):
    tiny = H.build("tiny", 0).to(dev)
    se = k.StreamingEncoder(tiny.encoder)
    with pytest.raises(k.KvaeError):
        se.push(torch.zeros(1, 2, 400, device=dev))
    se = k.StreamingEncoder(small_encoder(dev, "bf16"))
    se.push(torch.zeros(2, 2, 100, device=dev))
    with pytest.raises(ValueError):
        se.push(torch.zeros(1, 2, 100, device=dev))
