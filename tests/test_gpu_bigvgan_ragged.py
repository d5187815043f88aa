"""GPU checks of BigVGANFlowVAE's ragged batches: with ``valid_len``, every clip of ``extract_latents`` /
``inference_from_latents`` is ``torch.equal`` to the same call on that clip alone, rows past its output length are 0,
and whatever the caller left in the padding is ignored."""
import ctypes
import os
import sys

import pytest
import torch

import helpers as H
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


class AttrDict(dict):
    __getattr__ = dict.__getitem__


WIDE = AttrDict(BIGVGAN_H, causal=True, upsample_initial_channel=256, resblock="1", activation="snakebeta",
                resblock_dilation_sizes=[[1, 3, 5], [1, 3, 5]], snake_logscale=True)
BENCH = AttrDict(causal=True, latent_dim=512, use_vae=True, downsample_channels=[12, 24, 48, 96, 192, 384, 768],
                 downsample_rates=[2, 2, 4, 4, 4, 5], flow_hidden_channels=64, resblock_kernel_sizes=[3, 7, 11],
                 resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
                 upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=1024, resblock="1",
                 activation="snakebeta", snake_logscale=True)


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


def _padded(shape, lens, dev, dtype=torch.float32, pad=float("nan"), scale=1.0):
    x = scale * torch.randn(shape, generator=torch.Generator().manual_seed(sum(lens))).to(dev, dtype)
    for b, n in enumerate(lens):
        x[b, :, n:] = pad                           # the library must not read the caller's padding
    return x


def _check_decode(m, z, lens, noise=None, do_sample=False):
    y = m.inference_from_latents(z, do_sample=do_sample, noise=noise, valid_len=lens)
    assert y.shape == (z.shape[0], 1, m.wav_length(z.shape[2])) and y.dtype == z.dtype
    for b, n in enumerate(lens):
        nz = None if noise is None else noise[b:b + 1, :, :n]
        ref = m.inference_from_latents(z[b:b + 1, :, :n], do_sample=do_sample, noise=nz)
        L = m.wav_length(n)
        assert ref.shape[2] == L
        assert torch.equal(y[b:b + 1, :, :L], ref), f"clip {b} ({n} frames)"
        assert not y[b, :, L:].any()
    return y


def _check_encode(m, x, lens):
    y = m.extract_latents(x, valid_len=lens)
    assert y.shape[2] == m.latent_length(x.shape[2]) and y.dtype == x.dtype
    for b, n in enumerate(lens):
        ref = m.extract_latents(x[b:b + 1, :, :n])
        L = m.latent_length(n)
        assert ref.shape[2] == L
        assert torch.equal(y[b:b + 1, :, :L], ref), f"clip {b} ({n} samples)"
        assert not y[b, :, L:].any()
    return y


@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
def test_golden_config_ragged(dev, causal):
    m = _model(dict(BIGVGAN_H, causal=causal), dev).set_precision(None)
    T, lens = 37, [17, 37, 1, 30]                              # unsorted, with 1 frame and the full length
    _check_decode(m, _padded((4, 16, T), lens, dev), lens)
    n_wav = [8 * 37, 101, 8 * 20 + 3, 13]                      # not multiples of the ratio 8
    _check_encode(m, _padded((4, 1, 8 * 37), n_wav, dev, scale=0.3), n_wav)


def test_sampling_branch_with_noise(dev):
    m = _model(dict(BIGVGAN_H, causal=False), dev).set_precision(None)
    lens = [9, 37, 23]
    z = _padded((3, 32, 37), lens, dev)
    noise = _padded((3, 16, 37), lens, dev, pad=1e30)          # m + exp(logs) * noise is not 0 on padded rows
    _check_decode(m, z, lens, noise=noise, do_sample=True)


def test_bf16_inputs(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    lens = [37, 4, 20]
    _check_decode(m, _padded((3, 16, 37), lens, dev, torch.bfloat16), lens)
    n_wav = [250, 8 * 37, 19]
    _check_encode(m, _padded((3, 1, 8 * 37), n_wav, dev, torch.bfloat16, scale=0.3), n_wav)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_tensor_core_split_wide_config(dev, prec):
    """WIDE: ups.0 (256 -> 128) reads the frames, the 128-channel AMP blocks 4 x and the 64-channel ones 8 x as many
    rows, so clips of 80 / 40 / 12 / 5 frames fall on both sides of the 64-row threshold at every tensor-core layer."""
    m = _model(WIDE, dev).set_precision(prec)
    lens = [12, 80, 5, 40]
    _check_decode(m, _padded((4, 16, 80), lens, dev, pad=0.5), lens)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_tensor_core_split_bench_config(dev, prec):
    """The bench config: decoder clips of 70 / 30 / 7 / 1 frames (ups.0 at 1024 channels reads frames, the 512-channel
    blocks 8 x as many rows); encoder clips around the 64-row threshold of the 192 / 384 / 768-channel stages (their
    rows are 1 / 64, 1 / 256 and 1 / 1280 of the samples).  Three encoder clips are not whole frames of 1280 samples,
    so the strided convs of their own calls read inputs that are not whole stride groups."""
    m = _model(BENCH, dev, seed=1).set_precision(prec)
    lens = [30, 70, 1, 7]
    _check_decode(m, _padded((4, 512, 70), lens, dev, pad=0.5), lens)
    n_wav = [1280 * 3 + 17, 1280 * 78, 1280 * 16 + 641, 1280 * 4 + 1279]
    _check_encode(m, _padded((4, 1, 1280 * 78), n_wav, dev, pad=0.5, scale=0.3), n_wav)


def test_full_lengths_equal_the_plain_call(dev):
    m = _model(WIDE, dev).set_precision("bf16")
    z = torch.randn(3, 16, 90, device=dev)
    assert torch.equal(m.inference_from_latents(z, do_sample=False, valid_len=[90] * 3),
                       m.inference_from_latents(z, do_sample=False))
    m = _model(dict(BIGVGAN_H, causal=False), dev).set_precision(None)
    x = 0.3 * torch.randn(2, 1, 301, device=dev)
    assert torch.equal(m.extract_latents(x, valid_len=[301, 301]), m.extract_latents(x))


def test_bad_lengths_are_refused(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    z = torch.randn(2, 16, 20, device=dev)
    for bad in ([0, 20], [21, 20], [20], [20, 20, 20]):
        with pytest.raises(ValueError):
            m.inference_from_latents(z, do_sample=False, valid_len=bad)
    with pytest.raises(ValueError):                            # more clips than one ragged call takes
        m.inference_from_latents(torch.randn(65, 16, 4, device=dev), do_sample=False, valid_len=[4] * 65)
    with pytest.raises(ValueError):                            # 3 samples give 0 latent frames
        m.extract_latents(torch.randn(2, 1, 64, device=dev), valid_len=[64, 3])
    # the library refuses the same on its own
    L = _lib.lib()
    x = torch.randn(2, 4, 10, device=dev)
    bad = (ctypes.c_int * 2)(10, 11)
    with pytest.raises(_lib.KvaeError):
        _lib.check(L.kvae_zero_tail_cf(x.data_ptr(), 2, 4, 10, 10, bad, _lib.KVAE_F32, _lib.stream_ptr(dev)))
    act = m.resblocks[0].activations[0]
    with pytest.raises(_lib.KvaeError):
        act.ragged(torch.randn(2, act.act.alpha.numel(), 10, device=dev), [0, 10])


def test_zero_tail_pitched(dev):
    """kvae_zero_tail_cf on rows at a pitch wider than T: zeroes [valid_len[b], T) only."""
    y = torch.randn(3, 5, 300, device=dev)
    ref = y.clone()
    lens = [0, 129, 200]
    _lib.check(_lib.lib().kvae_zero_tail_cf(y.data_ptr(), 3, 5, 200, 300, (ctypes.c_int * 3)(*lens), _lib.KVAE_F32,
                                            _lib.stream_ptr(dev)))
    for b, n in enumerate(lens):
        ref[b, :, n:200] = 0
    assert torch.equal(y, ref)
    H.report("BigVGANFlowVAE ragged batches", "per-clip torch.equal")
