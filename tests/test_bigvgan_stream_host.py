"""Host-side checks of the BigVGAN streaming decoder: the lookahead that ``bigvgan_stream_geometry`` derives from the
layer definitions against the CPU oracle, and the argument checks that need no GPU."""
import os
import sys

import pytest
import torch

import helpers  # noqa: F401  (sys.path)
import kalle_audio_b200 as k
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.bigvgan_stream import bigvgan_stream_geometry
from oracle import bigvgan_oracle as BO

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


# bench.py's measure_bigvgan geometry (rates 8/5/4/2/2/2, AMPBlock1 k 3/7/11, causal) with few channels: the lookahead
# depends on kernels, dilations and strides only, and the float64 oracle stays fast
BENCH_GEOMETRY = dict(BIGVGAN_H, causal=True, latent_dim=8, resblock_kernel_sizes=[3, 7, 11],
                      resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
                      upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=64, resblock="1",
                      activation="snakebeta", snake_logscale=True)

CASES = [("golden_causal", dict(BIGVGAN_H, causal=True), 40, 30, 119),
         ("golden_noncausal", dict(BIGVGAN_H, causal=False), 40, 30, 235),
         ("bench_geometry", BENCH_GEOMETRY, 24, 14, 10055)]


def _probe(h, T, f, poison):
    """First output sample that a change of latent frame f reaches (float64 oracle)."""
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)            # the oracle's anti-aliasing filters follow the default dtype
    try:
        torch.manual_seed(0)
        m = BV.BigVGANFlowVAE(AttrDict(h))
        sd = {n: p.detach().double() for n, p in m.state_dict().items()}
        z = torch.randn(1, h["latent_dim"], T, generator=torch.Generator().manual_seed(1))
        z2 = z.clone()
        if poison:
            z2[..., f] = float("nan")
            changed = torch.isnan(BO.inference_from_latents(sd, h, z2))
        else:
            z2[..., f] += 1.0
            changed = BO.inference_from_latents(sd, h, z) != BO.inference_from_latents(sd, h, z2)
    finally:
        torch.set_default_dtype(prev)
    return int(changed.flatten().nonzero().min())


@pytest.mark.parametrize("tag,h,T,f,expect", CASES, ids=[c[0] for c in CASES])
def test_lookahead_is_the_exact_dependency(tag, h, T, f, expect):
    """A NaN in frame f reaches every sample that reads it, however small the path's weights: the first NaN sample is
    exactly f * ratio - lookahead, so the bound is tight."""
    g = bigvgan_stream_geometry(h)
    assert g["lookahead"] == expect
    assert _probe(h, T, f, poison=True) == f * g["ratio"] - g["lookahead"]


@pytest.mark.parametrize("tag,h,T,f,expect", CASES, ids=[c[0] for c in CASES])
def test_finite_perturbation_stays_inside_the_lookahead(tag, h, T, f, expect):
    """A finite change of frame f never changes a sample before f * ratio - lookahead.  It usually starts later: the
    contributions through the outer taps of many Kaiser-sinc filters in series round away even in float64, which is
    why such a probe reads a smaller lookahead than the one a bit-exact stream has to wait for."""
    g = bigvgan_stream_geometry(h)
    assert _probe(h, T, f, poison=False) >= f * g["ratio"] - g["lookahead"]


def test_geometry_rows():
    g = bigvgan_stream_geometry(BENCH_GEOMETRY)
    assert g["ratio"] == 1280
    ops = {r["module"]: r for r in g["ops"]}
    assert ops["conv_pre"] == dict(op="conv", module="conv_pre", rate=1, rows_read=7, span=6, dilation=1, stride=1,
                                   lookahead=3)
    assert ops["ups.0.0"]["rows_read"] == 2 and ops["ups.0.0"]["rate"] == 1 and ops["ups.0.0"]["lookahead"] == 0
    assert ops["resblocks.2.convs1.2"] == dict(op="conv", module="resblocks.2.convs1.2", rate=8, rows_read=51, span=50,
                                               dilation=5, stride=1, lookahead=0)
    assert ops["activation_post"]["rate"] == 1280 and ops["activation_post"]["rows_read"] == 11
    assert sum(r["op"] == "act" for r in g["ops"]) == 6 * 3 * 6 + 1


def test_argument_checks_without_gpu():
    with pytest.raises(TypeError):
        k.BigVGANStreamingDecoder(torch.nn.Conv1d(1, 1, 1))
    m = BV.BigVGANFlowVAE(AttrDict(BIGVGAN_H, causal=True))
    sd = k.BigVGANStreamingDecoder(m)
    assert sd.lookahead == 119 and sd.ratio == 8
    with pytest.raises(k.KvaeError):
        sd.push(torch.zeros(1, 16, 3))
    with pytest.raises(ValueError):
        k.BigVGANStreamingDecoder(m, max_frames=0)
