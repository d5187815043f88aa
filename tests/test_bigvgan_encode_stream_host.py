"""Host-side checks of the BigVGAN streaming encoder: the lookahead and left context that
``bigvgan_encode_stream_geometry`` derives from the layer definitions against the float64 oracle, the frame counts, and
the argument checks that need no GPU."""
import os
import sys

import pytest
import torch

import helpers  # noqa: F401  (sys.path)
import kalle_audio_b200 as k
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV
from oracle import bigvgan_oracle as BO

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


# bench.py's encoder geometry (16 kHz, rates 2/2/4/4/4/5, ratio 1280) with narrow channels: the reach depends on
# kernels, dilations and strides only, and the float64 oracle stays fast
BENCH_RATES = dict(BIGVGAN_H, downsample_channels=[12] + [4] * 6, downsample_rates=[2, 2, 4, 4, 4, 5], latent_dim=4)

# (tag, config, lookahead, context, probed frame t, clip length)
CASES = [("golden", dict(BIGVGAN_H), 702, 706, 120, 2400),
         ("bench_rates", BENCH_RATES, 113542, 114478, 100, 250000)]


def _nan_frames(h, n, poison):
    """Frames of the float64 oracle's extract_latents that a NaN at each sample in ``poison`` reaches."""
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(0)
        m = BV.BigVGANFlowVAE(AttrDict(h, causal=True))
        sd = {name: p.detach().double() for name, p in m.state_dict().items()}
        x = torch.randn(1, 1, n, generator=torch.Generator().manual_seed(1))
        x[..., poison] = float("nan")
        return torch.isnan(BO.extract_latents(sd, AttrDict(h, causal=True), x)).any(1)[0]
    finally:
        torch.set_default_dtype(prev)


@pytest.mark.parametrize("tag,h,la,ctx,t,n", CASES, ids=[c[0] for c in CASES])
def test_lookahead_and_context_are_the_exact_dependency(tag, h, la, ctx, t, n):
    """Frame t reads exactly the samples t * ratio - context .. t * ratio + ratio - 1 + lookahead: a NaN at either end
    reaches it, a NaN one sample further out does not."""
    g = k.bigvgan_encode_stream_geometry(h)
    assert (g["lookahead"], g["context"]) == (la, ctx)
    r = g["ratio"]
    last, first = t * r + r - 1 + la, t * r - ctx
    assert _nan_frames(h, n, [last])[t] and _nan_frames(h, n, [first])[t]
    assert not _nan_frames(h, n, [last + 1])[t] and not _nan_frames(h, n, [first - 1])[t]


@pytest.mark.parametrize("h", [dict(BIGVGAN_H), BENCH_RATES], ids=["golden", "bench_rates"])
def test_frame_counts(h):
    m = BV.BigVGANFlowVAE(AttrDict(h, causal=True))
    se = k.BigVGANStreamingEncoder(m)
    for n in [0, 1, 2, 7, 8, 9, 700, 703, 711, 1409, 5000, 113542 + 1280, 250001]:
        assert se.frames(n, True) == m.latent_length(n)
        assert se.frames(n) == max(0, (n - se.lookahead) // se.ratio)


def test_geometry_rows():
    g = k.bigvgan_encode_stream_geometry(BENCH_RATES)
    assert g["ratio"] == 1280 and len(g["ops"]) == 2 + 6 * 13
    strided = [r for r in g["ops"] if r["stride"] > 1]
    assert [(r["stride"], r["span"], r["padding"], r["rate"]) for r in strided] == \
        [(2, 3, 1, 1), (2, 3, 1, 2), (4, 7, 3, 4), (4, 7, 3, 16), (4, 7, 3, 64), (5, 9, 4, 256)]
    assert max(r["dilation"] for r in g["ops"]) == 32


def test_argument_checks_without_gpu():
    with pytest.raises(TypeError):
        k.BigVGANStreamingEncoder(torch.nn.Conv1d(1, 1, 1))
    m = BV.BigVGANFlowVAE(AttrDict(BIGVGAN_H, causal=True))
    se = k.BigVGANStreamingEncoder(m)
    assert (se.lookahead, se.context, se.ratio, se.max_samples, se.out_channels) == (702, 706, 8, 128, 32)
    with pytest.raises(ValueError):
        k.BigVGANStreamingEncoder(m, max_samples=0)
    with pytest.raises(k.KvaeError):
        se.push(torch.zeros(1, 1, 3))              # CPU audio
    with pytest.raises(ValueError):
        se.flush()                                 # nothing pushed


def test_stream_conv_refusals_without_gpu():
    """kvae_conv1d_stream_fwd refuses before any device access (the placeholder pointers are never dereferenced); its
    module method takes no transposed conv."""
    with pytest.raises(ValueError, match="transposed"):
        BV.ConvTranspose1d(64, 64, 8, 4).conv_window(None, None, None, 0, 0, 0, 4, -1)
    L = _lib.lib()
    ptr = 1 << 12

    def call(x0, nx, o0, o1, t_end):
        # Cin = Cout = 64, K = 8, stride 4, padding 3: output o reads input rows 4 o - 3 .. 4 o + 4
        return L.kvae_conv1d_stream_fwd(ptr, 256, x0, nx, ptr, 64, o0, o1, t_end, ptr, None, 1, 64, 64, 8, 4, 1, 3,
                                        _lib.KVAE_F32, 1, ptr, 1 << 24, None)

    assert call(6, 40, 5, 8, -1) != 0 and b"multiple of the stride" in L.kvae_last_error()
    assert call(20, 40, 5, 8, -1) != 0 and b"window" in L.kvae_last_error()     # output 5 reads row 17 < 20
    assert call(16, 12, 5, 8, -1) != 0 and b"window" in L.kvae_last_error()     # output 7 reads row 32 > 27
    assert call(0, 40, 0, 12, 40) != 0 and b"past the stream" in L.kvae_last_error()
