"""GPU checks of BigVGANStreamingEncoder: the concatenated stream equals ``extract_latents`` of the whole clip with
``torch.equal`` (frame count included), for clips that are not whole frames its ragged call too, and the stream-form
conv kvae_conv1d_stream_fwd equals the whole-layer rows on every engine."""
import os
import random
import sys

import pytest
import torch

import helpers as H
import kalle_audio_b200 as k
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


class AttrDict(dict):
    __getattr__ = dict.__getitem__


# a tensor-core encoder: the rate-4 strided conv (64 -> 128) and both ResStacks run on tcgen05
SMALL_TC = AttrDict(BIGVGAN_H, causal=True, downsample_channels=[12, 64, 128], downsample_rates=[2, 4], latent_dim=32)
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
    return BV.BigVGANFlowVAE(AttrDict(h)).eval().to(dev)


def _stream(se, x, sizes):
    outs, i = [], 0
    for n in sizes:
        outs.append(se.push(x[:, :, i:i + n]))
        i += n
    assert i == x.shape[2]
    outs.append(se.flush())
    return torch.cat(outs, dim=2), outs


def _ragged_sizes(n, seed):
    rng = random.Random(seed)
    sizes = [0, 1, 3, 0, 1]
    while sum(sizes) < n:
        sizes.append(rng.choice([0, 1, 2, 5, 17, 64, 129, 700, 1280]))
    sizes[-1] -= sum(sizes) - n
    return sizes


@pytest.mark.parametrize("B,L", [(1, 1000), (1, 3001), (3, 2403)])
def test_golden_config_ragged_pushes(dev, B, L):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    x = 0.3 * torch.randn(B, 1, L, device=dev)
    ref = m.extract_latents(x)
    assert ref.shape[2] == m.latent_length(L)
    got = {}
    for graphs in (False, True):
        se = k.BigVGANStreamingEncoder(m, max_samples=256, use_cuda_graphs=graphs)
        sizes = _ragged_sizes(L, L + graphs)
        y, outs = _stream(se, x, sizes)
        assert y.shape == ref.shape and torch.equal(y, ref), f"graphs={graphs}: max diff {(y - ref).abs().max()}"
        total = 0
        for j in range(len(sizes)):                 # frames emitted after n samples: frames(n)
            total += outs[j].shape[2]
            assert total == se.frames(sum(sizes[:j + 1]))
        got[graphs] = y
    assert torch.equal(got[False], got[True])


@pytest.mark.parametrize("prec", [None, "fp32", "bf16"])
def test_small_tensor_core_encoder(dev, prec):
    m = _model(SMALL_TC, dev).set_precision(prec)
    x = 0.3 * torch.randn(2, 1, 8 * 100, device=dev)     # whole frames, >= 64 rows at every layer
    ref = m.extract_latents(x)
    se = k.BigVGANStreamingEncoder(m, max_samples=200)
    y, _ = _stream(se, x, _ragged_sizes(800, 5))
    assert torch.equal(y, ref), f"max diff {(y - ref).abs().max()}"
    on_tc = [c for c, e in se._engine.items() if e is not None]
    if prec is None:
        assert not on_tc
    else:
        assert "audio_encoder.generator.5.layer" in on_tc and len(on_tc) >= 25
        assert not torch.equal(y, m.set_precision(None).extract_latents(x))


@pytest.mark.parametrize("prec", [None, "bf16"])
@pytest.mark.parametrize("L", [803, 1001])
def test_non_frame_lengths_equal_the_ragged_call(dev, prec, L):
    """A clip that is not whole frames: the stream equals the whole-clip call, whose strided tensor-core convs read
    inputs that are not whole stride groups, and the ragged call on the clip padded to whole frames."""
    m = _model(SMALL_TC, dev).set_precision(prec)
    x = 0.3 * torch.randn(1, 1, L, device=dev)
    xp = torch.nn.functional.pad(x, (0, -L % 8))
    ref = m.extract_latents(xp, valid_len=[L])[:, :, :m.latent_length(L)]
    y, _ = _stream(k.BigVGANStreamingEncoder(m), x, [L // 3, 0, L - L // 3])
    assert torch.equal(y, ref), f"max diff {(y - ref).abs().max()}"
    assert torch.equal(m.extract_latents(x), ref)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_bench_config_30s(dev, prec):
    m = _model(BENCH, dev).set_precision(prec)
    x = 0.3 * torch.randn(1, 1, 16000 * 30, device=dev)     # 375 whole frames
    ref = m.extract_latents(x)
    se = k.BigVGANStreamingEncoder(m)
    y, _ = _stream(se, x, [4 * 1280] * 93 + [16000 * 30 - 93 * 4 * 1280])
    assert y.shape == (1, 1024, 375) and torch.equal(y, ref), f"max diff {(y - ref).abs().max()}"
    assert se.graph_replays > 0


def test_bf16_audio(dev):
    m = _model(dict(BIGVGAN_H, causal=False), dev).set_precision(None)
    x = (0.3 * torch.randn(2, 1, 1203, device=dev)).bfloat16()
    ref = m.extract_latents(x)
    y, _ = _stream(k.BigVGANStreamingEncoder(m), x, [4, 1, 900, 298])
    assert y.dtype == torch.bfloat16 and torch.equal(y, ref)


def test_graph_replay_in_steady_state(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    x = 0.3 * torch.randn(1, 1, 64 * 60, device=dev)
    ref = m.extract_latents(x)
    se = k.BigVGANStreamingEncoder(m)
    y, _ = _stream(se, x, [64] * 60)
    assert torch.equal(y, ref)
    caps = se.graph_captures
    assert caps < 30 and se.graph_replays == 60 - caps
    # a second clip after flush reuses the graphs of the first one: every push replays
    y2, _ = _stream(se, x, [64] * 60)
    assert torch.equal(y2, ref) and se.graph_captures == caps and se.graph_replays == 120 - caps


def test_weight_change_and_errors(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    x = 0.3 * torch.randn(1, 1, 900, device=dev)
    se = k.BigVGANStreamingEncoder(m)
    se.push(x[:, :, :100])
    with pytest.raises(ValueError):
        se.push(torch.zeros(2, 1, 10, device=dev))        # batch size changed
    with pytest.raises(ValueError):
        se.push(x[:, :, 100:110].bfloat16())               # dtype changed
    m.audio_encoder.generator[0].layer.weight_g.mul_(1.5)
    with pytest.raises(RuntimeError, match="weights"):
        se.push(x[:, :, 100:200])
    se.reset()                                             # a new stream with the new weights
    y, _ = _stream(se, x, [100, 300, 500])
    assert torch.equal(y, m.extract_latents(x))


# (stride, K, dilation, padding, T): the encoder's k3 convs up to dilation 32 and its strided convs (K = 2 s), and the
# decoder's stride-1 convs: a causal layer (padding d (K - 1); the stream keeps its first T rows) and a non-causal one
STREAM_CONVS = {"k3d1": (1, 3, 1, 1, 200), "k3d32": (1, 3, 32, 32, 300), "s2": (2, 4, 1, 1, 301),
                "s4": (4, 8, 1, 3, 403), "s5": (5, 10, 1, 4, 502), "causal_k7d5": (1, 7, 5, 30, 250),
                "k11d5": (1, 11, 5, 25, 260)}


@pytest.mark.parametrize("engine", [0, 1, 2])
@pytest.mark.parametrize("geom", list(STREAM_CONVS))
def test_stream_conv_rows_equal_whole_layer(dev, engine, geom):
    """kvae_conv1d_stream_fwd on pitched windows at random origins (multiples of the stride, some below row 0), with
    and without a stream end (inside a partial stride group for most T), equals those rows of the whole-layer call
    kvae_conv1d_win_fwd on the same engine.  Window rows below 0 or past the stream end hold NaN: they must read as
    zero.  Window-relative addressing gives the same rows."""
    s, K, d, p, T = STREAM_CONVS[geom]
    Cin, Cout = 64, 128
    rng = random.Random(17 * engine + s)
    torch.manual_seed(engine)
    L = _lib.lib()
    w = torch.randn(Cout, Cin, K, device=dev) * 0.05
    bias = torch.randn(Cout, device=dev)
    x = torch.randn(2, Cin, T, device=dev)
    nb = L.kvae_conv1d_packed_bytes(Cin, Cout, K, engine)
    packed = torch.empty(nb, dtype=torch.uint8, device=dev)
    _lib.check(L.kvae_conv1d_pack(w.data_ptr(), 0, Cin, Cout, K, engine, packed.data_ptr(), nb, 0))
    # whole layer over the clip padded with zeros to whole stride groups (the tensor-core whole call needs them)
    Tp = -(-T // s) * s
    xp = torch.nn.functional.pad(x, (0, Tp - T)).contiguous()
    T_out = (T + 2 * p - d * (K - 1) - 1) // s + 1
    Tp_out = (Tp + 2 * p - d * (K - 1) - 1) // s + 1
    ref = torch.empty(2, Cout, Tp_out, device=dev)
    ns = L.kvae_conv1d_win_scratch_bytes(2, Cin, Tp, engine)
    sc = torch.empty(max(ns, 1), dtype=torch.uint8, device=dev)
    _lib.check(L.kvae_conv1d_win_fwd(xp.data_ptr(), Tp, ref.data_ptr(), Tp_out, packed.data_ptr(), bias.data_ptr(), 0,
                                     2, Cin, Cout, Tp, K, s, d, p, 0, Tp_out, _lib.KVAE_F32, engine, sc.data_ptr(), ns,
                                     0))
    ref = ref[:, :, :T_out]
    cases = [(0, T_out, True)]
    for _ in range(8):
        o0 = rng.randrange(0, T_out - 1)
        o1 = rng.randrange(o0 + 1, min(T_out, o0 + 150) + 1)
        cases.append((o0, o1, rng.random() < 0.5))
    for o0, o1, end in cases:
        lo = o0 * s - p                                      # rows the outputs read
        hi = (o1 - 1) * s - p + d * (K - 1) + 1
        if not end and hi > T:
            end = True
        x0 = (lo // s - rng.randrange(0, 3)) * s             # whole groups before the first row read, maybe < 0
        x1 = hi + rng.randrange(0, 7) if end else min(T, hi + rng.randrange(0, 7))
        nx = x1 - x0
        win = torch.full((2, Cin, nx + 5), float("nan"), device=dev)     # pitched, NaN outside the clip
        a, b = max(0, x0), min(T, x1)
        if b > a:
            win[:, :, a - x0:b - x0] = x[:, :, a:b]
        t_end = T if end else -1
        ybuf = torch.full((2, Cout, o1 - o0 + 3), float("nan"), device=dev)
        ns = L.kvae_conv1d_stream_scratch_bytes(2, Cin, nx, s, engine)
        sc = torch.empty(max(ns, 1), dtype=torch.uint8, device=dev)
        args = (packed.data_ptr(), bias.data_ptr(), 2, Cin, Cout, K, s, d, p, _lib.KVAE_F32, engine, sc.data_ptr(), ns,
                0)
        _lib.check(L.kvae_conv1d_stream_fwd(win.data_ptr(), nx + 5, x0, nx, ybuf.data_ptr(), o1 - o0 + 3, o0, o1,
                                            t_end, *args))
        torch.cuda.synchronize()
        assert torch.equal(ybuf[:, :, :o1 - o0], ref[:, :, o0:o1]), (o0, o1, x0, nx, end)
        assert torch.isnan(ybuf[:, :, o1 - o0:]).all()       # nothing written past the requested rows
        if lo >= x0 >= 0:                                    # no output reads below the window: window-relative rows
            q = x0 // s
            y2 = torch.full((2, Cout, o1 - o0), float("nan"), device=dev)
            _lib.check(L.kvae_conv1d_stream_fwd(win.data_ptr(), nx + 5, 0, nx, y2.data_ptr(), o1 - o0, o0 - q, o1 - q,
                                                t_end - x0 if end else -1, *args))
            torch.cuda.synchronize()
            assert torch.equal(y2, ref[:, :, o0:o1]), ("relative", o0, o1, x0)
    H.report(f"stream conv {geom} engine {engine}", "bit-exact")
