"""GPU checks of BigVGANStreamingDecoder: the concatenated stream equals ``inference_from_latents`` of the whole
utterance with ``torch.equal`` (output length included), and the window-form activation kernel equals the whole-row
one on every window the stream hands it."""
import os
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
    for n, p in m.named_parameters():               # snake parameters away from their init: a less symmetric test
        if n.endswith(("alpha", "beta")):
            p.data = 0.2 * torch.randn_like(p) if m.h.snake_logscale else 1.0 + 0.3 * torch.rand_like(p)
    return m.to(dev)


def _stream(sd, z, sizes, noise=None):
    outs, i = [], 0
    for n in sizes:
        outs.append(sd.push(z[:, :, i:i + n], None if noise is None else noise[:, :, i:i + n]))
        i += n
    assert i == z.shape[2]
    outs.append(sd.flush())
    return torch.cat(outs, dim=2), outs


RAGGED = [0, 1, 3, 0, 1, 20, 2, 7, 1, 5]            # 0- and 1-frame pushes, one longer than max_frames=16


@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
@pytest.mark.parametrize("B", [1, 2])
def test_golden_config_ragged_pushes(dev, causal, B):
    m = _model(dict(BIGVGAN_H, causal=causal), dev).set_precision(None)
    z = torch.randn(B, 16, sum(RAGGED), device=dev)
    ref = m.inference_from_latents(z, do_sample=False)
    got = {}
    for graphs in (False, True):
        sd = k.BigVGANStreamingDecoder(m, max_frames=16, use_cuda_graphs=graphs)
        y, outs = _stream(sd, z, RAGGED)
        assert y.shape == ref.shape and torch.equal(y, ref), f"graphs={graphs}: max diff {(y - ref).abs().max()}"
        got[graphs] = y
        total = 0
        for j in range(len(RAGGED)):                # emitted = max(0, n * ratio - lookahead) after n frames
            total += outs[j].shape[2]
            pushed = sum(RAGGED[:j + 1])
            assert total == max(0, pushed * sd.ratio - sd.lookahead)
    assert torch.equal(got[False], got[True])


def test_graph_replay_in_steady_state(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    z = torch.randn(1, 16, 60, device=dev)
    ref = m.inference_from_latents(z, do_sample=False)
    sd = k.BigVGANStreamingDecoder(m, use_cuda_graphs=True)
    y, _ = _stream(sd, z, [2] * 30)
    assert torch.equal(y, ref)
    assert sd.graph_replays >= 15 and sd.graph_captures <= 15
    # a second utterance after flush reuses the graphs of the first one
    caps = sd.graph_captures
    y2, _ = _stream(sd, z, [2] * 30)
    assert torch.equal(y2, ref) and sd.graph_captures == caps


@pytest.mark.parametrize("prec", [None, "fp32", "bf16"])
def test_wide_config_tensor_cores(dev, prec):
    m = _model(WIDE, dev).set_precision(prec)
    z = torch.randn(1, 16, 70, device=dev)          # >= 64 frames: the whole decode puts every eligible layer on tcgen05
    ref = m.inference_from_latents(z, do_sample=False)
    sd = k.BigVGANStreamingDecoder(m, max_frames=8)
    y, _ = _stream(sd, z, [1, 4, 4, 3, 9, 4] + [5] * 9)
    assert torch.equal(y, ref), f"max diff {(y - ref).abs().max()}"
    on_tc = [c for c, e in sd._engine.items() if e is not None]
    if prec is None:
        assert not on_tc
    else:
        assert "ups.0.0" in on_tc and len(on_tc) >= 20
        assert not torch.equal(y, m.set_precision(None).inference_from_latents(z, do_sample=False))


@pytest.mark.parametrize("hop", [1, 4])
def test_bench_config_bf16(dev, hop):
    m = _model(BENCH, dev).set_precision("bf16")
    z = torch.randn(1, 512, 80, device=dev)
    ref = m.inference_from_latents(z, do_sample=False)
    sd = k.BigVGANStreamingDecoder(m, max_frames=16)
    y, _ = _stream(sd, z, [hop] * (80 // hop))
    assert torch.equal(y, ref), f"max diff {(y - ref).abs().max()}"
    assert sd.graph_replays > 0


def test_sampling_branch_with_noise(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    z = torch.randn(2, 32, 25, device=dev)
    nz = torch.randn(2, 16, 25, device=dev)
    ref = m.inference_from_latents(z, do_sample=True, noise=nz)
    sd = k.BigVGANStreamingDecoder(m, do_sample=True)
    y, _ = _stream(sd, z, [3, 0, 5, 1, 16], noise=nz)
    assert torch.equal(y, ref)
    with pytest.raises(ValueError):
        sd.push(z[:, :16, :2])                       # do_sample wants mean | log-scale


def test_bf16_latents(dev):
    m = _model(dict(BIGVGAN_H, causal=False), dev).set_precision(None)
    z = torch.randn(1, 16, 30, device=dev).bfloat16()
    ref = m.inference_from_latents(z, do_sample=False)
    y, _ = _stream(k.BigVGANStreamingDecoder(m), z, [4, 1, 9, 16])
    assert y.dtype == torch.bfloat16 and torch.equal(y, ref)


def test_interleaved_streams_and_errors(dev):
    m = _model(dict(BIGVGAN_H, causal=True), dev).set_precision(None)
    za, zb = torch.randn(1, 16, 24, device=dev), torch.randn(2, 16, 24, device=dev)
    ra, rb = m.inference_from_latents(za, do_sample=False), m.inference_from_latents(zb, do_sample=False)
    sa, sb = k.BigVGANStreamingDecoder(m), k.BigVGANStreamingDecoder(m)
    oa, ob = [], []
    for i in range(0, 24, 3):
        oa.append(sa.push(za[:, :, i:i + 3]))
        ob.append(sb.push(zb[:, :, i:i + 3]))
    oa.append(sa.flush())
    ob.append(sb.flush())
    assert torch.equal(torch.cat(oa, 2), ra) and torch.equal(torch.cat(ob, 2), rb)
    # batch size change, CPU input, weight update inside a stream
    sa.push(za[:, :, :4])
    with pytest.raises(ValueError):
        sa.push(zb[:, :, 4:8])
    with pytest.raises(k.KvaeError):
        sa.push(za[:, :, 4:8].cpu())
    m.conv_post.weight_g.mul_(1.5)
    with pytest.raises(RuntimeError, match="weights"):
        sa.push(za[:, :, 4:8])
    sa.reset()                                      # a new stream with the new weights
    y, _ = _stream(sa, za, [5, 5, 5, 9])
    assert torch.equal(y, m.inference_from_latents(za, do_sample=False))


@pytest.mark.parametrize("T", [3, 11, 40, 1500])
def test_window_activation_kernel(dev, T):
    """kvae_aa_act_win_fwd on windows with and without the start / end edge, including windows shorter than the
    filters, equals the whole-row kernel (Activation1d) on the same rows."""
    torch.manual_seed(T)
    act = BV.Activation1d(BV.SnakeBeta(6, alpha_logscale=True))
    act.act.alpha.data = 0.3 * torch.randn(6)
    act.act.beta.data = 0.3 * torch.randn(6)
    act = act.to(dev)
    x = torch.randn(2, 6, T, device=dev)
    ref = act(x)
    L = _lib.lib()
    fu = act.upsample.filter.reshape(-1).contiguous()
    fd = act.downsample.lowpass.filter.reshape(-1).contiguous()
    ranges = {(0, T), (0, 1), (T - 1, T), (min(5, T - 1), T), (0, max(1, T - 5)), (T // 3, max(T // 3 + 1, 2 * T // 3))}
    for o0, o1 in sorted(ranges):
        end = o1 == T
        x0 = max(0, o0 - 5)
        x1 = T if end else min(T, o1 + 5)
        if not end and o1 + 5 > T:
            continue
        win = torch.zeros(2, 6, x1 - x0 + 7, device=dev)          # pitched: wider than the rows it holds
        win[:, :, :x1 - x0] = x[:, :, x0:x1]
        y = torch.full((2, 6, o1 - o0), float("nan"), device=dev)
        _lib.check(L.kvae_aa_act_win_fwd(win.data_ptr(), win.shape[2], x0, x1 - x0, y.data_ptr(), o1 - o0, o0, o1,
                                         T if end else -1, act.act.alpha.data_ptr(), act.act.beta.data_ptr(), 1,
                                         fu.data_ptr(), fd.data_ptr(), 2, 6, _lib.KVAE_F32, _lib.stream_ptr(dev)))
        assert torch.equal(y, ref[:, :, o0:o1]), (o0, o1)
    # a window missing rows the outputs read is refused
    if T >= 40:
        assert L.kvae_aa_act_win_fwd(x.data_ptr(), T, 10, 20, x.data_ptr(), T, 10, 25, -1, act.act.alpha.data_ptr(),
                                     None, 1, fu.data_ptr(), fd.data_ptr(), 2, 6, _lib.KVAE_F32, 0) != 0
    H.report(f"window activation T={T}", "bit-exact")


# (transposed, stride, K, dilation, padding, T, output rows [o0, o1); None = the whole natural range)
WINDOW_CONVS = {
    "conv": (False, 1, 7, 3, 2, 90, (5, 61)),          # stride-1 conv: rows away from both ends
    "convT": (True, 4, 8, 1, 2, 90, (12, 68)),         # transposed conv: whole stride groups
    "strided": (False, 4, 8, 1, 2, 88, None),          # strided conv: full range only, whole stride groups of input
    "causal": (False, 1, 7, 3, 18, 90, (0, 90)),       # causal conv: the first T rows of the symmetric layer
    "causalT": (True, 4, 8, 1, 0, 90, (0, 360)),       # causal transposed conv: the last `stride` rows dropped
}


@pytest.mark.parametrize("engine", [0, 1, 2])
@pytest.mark.parametrize("geom", list(WINDOW_CONVS))
def test_window_conv_rows_equal_whole_layer(dev, engine, geom):
    """kvae_conv1d_win_fwd with weights from kvae_conv1d_pack: output rows [o0, o1) of a pitched window, written to a
    pitched output, equal those rows of the whole-layer call on the same engine (engine 0: kvae_conv1d_fwd; tcgen05:
    the full range of a contiguous input).  The causal cases are the truncated whole-layer calls of BigVGANFlowVAE."""
    torch.manual_seed(engine)
    transposed, s, K, d, p, T, rows = WINDOW_CONVS[geom]
    Cin, Cout = 128, 64
    T_nat = (T - 1) * s - 2 * p + d * (K - 1) + 1 if transposed else (T + 2 * p - d * (K - 1) - 1) // s + 1
    w = torch.randn((Cin, Cout, K) if transposed else (Cout, Cin, K), device=dev) * 0.05
    bias = torch.randn(Cout, device=dev)
    xbuf = torch.randn(2, Cin, T + 9, device=dev)
    x = xbuf[:, :, :T]                                   # pitched: 9 spare rows per channel
    L = _lib.lib()
    nb = L.kvae_conv1d_packed_bytes(Cin, Cout, K, engine)
    packed = torch.empty(nb, dtype=torch.uint8, device=dev)
    _lib.check(L.kvae_conv1d_pack(w.data_ptr(), int(transposed), Cin, Cout, K, engine, packed.data_ptr(), nb, 0))
    ref = torch.empty(2, Cout, T_nat, device=dev)
    if engine == 0:
        ns = L.kvae_conv1d_scratch_bytes(Cin, Cout, K)
        sc = torch.empty(ns, dtype=torch.uint8, device=dev)
        _lib.check(L.kvae_conv1d_fwd(x.contiguous().data_ptr(), ref.data_ptr(), w.data_ptr(), bias.data_ptr(),
                                     int(transposed), 2, Cin, Cout, T, K, s, d, p, _lib.KVAE_F32, sc.data_ptr(), ns, 0))
    else:
        ns = L.kvae_conv1d_win_scratch_bytes(2, Cin, T, engine)
        sc = torch.empty(ns, dtype=torch.uint8, device=dev)
        _lib.check(L.kvae_conv1d_win_fwd(x.contiguous().data_ptr(), T, ref.data_ptr(), T_nat, packed.data_ptr(),
                                         bias.data_ptr(), int(transposed), 2, Cin, Cout, T, K, s, d, p, 0, T_nat,
                                         _lib.KVAE_F32, engine, sc.data_ptr(), ns, 0))
    o0, o1 = rows or (0, T_nat)
    ybuf = torch.full((2, Cout, o1 - o0 + 3), float("nan"), device=dev)
    ns = L.kvae_conv1d_win_scratch_bytes(2, Cin, T, engine)
    sc = torch.empty(max(ns, 1), dtype=torch.uint8, device=dev)
    _lib.check(L.kvae_conv1d_win_fwd(x.data_ptr(), T + 9, ybuf.data_ptr(), o1 - o0 + 3, packed.data_ptr(),
                                     bias.data_ptr(), int(transposed), 2, Cin, Cout, T, K, s, d, p, o0, o1,
                                     _lib.KVAE_F32, engine, sc.data_ptr(), ns, 0))
    torch.cuda.synchronize()
    assert torch.equal(ybuf[:, :, :o1 - o0], ref[:, :, o0:o1])
    assert torch.isnan(ybuf[:, :, o1 - o0:]).all()      # nothing written past the requested rows
