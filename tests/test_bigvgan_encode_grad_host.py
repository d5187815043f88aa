"""Host-side checks behind BigVGANFlowVAE.encode_with_grad, without a GPU:

  * the data-gradient geometry that kvae_conv1d_win_bwd runs for the encoder's strided convs (kvae_conv1d_dgrad_form):
    applied in float64 as F.conv_transpose1d of the output gradient with the layer's own weight, continued to the
    layer's T input rows (output_padding), it equals torch.autograd.grad of F.conv1d for every strided conv of the
    golden and bench encoders and every T mod s, the rows past the transposed conv's natural length included;
  * kvae_conv1d_win_bwd's argument checks with placeholder pointers (refused before any device access): a strided
    Conv1d is accepted and sized, a strided dilated conv and a T_gy out of range are refused, padding past d (K - 1)
    is accepted on the CUDA cores only, and the scratch size of the geometries accepted before (stride-1 convs,
    transposed convs) is unchanged."""
import ctypes
import os
import sys

import pytest
import torch
import torch.nn.functional as F

import helpers  # noqa: F401  (sys.path)
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402

BENCH_ENCODER = dict(BIGVGAN_H, downsample_channels=[12, 24, 48, 96, 192, 384, 768], downsample_rates=[2, 2, 4, 4, 4, 5])
CONFIGS = {"golden": BIGVGAN_H, "bench": BENCH_ENCODER}


@pytest.fixture(autouse=True)
def _grad_mode():
    """Other test modules turn grad mode off when they are imported; these tests need it on."""
    with torch.enable_grad():
        yield


def _form(transposed, Cin, Cout, K, s, d, p):
    out = (ctypes.c_int * 7)()
    _lib.check(_lib.lib().kvae_conv1d_dgrad_form(int(transposed), Cin, Cout, K, s, d, p, ctypes.byref(out)))
    return list(out)


def _encoder_convs(h):
    ops, _ = BV._encoder_program(h)
    return [op for op in ops if op.kind == "conv"]


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_strided_data_gradient_vs_autograd(tag):
    gen = torch.Generator().manual_seed(11)
    Cin, Cout = 3, 2
    strided = [op for op in _encoder_convs(CONFIGS[tag]) if op.geom.s > 1]
    assert len(strided) == len(CONFIGS[tag]["downsample_rates"])
    past_natural = 0
    for op in strided:
        K, s, p = op.geom.K, op.geom.s, op.geom.pl
        kind, cin, cout, s2, d2, p2, flip = _form(False, Cin, Cout, K, s, 1, p)
        assert (kind, cin, cout, s2, d2, p2, flip) == (1, Cout, Cin, s, 1, p, 0), op.module
        w = torch.randn(Cout, Cin, K, dtype=torch.float64, generator=gen)
        for T in range(K, K + 3 * s):                       # every T mod s, more than once
            x = torch.randn(2, Cin, T, dtype=torch.float64, generator=gen, requires_grad=True)
            y = F.conv1d(x, w, stride=s, padding=p)
            gy = torch.randn(y.shape, dtype=torch.float64, generator=gen)
            ref, = torch.autograd.grad(y, x, gy)
            natural = (y.shape[2] - 1) * s2 - 2 * p2 + K
            assert 0 <= T - natural < s2, (op.module, T)
            gx = F.conv_transpose1d(gy, w, stride=s2, padding=p2, output_padding=T - natural)
            assert gx.shape == ref.shape, (op.module, T)
            assert torch.allclose(gx, ref, rtol=1e-12, atol=1e-12), (op.module, T)
            if T > natural and ref[:, :, natural:].abs().max() > 0:
                past_natural += 1                            # rows past the natural length carry real gradient
    assert past_natural > 0


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_stride_one_form_is_the_conv_geometry(tag):
    """For every stride-1 encoder conv the new query restates kvae_conv1d_dgrad_geom (a Conv1d, kind 0)."""
    L = _lib.lib()
    for op in _encoder_convs(CONFIGS[tag]):
        if op.geom.s != 1:
            continue
        g = op.geom
        geom = (ctypes.c_int * 6)()
        _lib.check(L.kvae_conv1d_dgrad_geom(0, 64, 128, g.K, 1, g.d, g.pl, ctypes.byref(geom)))
        assert _form(False, 64, 128, g.K, 1, g.d, g.pl) == [0] + list(geom), op.module


def _align(n):
    return (n + 1023) // 1024 * 1024


def _expected_scratch(transposed, B, Cin, Cout, T, T_gy, K, s, engine):
    """kvae_conv1d_win_bwd's scratch layout: packed data-gradient weight, gy staged (in whole stride groups for a
    transposed layer), the weight gradient, x channels-last bf16 (engine 1; whole stride groups for a strided Conv1d),
    gx in whole stride groups (tcgen05, strided Conv1d with T not a multiple of s)."""
    L = _lib.lib()
    Tg = -(-T_gy // s) * s if transposed else T_gy
    Tx = T if transposed else -(-T // s) * s
    n = L.kvae_conv1d_packed_bytes(Cout, Cin, K, engine) + L.kvae_conv1d_win_scratch_bytes(B, Cout, Tg, engine)
    n += _align(Cin * Cout * K * 4)
    if engine == 1:
        n += _align(B * Tx * Cin * 2)
    if engine and Tx != T:
        n += _align(B * Cin * Tx * 4)
    return n


def test_win_bwd_arguments_without_gpu():
    L = _lib.lib()
    ptr = 1 << 12

    def call(transposed, Cin, Cout, T, T_gy, K, s, d, p, engine, scratch_bytes):
        return L.kvae_conv1d_win_bwd(ptr, ptr, T_gy, ptr, ptr, ptr, ptr, ptr, ptr, ptr, int(transposed), 2, Cin, Cout, T,
                                     K, s, d, p, _lib.KVAE_F32, engine, ptr, scratch_bytes, None)

    def size(transposed, Cin, Cout, T, T_gy, K, s, engine):
        return L.kvae_conv1d_win_bwd_scratch_bytes(int(transposed), 2, Cin, Cout, T, T_gy, K, s, engine)

    # the bench encoder's strided convs (192 -> 384, K 8, s 4, p 3; 384 -> 768, K 10, s 5, p 4) at every T mod s:
    # accepted (the call gets as far as the scratch check) and sized by the layout above
    for Cin, Cout, K, s, p in ((192, 384, 8, 4, 3), (384, 768, 10, 5, 4)):
        for T in range(400, 400 + s):
            T_gy = (T + 2 * p - K) // s + 1
            for engine in (0, 1, 2):
                n = size(False, Cin, Cout, T, T_gy, K, s, engine)
                assert n == _expected_scratch(False, 2, Cin, Cout, T, T_gy, K, s, engine), (Cin, T, engine)
                assert call(False, Cin, Cout, T, T_gy, K, s, 1, p, engine, n - 1) != 0
                assert b"scratch too small" in L.kvae_last_error(), (Cin, T, engine, L.kvae_last_error())
                # T_gy past the layer's output length, and no rows at all
                assert call(False, Cin, Cout, T, T_gy + 1, K, s, 1, p, engine, n) != 0
                assert b"T_gy" in L.kvae_last_error()
                assert call(False, Cin, Cout, T, 0, K, s, 1, p, engine, n) != 0
                assert b"T_gy" in L.kvae_last_error()
    # a strided dilated conv has no data-gradient geometry on any engine
    for engine in (0, 1, 2):
        assert call(False, 64, 64, 400, 100, 4, 4, 2, 3, engine, 1 << 30) != 0
        assert b"dilation" in L.kvae_last_error()
    # padding past d (K - 1) (a stride-1 Conv1d, a strided one, a ConvTranspose1d): the CUDA cores only
    for tr, K, s, d, p, T, T_gy in ((False, 3, 1, 2, 5, 400, 406), (False, 4, 2, 1, 4, 400, 203),
                                    (True, 4, 2, 1, 4, 100, 194)):
        for engine in (0, 1, 2):
            n = size(tr, 64, 64, T, T_gy, K, s, engine)
            assert call(tr, 64, 64, T, T_gy, K, s, d, p, engine, n - 1) != 0
            assert (b"scratch too small" if engine == 0 else b"padding") in L.kvae_last_error(), (tr, engine)
            assert call(tr, 64, 64, T, T_gy + 1, K, s, d, p, engine, n) != 0
            assert (b"T_gy" if engine == 0 else b"padding") in L.kvae_last_error(), (tr, engine)
    # the geometries accepted before keep their scratch size: stride-1 convs (one with a non-multiple-of-64 T) and the
    # decoder's transposed convs
    for tr, Cin, Cout, T, T_gy, K, s in ((False, 768, 768, 401, 401, 3, 1), (False, 64, 64, 1000, 1000, 7, 1),
                                         (True, 512, 256, 101, 505, 10, 5), (True, 128, 64, 77, 308, 8, 4)):
        for engine in (0, 1, 2):
            assert size(tr, Cin, Cout, T, T_gy, K, s, engine) == _expected_scratch(tr, 2, Cin, Cout, T, T_gy, K, s, engine)
