"""Host-side checks of the math behind BigVGANFlowVAE.decode_with_grad, in float64 on the CPU:

  * the data-gradient geometry that kvae_conv1d_win_bwd runs (kvae_conv1d_dgrad_geom): applied as a plain F.conv1d of
    the output gradient with the transposed / tap-reversed weight, the stated left padding and zeros past the end, it
    equals torch.autograd.grad of the layer for every conv and transposed conv of the golden and bench decoders,
    causal and not (the bench rates include K = 10 at rate 5, odd K - s), and for the paddings past d (K - 1) that the
    stand-alone layers accept (kvae_conv1d_dgrad_form);
  * the backward chain of the anti-aliased activation as aa_act_bwd_kernel computes it (adjoint of the decimation,
    replicate padding folded back, the Snake derivative, adjoint of the up-filter, folded again; the parameter terms)
    against autograd through oracle.bigvgan_oracle.aa_activation."""
import ctypes
import os
import sys

import pytest
import torch
import torch.nn.functional as F

import helpers  # noqa: F401  (sys.path)
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV
from oracle import bigvgan_oracle as BO

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


BENCH_GEOMETRY = dict(BIGVGAN_H, latent_dim=8, resblock_kernel_sizes=[3, 7, 11], resblock_dilation_sizes=[[1, 3, 5]] * 3,
                      upsample_rates=[8, 5, 4, 2, 2, 2], upsample_kernel_sizes=[16, 10, 8, 4, 4, 4],
                      upsample_initial_channel=64, resblock="1", activation="snakebeta", snake_logscale=True,
                      downsample_channels=[12] + [4] * 6, downsample_rates=[2, 2, 4, 4, 4, 5])
CONFIGS = {"golden": BIGVGAN_H, "bench_geometry": BENCH_GEOMETRY}


@pytest.fixture(autouse=True)
def _grad_mode():
    """Other test modules turn grad mode off when they are imported; these tests need it on."""
    with torch.enable_grad():
        yield


def _layer64(g, x, w):
    """The decoder's layer in float64, as oracle.bigvgan_oracle applies it (causal: truncated)."""
    if g.kind == "convT":
        y = F.conv_transpose1d(x, w, stride=g.s, padding=g.p)
        return y[:, :, :-g.s] if g.causal else y
    y = F.conv1d(x, w, padding=g.pl, dilation=g.d)
    return y[:, :, :x.shape[2]] if g.causal else y


def _dgrad_geom(transposed, Cin, Cout, K, s, d, p):
    out = (ctypes.c_int * 6)()
    _lib.check(_lib.lib().kvae_conv1d_dgrad_geom(int(transposed), Cin, Cout, K, s, d, p, ctypes.byref(out)))
    return list(out)


@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_data_gradient_geometry_vs_autograd(tag, causal):
    h = dict(CONFIGS[tag], causal=causal)
    m = BV.BigVGANFlowVAE(AttrDict(h))
    ops, _ = BV._program(h)
    gen = torch.Generator().manual_seed(3)
    Cin, Cout, seen = 3, 2, set()
    for op in ops:
        if op.kind not in ("conv", "convT"):
            continue
        mod, g = BV._module(m, op.module), op.geom
        key = (op.kind, g.K, g.d, g.s, g.causal, mod.padding[0])
        if key in seen:
            continue
        seen.add(key)
        cin, cout, s2, d2, pl2, fl = _dgrad_geom(mod.transposed, Cin, Cout, g.K, g.s, g.d, mod.padding[0])
        assert (cin, cout) == (Cout, Cin), op.module
        wshape = (Cin, Cout, g.K) if mod.transposed else (Cout, Cin, g.K)
        w = torch.randn(*wshape, dtype=torch.float64, generator=gen)
        for T in (1, 2, 5, 9, 16, 33):
            x = torch.randn(2, Cin, T, dtype=torch.float64, generator=gen, requires_grad=True)
            try:
                y = _layer64(g, x, w)
            except RuntimeError:
                continue                                   # input shorter than the layer accepts
            if y.shape[2] < 1:
                continue
            gy = torch.randn(y.shape, dtype=torch.float64, generator=gen)
            ref, = torch.autograd.grad(y, x, gy)
            # the stated form: W' = the weight transposed with its taps reversed (Conv1d) or as it is (transposed)
            W = w.transpose(0, 1).flip(-1) if fl else w
            right = max(0, (T - 1) * s2 - pl2 + d2 * (g.K - 1) + 1 - gy.shape[2])   # zeros past the end of gy
            gx = F.conv1d(F.pad(gy, (pl2, right)), W, stride=s2, dilation=d2)[:, :, :T]
            assert gx.shape == ref.shape, (op.module, T)
            assert torch.allclose(gx, ref, rtol=1e-12, atol=1e-12), (op.module, T)
    assert len(seen) >= (4 if tag == "golden" else 10)


@pytest.mark.parametrize("transposed,K,s,d,p", [(0, 3, 1, 1, 3), (0, 3, 1, 2, 7), (0, 4, 2, 1, 4), (0, 3, 3, 1, 5),
                                               (1, 4, 2, 1, 4), (1, 3, 1, 1, 3)])
def test_large_padding_data_gradient_vs_autograd(transposed, K, s, d, p):
    """Padding past d (K - 1), which the stand-alone WNConv1d / WNConvTranspose1d accept (CUDA cores only): a stride-1
    Conv1d's form reads gy ahead (negative left padding), a strided Conv1d's is the ConvTranspose1d continued over zero
    gy rows, a ConvTranspose1d's the strided Conv1d; each against torch.autograd.grad in float64."""
    Cin, Cout = 3, 2
    out = (ctypes.c_int * 7)()
    _lib.check(_lib.lib().kvae_conv1d_dgrad_form(transposed, Cin, Cout, K, s, d, p, ctypes.byref(out)))
    kind, cin, cout, s2, d2, p2, flip = out
    assert (cin, cout) == (Cout, Cin)
    if not kind:        # the stride-1 / transposed contract of kvae_conv1d_dgrad_geom
        assert [kind] + _dgrad_geom(transposed, Cin, Cout, K, s, d, p) == list(out)
    gen = torch.Generator().manual_seed(5)
    w = torch.randn(*((Cin, Cout, K) if transposed else (Cout, Cin, K)), dtype=torch.float64, generator=gen)
    checked = 0
    for T in range(1, 4 * K + 3 * s):
        x = torch.randn(2, Cin, T, dtype=torch.float64, generator=gen, requires_grad=True)
        T_out = (T - 1) * s - 2 * p + K if transposed else (T + 2 * p - d * (K - 1) - 1) // s + 1
        if T_out < 1:
            continue
        y = (F.conv_transpose1d(x, w, stride=s, padding=p) if transposed
             else F.conv1d(x, w, stride=s, padding=p, dilation=d))
        gy = torch.randn(y.shape, dtype=torch.float64, generator=gen)
        ref, = torch.autograd.grad(y, x, gy)
        if kind:        # ConvTranspose1d of gy with the weight as it is, over enough zero rows of gy past its end
            z = max(0, -(-(T + 2 * p2 - K) // s2) + 1 - T_out)
            gx = F.conv_transpose1d(F.pad(gy, (0, z)), w, stride=s2, padding=p2)[:, :, :T]
        else:           # Conv1d of gy, left padding p2 (< 0: the first -p2 rows are skipped), zeros past its end
            W = w.transpose(0, 1).flip(-1) if flip else w
            right = max(0, (T - 1) * s2 - p2 + d2 * (K - 1) + 1 - T_out)
            gx = F.conv1d(F.pad(gy, (p2, right)), W, stride=s2, dilation=d2)[:, :, :T]
        assert gx.shape == ref.shape, T
        assert torch.allclose(gx, ref, rtol=1e-12, atol=1e-12), T
        checked += 1
    assert checked >= 5
    if not transposed and s == 1:
        assert p2 < 0


def test_data_gradient_geometry_still_refused():
    """What kvae_conv1d_dgrad_geom still refuses: a strided Conv1d (its form is a ConvTranspose1d, through
    kvae_conv1d_dgrad_form) and a dilated transposed conv.  Padding past d (K - 1) is accepted (see above)."""
    L = _lib.lib()
    out = (ctypes.c_int * 6)()
    assert L.kvae_conv1d_dgrad_geom(0, 64, 64, 3, 2, 1, 1, ctypes.byref(out)) != 0          # strided Conv1d
    assert L.kvae_conv1d_dgrad_geom(1, 64, 64, 4, 2, 2, 1, ctypes.byref(out)) != 0          # dilated transposed conv
    assert L.kvae_conv1d_dgrad_geom(1, 64, 64, 10, 5, 1, 2, ctypes.byref(out)) == 0
    assert list(out) == [64, 64, 5, 1, 2, 0]


# ------------------------------------------------------------------------------------------------- activation chain
def _filters():
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)              # the filter design in float64, as the oracle's under it
    try:
        fu = BV._kaiser_sinc_filter1d(0.25, 0.3, 12).reshape(-1)
    finally:
        torch.set_default_dtype(prev)
    return fu, fu.clone()                                  # Activation1d: up and down filters of ratio 2, 12 taps


def aa_bwd_restated(x, gy, alpha, beta, logscale):
    """(gx, d alpha, d beta or None) of Activation1d in float64, the chain of aa_act_bwd_kernel written out."""
    B, C, T = x.shape
    fu, fd = _filters()
    U = torch.zeros(2 * T, T + 10, dtype=torch.float64)    # u[n] = 2 sum_i xp[i] fu[n + 15 - 2 i]
    for n in range(2 * T):
        for i in range(T + 10):
            k = n + 15 - 2 * i
            if 0 <= k < 12:
                U[n, i] = fu[k]
    D = torch.zeros(T, 2 * T + 10, dtype=torch.float64)    # y[t] = sum_m vp[2 t + m] fd[m]
    for t in range(T):
        D[t, 2 * t:2 * t + 12] = fd
    ix = (torch.arange(T + 10) - 5).clamp(0, T - 1)
    iv = (torch.arange(2 * T + 10) - 5).clamp(0, 2 * T - 1)
    a = alpha.view(1, -1, 1)
    b = a if beta is None else beta.view(1, -1, 1)
    if logscale:
        a, b = torch.exp(a), torch.exp(b)
    inv_b = 1.0 / (b + 1e-9)
    u = 2 * x[:, :, ix] @ U.t()
    gvp = gy @ D                                            # adjoint of the decimation
    gv = torch.zeros_like(u).index_add_(2, iv, gvp)         # replicate padding of v folded back
    s2 = torch.sin(2 * a * u)
    gu = gv * (1 + inv_b * a * s2)
    gxp = 2 * gu @ U                                        # adjoint of the up-filter
    gx = torch.zeros_like(x).index_add_(2, ix, gxp)         # clamped x indices folded back
    da = (gv * inv_b * u * s2).sum((0, 2))                  # dv/da
    db = (gv * -(torch.sin(a * u) ** 2) * inv_b ** 2).sum((0, 2))   # dv/db
    fa = a.view(-1) if logscale else 1.0
    fb = b.view(-1) if logscale else 1.0
    if beta is None:
        return gx, (da + db) * fa, None
    return gx, da * fa, db * fb


@pytest.mark.parametrize("T", [1, 4, 11, 40])
@pytest.mark.parametrize("snake", ["snake", "snakebeta"])
@pytest.mark.parametrize("logscale", [True, False], ids=["log", "lin"])
def test_activation_chain_vs_autograd(T, snake, logscale):
    gen = torch.Generator().manual_seed(T)
    B, C = 2, 3
    x = torch.randn(B, C, T, dtype=torch.float64, generator=gen, requires_grad=True)
    alpha = (0.3 * torch.randn(C, dtype=torch.float64, generator=gen) if logscale else
             1.0 + 0.3 * torch.rand(C, dtype=torch.float64, generator=gen)).requires_grad_(True)
    beta = None
    sd = {"a.act.alpha": alpha}
    if snake == "snakebeta":
        beta = (0.3 * torch.randn(C, dtype=torch.float64, generator=gen) if logscale else
                1.0 + 0.3 * torch.rand(C, dtype=torch.float64, generator=gen)).requires_grad_(True)
        sd["a.act.beta"] = beta
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)              # the alias-free filters follow the default dtype
    try:
        y = BO.aa_activation(sd, "a", x, logscale)
    finally:
        torch.set_default_dtype(prev)
    gy = torch.randn(y.shape, dtype=torch.float64, generator=gen)
    refs = torch.autograd.grad(y, [x, alpha] + ([beta] if beta is not None else []), gy)
    gx, da, db = aa_bwd_restated(x.detach(), gy, alpha.detach(), None if beta is None else beta.detach(), logscale)
    assert torch.allclose(gx, refs[0], rtol=1e-10, atol=1e-12)
    assert torch.allclose(da, refs[1], rtol=1e-10, atol=1e-12)
    if beta is not None:
        assert torch.allclose(db, refs[2], rtol=1e-10, atol=1e-12)
