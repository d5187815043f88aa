"""Drop-in for the inference path of the reference's 12.5 Hz VAE, ``BigVGANFlowVAE`` (/root/reference/backup/flows.py).

Module tree, constructor argument (the hyper-parameter object ``h``) and ``state_dict`` keys mirror the reference:
``audio_encoder`` (Encoder :191-241: Conv1d_S / LeakyReLU / ResStack), ``flow`` (VITS's ResidualCouplingBlock
:613-792, the training objective's flow: ``flow(z, x_mask, reverse=False)`` under autograd), ``conv_pre``, ``ups``,
``resblocks`` (AMPBlock1 / AMPBlock2 :243-330 with their anti-aliased ``Activation1d``), ``activation_post``,
``conv_post``.  Implemented:

    extract_latents(x)                      :494-496   waveform [B, 1, L] -> [B, 2 D, L / prod(downsample_rates)]
    inference_from_latents(x, do_sample)    :498-529   latents -> waveform [B, 1, T * prod(upsample_rates)]
    decode_with_grad(x, do_sample)          :498-529   the same under autograd (gradients to the latents and the
                                                       decoder's parameters)
    encode_with_grad(x)                     :494-496   extract_latents under autograd (gradients to the audio and the
                                                       encoder's parameters)

The first two take ``valid_len`` for a batch of clips of different lengths, each clip bit-identical to its own call (the
ragged path below ``_run_ragged``; ``latent_length`` / ``wav_length`` give the per-clip output lengths).

Every step runs through libkvae: convolutions and transposed convolutions (causal or not; weight norm folded on the
device) through the layer-level conv -- on the tensor cores for the layers whose channel counts are multiples of 64
(``set_precision``), ``kvae_conv1d_pack`` + ``kvae_conv1d_win_fwd`` over the rows the layer keeps, otherwise the fp32
CUDA-core ``kvae_conv1d_fwd`` -- the anti-aliased Snake / SnakeBeta activation as ONE fused kernel (``kvae_aa_act_fwd``:
x2 Kaiser-sinc upsampling, activation, low-pass + x2 decimation -- six eager kernels and four double-rate intermediates
in the reference), LeakyReLU / tanh / residual adds / the AMP average / the Gaussian sample as small elementwise
kernels.  Under grad mode each of them has an autograd node whose backward is a libkvae call too (``decode_with_grad``,
``encode_with_grad``): the ``_*Fn`` classes below, and for the convs the node every ``layers`` conv uses, whose backward
is ``kvae_conv1d_win_bwd`` on the engine the forward ran on.  The causal layers set ``keep``, the output rows they keep.
The flow's steps between its convs are the flow.cuh kernels (see "the flow" below).  ``forward`` (the reference's
training pass, whose return contract is not recorded here) is not built.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import torch
from torch import nn

from . import _lib
from .layers import TC_MIN_ROWS, WNConv1d, WNConvTranspose1d, _WNConvBase

_RAGGED_MAX_CLIPS = 64       # kRaggedMaxClips (elementwise.cuh): lengths travel by value into the kernels


def _kaiser_sinc_filter1d(cutoff: float, half_width: float, kernel_size: int) -> torch.Tensor:
    """Filter design of alias_free_torch (filter.py): Kaiser window x sinc, normalised to unit sum.  Load-time only."""
    half_size = kernel_size // 2
    delta_f = 4 * half_width
    A = 2.285 * (half_size - 1) * math.pi * delta_f + 7.95
    beta = 0.1102 * (A - 8.7) if A > 50.0 else (0.5842 * (A - 21) ** 0.4 + 0.07886 * (A - 21.0) if A >= 21.0 else 0.0)
    window = torch.kaiser_window(kernel_size, beta=beta, periodic=False)
    time = (torch.arange(-half_size, half_size) + 0.5) if kernel_size % 2 == 0 else torch.arange(kernel_size) - half_size
    arg = 2 * cutoff * time
    sinc = torch.where(arg == 0, torch.ones_like(arg), torch.sin(math.pi * arg) / math.pi / arg)
    f = 2 * cutoff * window * sinc
    return (f / f.sum()).view(1, 1, kernel_size)


# ------------------------------------------------------------------------------------------------- kernel wrappers
def _k(t: torch.Tensor) -> torch.Tensor:
    t = t if t.dtype in (torch.float32, torch.bfloat16) else t.float()
    return t.contiguous()


def _grad_on(*ts) -> bool:
    """Whether a step under the current grad mode gets an autograd node: some input or parameter requires grad."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)


def _unary(x: torch.Tensor, op: int, param: float = 0.0) -> torch.Tensor:
    _lib.require_cuda(x, "bigvgan")
    if torch.is_grad_enabled() and _grad_on(x):
        return _UnaryFn.apply(x, op, param)
    xin = _k(x)
    y = torch.empty_like(xin)
    _lib.check(_lib.lib().kvae_unary_fwd(xin.data_ptr(), y.data_ptr(), xin.numel(), op, float(param),
                                         _lib.dtype_code(xin.dtype), _lib.stream_ptr(x.device)))
    return y if y.dtype == x.dtype else y.to(x.dtype)


def _axpby(a: torch.Tensor, b: torch.Tensor, alpha: float, beta: float) -> torch.Tensor:
    if torch.is_grad_enabled() and _grad_on(a, b):
        return _AxpbyFn.apply(a, b, alpha, beta)
    ain, bin_ = _k(a), _k(b).to(_k(a).dtype)
    out = torch.empty_like(ain)
    _lib.check(_lib.lib().kvae_axpby(ain.data_ptr(), bin_.data_ptr(), out.data_ptr(), ain.numel(), alpha, beta,
                                     _lib.dtype_code(ain.dtype), _lib.stream_ptr(a.device)))
    return out if out.dtype == a.dtype else out.to(a.dtype)


def _gauss_sample(mean: torch.Tensor, logs: torch.Tensor, noise: torch.Tensor) -> torch.Tensor:
    """mean + noise * exp(logs) (flows.py:500-501), in the dtype of ``mean``."""
    if _grad_on(mean, logs):
        raise RuntimeError("_gauss_sample: differentiate through _GaussSampleFn on the whole latents (decode_with_grad)")
    m = _k(mean)
    lg, nz = _k(logs).to(m.dtype), _k(noise).to(m.dtype)
    z = torch.empty_like(m)
    if m.numel():
        _lib.check(_lib.lib().kvae_gauss_sample(m.data_ptr(), lg.data_ptr(), nz.data_ptr(), z.data_ptr(), m.numel(),
                                                _lib.dtype_code(m.dtype), _lib.stream_ptr(m.device)))
    return z if z.dtype == mean.dtype else z.to(mean.dtype)


# ------------------------------------------------------------------------------------------------- autograd nodes
# The backward of every step is a libkvae call (decode_with_grad; the flows.py interfaces each differentiates are cited
# in include/kvae.h).  Forward values are those of the no-grad calls: the same kernels on the same engines.
class _UnaryFn(torch.autograd.Function):
    """LeakyReLU (op 0) / tanh (op 1): kvae_unary_fwd / kvae_unary_bwd (tanh's backward reads the output)."""

    @staticmethod
    def forward(ctx, x, op, param):
        y = _unary(x, op, param)
        ctx.op, ctx.param, ctx.x_dtype = op, param, x.dtype
        ctx.save_for_backward(_k(x) if op == 0 else _k(y))
        return y

    @staticmethod
    def backward(ctx, gy):
        t, = ctx.saved_tensors
        g = gy.detach().to(t.dtype).contiguous()
        gx = torch.empty_like(t)
        _lib.check(_lib.lib().kvae_unary_bwd(t.data_ptr(), g.data_ptr(), gx.data_ptr(), t.numel(), ctx.op, float(ctx.param),
                                             _lib.dtype_code(t.dtype), _lib.stream_ptr(t.device)))
        return gx.to(ctx.x_dtype), None, None


class _AxpbyFn(torch.autograd.Function):
    """out = alpha a + beta b: ga = alpha g and gb = beta g through kvae_axpby itself (g as is for a coefficient 1,
    nothing for 0)."""

    @staticmethod
    def forward(ctx, a, b, alpha, beta):
        ctx.coef, ctx.dtypes = (alpha, beta), (a.dtype, b.dtype)
        return _axpby(a, b, alpha, beta)

    @staticmethod
    def backward(ctx, gout):
        g = _k(gout.detach())
        out = []
        for c, dt, need in zip(ctx.coef, ctx.dtypes, ctx.needs_input_grad[:2]):
            if not need or c == 0.0:
                out.append(None)
            elif c == 1.0:
                out.append(g.to(dt))
            else:
                r = torch.empty_like(g)
                _lib.check(_lib.lib().kvae_axpby(g.data_ptr(), g.data_ptr(), r.data_ptr(), g.numel(), c, 0.0,
                                                 _lib.dtype_code(g.dtype), _lib.stream_ptr(g.device)))
                out.append(r.to(dt))
        return out[0], out[1], None, None


class _GaussSampleFn(torch.autograd.Function):
    """z = mean + noise exp(logs) on the latents x = [B, 2 D, T] (mean | logs): kvae_gauss_sample /
    kvae_gauss_sample_bwd (gmean = gz, glogs = gz noise exp(logs))."""

    @staticmethod
    def forward(ctx, x, noise, D):
        m_q, logs_q = torch.split(x, D, dim=1)
        z = _gauss_sample(m_q, logs_q, noise)
        xin = _k(x)
        ctx.save_for_backward(xin, _k(noise).to(xin.dtype))
        ctx.x_dtype = x.dtype
        return z

    @staticmethod
    def backward(ctx, gz):
        xin, nz = ctx.saved_tensors
        B, D2, T = xin.shape
        g = gz.detach().to(xin.dtype).contiguous()
        gx = torch.empty_like(xin)
        _lib.check(_lib.lib().kvae_gauss_sample_bwd(xin.data_ptr(), nz.data_ptr(), g.data_ptr(), gx.data_ptr(), B, D2 // 2,
                                                    T, _lib.dtype_code(xin.dtype), _lib.stream_ptr(xin.device)))
        return gx.to(ctx.x_dtype), None, None


class _AaActFn(torch.autograd.Function):
    """Activation1d: kvae_aa_act_fwd / kvae_aa_act_bwd (x saved; the double-rate signal is rebuilt in the backward)."""

    @staticmethod
    def forward(ctx, x, alpha, beta, mod):
        y = mod(x)
        ctx.mod, ctx.x_dtype = mod, x.dtype
        ctx.p_dtypes = (alpha.dtype, None if beta is None else beta.dtype)
        ctx.save_for_backward(_k(x))
        return y

    @staticmethod
    def backward(ctx, gy):
        xin, = ctx.saved_tensors
        mod = ctx.mod
        B, C, T = xin.shape
        L = _lib.lib()
        g = gy.detach().to(xin.dtype).contiguous()
        gx = torch.empty_like(xin)
        alpha, beta, fu, fd = mod._params()
        want_p = any(ctx.needs_input_grad[1:3])         # frozen parameters: gx only
        da = torch.empty(C, dtype=torch.float32, device=xin.device) if want_p else None
        db = None if beta is None or not want_p else torch.empty_like(da)
        ns = L.kvae_aa_act_bwd_scratch_bytes(B, C, T) if want_p else 0
        scratch = torch.empty(ns, dtype=torch.uint8, device=xin.device) if want_p else None
        _lib.check(L.kvae_aa_act_bwd(xin.data_ptr(), g.data_ptr(), gx.data_ptr(), alpha.data_ptr(), _lib.ptr(beta),
                                     int(mod.act.alpha_logscale), fu.data_ptr(), fd.data_ptr(), _lib.ptr(da),
                                     _lib.ptr(db), B, C, T, _lib.dtype_code(xin.dtype), _lib.ptr(scratch), ns,
                                     _lib.stream_ptr(xin.device)))
        if not want_p:
            return gx.to(ctx.x_dtype), None, None, None
        return (gx.to(ctx.x_dtype), da.to(ctx.p_dtypes[0]), None if db is None else db.to(ctx.p_dtypes[1]), None)


class LeakyReLU(nn.Module):
    def __init__(self, negative_slope: float = 0.01, inplace: bool = False):
        super().__init__()
        self.negative_slope = negative_slope

    def forward(self, x):
        return _unary(x, 0, self.negative_slope)


class Snake(nn.Module):
    """Parameter holder of flows.py:9-61 (alpha); applied inside Activation1d's fused kernel."""

    def __init__(self, in_features, alpha=1.0, alpha_trainable=True, alpha_logscale=False):
        super().__init__()
        self.in_features, self.alpha_logscale = in_features, alpha_logscale
        init = torch.zeros if alpha_logscale else torch.ones
        self.alpha = nn.Parameter(init(in_features) * alpha, requires_grad=alpha_trainable)


class SnakeBeta(nn.Module):
    """Parameter holder of flows.py:64-125 (alpha, beta); applied inside Activation1d's fused kernel."""

    def __init__(self, in_features, alpha=1.0, alpha_trainable=True, alpha_logscale=False):
        super().__init__()
        self.in_features, self.alpha_logscale = in_features, alpha_logscale
        init = torch.zeros if alpha_logscale else torch.ones
        self.alpha = nn.Parameter(init(in_features) * alpha, requires_grad=alpha_trainable)
        self.beta = nn.Parameter(init(in_features) * alpha, requires_grad=alpha_trainable)


class _Filter(nn.Module):
    def __init__(self, ratio: int, kernel_size: int):
        super().__init__()
        self.register_buffer("filter", _kaiser_sinc_filter1d(0.5 / ratio, 0.6 / ratio, kernel_size))


class _Down(nn.Module):
    def __init__(self, ratio: int, kernel_size: int):
        super().__init__()
        self.lowpass = _Filter(ratio, kernel_size)


class Activation1d(nn.Module):
    """alias_free_torch.Activation1d (used at flows.py:266, 312, 443) with the same buffers (``upsample.filter``,
    ``downsample.lowpass.filter``) and ``act`` sub-module; forward is ONE kernel."""

    def __init__(self, activation, up_ratio: int = 2, down_ratio: int = 2, up_kernel_size: int = 12,
                 down_kernel_size: int = 12):
        super().__init__()
        if (up_ratio, down_ratio, up_kernel_size, down_kernel_size) != (2, 2, 12, 12):
            raise NotImplementedError("Activation1d: ratio 2 / 12 taps only (the values flows.py uses)")
        self.act = activation
        self.upsample = _Filter(up_ratio, up_kernel_size)
        self.downsample = _Down(down_ratio, down_kernel_size)

    def _params(self):
        """(alpha, beta or None, upsampling filter, low-pass filter): the fp32 device vectors the kernels read."""
        fu = self.upsample.filter.detach().float().reshape(-1).contiguous()
        fd = self.downsample.lowpass.filter.detach().float().reshape(-1).contiguous()
        alpha, beta = self.act.alpha.detach().float().contiguous(), getattr(self.act, "beta", None)
        return alpha, None if beta is None else beta.detach().float().contiguous(), fu, fd

    def forward(self, x):
        _lib.require_cuda(x, "Activation1d")
        if torch.is_grad_enabled() and _grad_on(x, self.act.alpha, getattr(self.act, "beta", None)):
            return _AaActFn.apply(x, self.act.alpha, getattr(self.act, "beta", None), self)
        xin = _k(x)
        B, C, T = xin.shape
        y = torch.empty_like(xin)
        alpha, beta, fu, fd = self._params()
        _lib.check(_lib.lib().kvae_aa_act_fwd(xin.data_ptr(), y.data_ptr(), alpha.data_ptr(), _lib.ptr(beta),
                                              int(self.act.alpha_logscale), fu.data_ptr(), fd.data_ptr(), B, C, T,
                                              _lib.dtype_code(xin.dtype), _lib.stream_ptr(x.device)))
        return y if y.dtype == x.dtype else y.to(x.dtype)

    def ragged(self, x, valid_len):
        """forward on a batch whose row b ends at valid_len[b] (kvae_aa_act_ragged_fwd): rows t < valid_len[b] equal
        forward(x[b:b+1, :, :valid_len[b]]), rows past it are 0.  x: contiguous fp32 / bf16 [B, C, T]."""
        B, C, T = x.shape
        y = torch.empty_like(x)
        alpha, beta, fu, fd = self._params()
        _lib.check(_lib.lib().kvae_aa_act_ragged_fwd(x.data_ptr(), y.data_ptr(), alpha.data_ptr(), _lib.ptr(beta),
                                                     int(self.act.alpha_logscale), fu.data_ptr(), fd.data_ptr(), B, C, T,
                                                     (ctypes.c_int * B)(*valid_len), _lib.dtype_code(x.dtype),
                                                     _lib.stream_ptr(x.device)))
        return y

    def window(self, win, x0, o0, o1, t_end):
        """Outputs [o0, o1) of the stream whose absolute rows [x0, x0 + W) are the window ``win`` [B, C, W] (fp32 /
        bf16, rows at any pitch); replicate padding at row 0 and, when t_end >= 0, at the stream end t_end
        (kvae_aa_act_win_fwd)."""
        B, C, W = win.shape
        y = torch.empty((B, C, o1 - o0), dtype=win.dtype, device=win.device)
        if win.stride(2) != 1 or win.stride(0) != C * win.stride(1):
            win = win.contiguous()
        alpha, beta, fu, fd = self._params()
        _lib.check(_lib.lib().kvae_aa_act_win_fwd(win.data_ptr(), win.stride(1), x0, W, y.data_ptr(), o1 - o0, o0, o1,
                                                  t_end, alpha.data_ptr(), _lib.ptr(beta), int(self.act.alpha_logscale),
                                                  fu.data_ptr(), fd.data_ptr(), B, C, _lib.dtype_code(win.dtype),
                                                  _lib.stream_ptr(win.device)))
        return y


class Conv1d(WNConv1d):
    """flows.py:566-620: weight-normed Conv1d, 'same' padding or causal (left padding d (K - 1), :607-608).  A causal conv
    is the symmetric-padded conv's first T outputs, which is how it runs here."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, dilation=1, causal=False, bias=True):
        self.causal = bool(causal)
        pad = dilation * (kernel_size - 1) if causal else int((kernel_size * dilation - dilation) / 2)
        super().__init__(in_channels, out_channels, kernel_size, stride=stride, padding=pad, dilation=dilation, bias=bias)

    def keep(self, T: int) -> int:
        return T if self.causal and self.kernel_size[0] > 1 else self.out_len(T)


class ConvTranspose1d(WNConvTranspose1d):
    """flows.py:336-391: padding (k - stride) // 2, or causal: k == 2 stride, no padding, last `stride` samples dropped."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, causal=False):
        self.causal = bool(causal)
        if causal and kernel_size != 2 * stride:
            raise AssertionError("kernel_size must be equal to 2*stride in Causal ConvTranspose1d.")
        super().__init__(in_channels, out_channels, kernel_size, stride=stride,
                         padding=0 if causal else (kernel_size - stride) // 2)
        self._drop = stride if causal else 0

    def keep(self, T: int) -> int:
        return self.out_len(T) - self._drop


class Conv1d_S(nn.Module):
    """flows.py:139-172 (weight_norm form): ``self.layer`` = weight-normed Conv1d with padding d (k - 1) // 2."""

    def __init__(self, in_channels, out_channels, kernel_size=1, stride=1, dilation=1):
        super().__init__()
        self.layer = WNConv1d(in_channels, out_channels, kernel_size, stride=stride,
                              padding=dilation * (kernel_size - 1) // 2, dilation=dilation)

    def forward(self, x):
        return self.layer(x)


class ResStack(nn.Module):
    """flows.py:174-189."""

    def __init__(self, channel, kernel_size=3, base=3, nums=4):
        super().__init__()
        self.layers = nn.ModuleList([
            nn.Sequential(LeakyReLU(), WNConv1d(channel, channel, kernel_size, dilation=base ** i, padding=base ** i),
                          LeakyReLU(), WNConv1d(channel, channel, kernel_size, dilation=1, padding=1))
            for i in range(nums)])

    def forward(self, x):
        for layer in self.layers:
            x = _axpby(x, layer(x), 1.0, 1.0)
        return x


class Encoder(nn.Module):
    """flows.py:191-241."""

    def __init__(self, in_channels=1, out_channels=100, base_channels=12, proj_kernel_size=3, stack_kernel_size=3,
                 stack_dilation_base=2, stacks=6, channels=(12, 24, 48, 96, 192, 384, 768),
                 down_sample_factors=(2, 2, 2, 2, 4, 4), use_vae=False):
        super().__init__()
        if use_vae:
            out_channels = out_channels * 2
        layers: List[nn.Module] = [Conv1d_S(in_channels, base_channels, kernel_size=proj_kernel_size), LeakyReLU(0.2)]
        for (in_c, out_c), f in zip(zip(channels[:-1], channels[1:]), down_sample_factors):
            layers += [Conv1d_S(in_c, out_c, kernel_size=f * 2, stride=f),
                       ResStack(out_c, stack_kernel_size, stack_dilation_base, stacks), LeakyReLU(0.2)]
        layers += [Conv1d_S(channels[-1], out_channels, proj_kernel_size)]
        self.generator = nn.Sequential(*layers)

    def forward(self, conditions, z_inputs=None):
        return self.generator(conditions)


def _make_act(h, channels):
    if h.activation == "snake":
        return Activation1d(Snake(channels, alpha_logscale=h.snake_logscale))
    if h.activation == "snakebeta":
        return Activation1d(SnakeBeta(channels, alpha_logscale=h.snake_logscale))
    raise NotImplementedError("activation incorrectly specified. check the config file and look for 'activation'.")


class AMPBlock1(nn.Module):
    """flows.py:243-291."""

    def __init__(self, h, channels, kernel_size=3, dilation=(1, 3, 5), activation=None, causal=True):
        super().__init__()
        self.convs1 = nn.ModuleList([Conv1d(channels, channels, kernel_size, dilation=d, causal=causal) for d in dilation])
        self.convs2 = nn.ModuleList([Conv1d(channels, channels, kernel_size, dilation=1, causal=causal) for _ in dilation])
        self.num_layers = len(self.convs1) + len(self.convs2)
        self.activations = nn.ModuleList([_make_act(h, channels) for _ in range(self.num_layers)])

    def forward(self, x):
        acts1, acts2 = self.activations[::2], self.activations[1::2]
        for c1, c2, a1, a2 in zip(self.convs1, self.convs2, acts1, acts2):
            x = _axpby(c2(a2(c1(a1(x)))), x, 1.0, 1.0)
        return x


class AMPBlock2(nn.Module):
    """flows.py:294-335."""

    def __init__(self, h, channels, kernel_size=3, dilation=(1, 3), activation=None, causal=True):
        super().__init__()
        self.convs = nn.ModuleList([Conv1d(channels, channels, kernel_size, dilation=d, causal=causal) for d in dilation])
        self.num_layers = len(self.convs)
        self.activations = nn.ModuleList([_make_act(h, channels) for _ in range(self.num_layers)])

    def forward(self, x):
        for c, a in zip(self.convs, self.activations):
            x = _axpby(c(a(x)), x, 1.0, 1.0)
        return x


# ------------------------------------------------------------------------------------------------- the flow
# ResidualCouplingBlock (flows.py:613-792, VITS): coupling layers with an unconditioned WaveNet, each followed by Flip.
# Between the convs every step is one flow.cuh kernel with its own autograd node: the split of x0 off the block input,
# the mask after `pre`, WN's gate and residual / skip update, and the coupling update, which writes its output with the
# following Flip applied and also the next layer's `pre` input, so channel splits, concatenations and flips are no pass
# of their own.
def _flow_call(name, *args):
    _lib.check(getattr(_lib.lib(), name)(*args))


def _flow_split(x, flip):
    B, C, T = x.shape
    xs = torch.empty_like(x)
    x0 = torch.empty((B, C // 2, T), dtype=x.dtype, device=x.device)
    _flow_call("kvae_flow_split", x.data_ptr(), xs.data_ptr(), x0.data_ptr(), B, C, T, int(flip),
               _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    return xs, x0


def _flow_mask(x, mask):
    B, C, T = x.shape
    y = torch.empty_like(x)
    _flow_call("kvae_flow_mask", x.data_ptr(), mask.data_ptr(), y.data_ptr(), B, C, T, _lib.dtype_code(x.dtype),
               _lib.stream_ptr(x.device))
    return y


def _wn_gate(a):
    B, H2, T = a.shape
    acts = torch.empty((B, H2 // 2, T), dtype=a.dtype, device=a.device)
    _flow_call("kvae_wn_gate_fwd", a.data_ptr(), acts.data_ptr(), B, H2 // 2, T, _lib.dtype_code(a.dtype),
               _lib.stream_ptr(a.device))
    return acts


def _wn_update(x, rs, skip, mask, last):
    B, H, T = x.shape
    x_out = None if last else torch.empty_like(x)
    skip_out = torch.empty_like(x)
    _flow_call("kvae_wn_update_fwd", x.data_ptr(), rs.data_ptr(), _lib.ptr(skip), mask.data_ptr(), _lib.ptr(x_out),
               skip_out.data_ptr(), B, H, int(last), T, _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    return x_out, skip_out


def _flow_coupling(x, m, mask, flip, reverse, want_y0):
    B, C, T = x.shape
    y = torch.empty_like(x)
    y0 = torch.empty((B, C // 2, T), dtype=x.dtype, device=x.device) if want_y0 else None
    _flow_call("kvae_flow_coupling_fwd", x.data_ptr(), m.data_ptr(), mask.data_ptr(), y.data_ptr(), _lib.ptr(y0), B, C,
               T, int(flip), int(reverse), _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device))
    return y, y0


def _g(t):
    return None if t is None else t.detach().contiguous()


class _FlowSplitFn(torch.autograd.Function):
    """(xs, x0) = (x or flip(x), its first half): kvae_flow_split / kvae_flow_split_bwd."""

    @staticmethod
    def forward(ctx, x, flip):
        ctx.set_materialize_grads(False)
        ctx.flip = flip
        return _flow_split(x, flip)

    @staticmethod
    def backward(ctx, gxs, gx0):
        gxs, gx0 = _g(gxs), _g(gx0)
        ref = gxs if gxs is not None else gx0
        if ref is None:
            return None, None
        B, C, T = gxs.shape if gxs is not None else (gx0.shape[0], 2 * gx0.shape[1], gx0.shape[2])
        gx = torch.empty((B, C, T), dtype=ref.dtype, device=ref.device)
        _flow_call("kvae_flow_split_bwd", _lib.ptr(gxs), _lib.ptr(gx0), gx.data_ptr(), B, C, T, int(ctx.flip),
                   _lib.dtype_code(ref.dtype), _lib.stream_ptr(ref.device))
        return gx, None


class _FlowMaskFn(torch.autograd.Function):
    """y = x * mask: kvae_flow_mask both ways (no gradient to the mask)."""

    @staticmethod
    def forward(ctx, x, mask):
        ctx.save_for_backward(mask)
        return _flow_mask(x, mask)

    @staticmethod
    def backward(ctx, gy):
        mask, = ctx.saved_tensors
        return _flow_mask(gy.detach().contiguous(), mask), None


class _WNGateFn(torch.autograd.Function):
    """acts = tanh(a[:, :H]) sigmoid(a[:, H:]): kvae_wn_gate_fwd / kvae_wn_gate_bwd (a saved)."""

    @staticmethod
    def forward(ctx, a):
        ctx.save_for_backward(a)
        return _wn_gate(a)

    @staticmethod
    def backward(ctx, g):
        a, = ctx.saved_tensors
        B, H2, T = a.shape
        g = g.detach().contiguous()
        ga = torch.empty_like(a)
        _flow_call("kvae_wn_gate_bwd", a.data_ptr(), g.data_ptr(), ga.data_ptr(), B, H2 // 2, T,
                   _lib.dtype_code(a.dtype), _lib.stream_ptr(a.device))
        return ga


class _WNUpdateFn(torch.autograd.Function):
    """WN's residual / skip update of one layer: kvae_wn_update_fwd / kvae_wn_update_bwd.  Returns (x_out, skip_out), or
    skip_out * mask (WN's output) for the last layer."""

    @staticmethod
    def forward(ctx, x, rs, skip, mask, last):
        ctx.set_materialize_grads(False)
        ctx.last, ctx.has_skip, ctx.shape = last, skip is not None, x.shape
        ctx.save_for_backward(mask)
        x_out, skip_out = _wn_update(x, rs, skip, mask, last)
        return skip_out if last else (x_out, skip_out)

    @staticmethod
    def backward(ctx, *grads):
        mask, = ctx.saved_tensors
        g_x, g_s = (None, _g(grads[0])) if ctx.last else (_g(grads[0]), _g(grads[1]))
        B, H, T = ctx.shape
        ref = g_s if g_s is not None else g_x
        if ref is None:
            return None, None, None, None, None
        gx = None if ctx.last else torch.empty((B, H, T), dtype=ref.dtype, device=ref.device)
        grs = torch.empty((B, H if ctx.last else 2 * H, T), dtype=ref.dtype, device=ref.device)
        # the skip input's gradient: g_skipout itself (written only where it is masked or missing)
        write_skip = ctx.has_skip and (ctx.last or g_s is None)
        gskip = torch.empty((B, H, T), dtype=ref.dtype, device=ref.device) if write_skip else None
        _flow_call("kvae_wn_update_bwd", _lib.ptr(g_x), _lib.ptr(g_s), mask.data_ptr(), _lib.ptr(gx), grs.data_ptr(),
                   _lib.ptr(gskip), B, H, int(ctx.last), T, _lib.dtype_code(ref.dtype), _lib.stream_ptr(ref.device))
        if ctx.has_skip and not write_skip:
            gskip = g_s
        return gx, grs, gskip, None, None


class _FlowCouplingFn(torch.autograd.Function):
    """(y, y0) of the coupling update (+ Flip): kvae_flow_coupling_fwd / kvae_flow_coupling_bwd (reads only the mask)."""

    @staticmethod
    def forward(ctx, x, m, mask, flip, reverse, want_y0):
        ctx.set_materialize_grads(False)
        ctx.flip, ctx.reverse, ctx.shape = flip, reverse, x.shape
        ctx.save_for_backward(mask)
        return _flow_coupling(x, m, mask, flip, reverse, want_y0)

    @staticmethod
    def backward(ctx, gy, gy0):
        mask, = ctx.saved_tensors
        gy, gy0 = _g(gy), _g(gy0)
        ref = gy if gy is not None else gy0
        if ref is None:
            return (None,) * 6
        B, C, T = ctx.shape
        gx = torch.empty((B, C, T), dtype=ref.dtype, device=ref.device)
        gm = torch.empty((B, C // 2, T), dtype=ref.dtype, device=ref.device)
        _flow_call("kvae_flow_coupling_bwd", _lib.ptr(gy), _lib.ptr(gy0), mask.data_ptr(), gx.data_ptr(), gm.data_ptr(),
                   B, C, T, int(ctx.flip), int(ctx.reverse), _lib.dtype_code(ref.dtype), _lib.stream_ptr(ref.device))
        return gx, gm, None, None, None, None


def _flow_inputs(x, x_mask, g, what):
    """x as a contiguous fp32 / bf16 [B, C, T] tensor and the mask [B, 1, T] as a detached contiguous tensor of x's
    dtype."""
    if g is not None:
        raise NotImplementedError(f"{what}: conditioning (g) is not supported: the flow has no cond_layer")
    _lib.require_cuda(x, what)
    if x.dim() != 3 or x.dtype not in (torch.float32, torch.bfloat16):
        raise ValueError(f"{what}: x must be a float32 or bfloat16 [B, C, T] tensor, got {x.dtype} {tuple(x.shape)}")
    B, _, T = x.shape
    if tuple(x_mask.shape) != (B, 1, T):
        raise ValueError(f"{what}: x_mask must be [B, 1, T] = {(B, 1, T)}, got {tuple(x_mask.shape)}")
    if x_mask.device != x.device:
        raise ValueError(f"{what}: x_mask is on {x_mask.device}, x on {x.device}")
    return x.contiguous(), x_mask.detach().to(x.dtype).contiguous()


class _PlainConv1d(_WNConvBase):
    """nn.Conv1d(in, out, 1) with its plain ``weight`` / ``bias`` (the coupling layers' ``pre`` and ``post``) on the
    layer-level conv: the engine choice of ``set_precision`` and the conv autograd node of every other layer."""
    transposed = False

    def __init__(self, in_channels, out_channels, kernel_size=1):
        super().__init__()
        conv = nn.Conv1d(in_channels, out_channels, kernel_size)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding, self.dilation = (int(kernel_size),), (1,), (0,), (1,)
        self.groups = 1
        self._parameters["weight"] = nn.Parameter(conv.weight.detach().clone())     # nn.Conv1d's key order
        self._parameters["bias"] = nn.Parameter(conv.bias.detach().clone())


class Flip(nn.Module):
    """flows.py Flip: torch.flip(x, [1]) (kvae_flow_split).  Inside ResidualCouplingBlock the coupling kernels apply
    it; called on its own it is one pass.  The forward direction returns (x, logdet = 0) as VITS does."""

    def forward(self, x, *args, reverse=False, **kwargs):
        _lib.require_cuda(x, "Flip")
        if x.dim() != 3 or x.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("Flip: x must be a float32 or bfloat16 [B, C, T] tensor")
        x = x.contiguous()
        if x.shape[1] % 2:
            raise ValueError("Flip: the flow's channel count is even")
        y = (_FlowSplitFn.apply(x, True) if _grad_on(x) else _flow_split(x, True))[0]
        return y if reverse else (y, torch.zeros(x.size(0), dtype=x.dtype, device=x.device))


class WN(nn.Module):
    """VITS modules.WN without conditioning: ``in_layers`` (hidden -> 2 hidden, kernel K, dilation rate^i) and
    ``res_skip_layers`` (hidden -> 2 hidden, the last hidden -> hidden), built interleaved as VITS builds them."""

    def __init__(self, hidden_channels, kernel_size, dilation_rate, n_layers, gin_channels=0, p_dropout=0):
        super().__init__()
        if gin_channels:
            raise NotImplementedError("WN: conditioning (gin_channels > 0) is not supported")
        if p_dropout:
            raise NotImplementedError("WN: dropout is not supported (the flow uses p_dropout = 0)")
        assert kernel_size % 2 == 1
        self.hidden_channels, self.kernel_size = hidden_channels, kernel_size
        self.dilation_rate, self.n_layers = dilation_rate, n_layers
        self.in_layers = nn.ModuleList()
        self.res_skip_layers = nn.ModuleList()
        for i in range(n_layers):
            d = dilation_rate ** i
            self.in_layers.append(WNConv1d(hidden_channels, 2 * hidden_channels, kernel_size, dilation=d,
                                           padding=int((kernel_size * d - d) / 2)))
            self.res_skip_layers.append(WNConv1d(hidden_channels, 2 * hidden_channels if i < n_layers - 1
                                                 else hidden_channels, 1))

    def forward(self, x, x_mask, g=None, **kwargs):
        x, mask = _flow_inputs(x, x_mask, g, "WN")
        return self._run(x, mask)

    def _run(self, x, mask):
        skip = None
        for i, (cin, crs) in enumerate(zip(self.in_layers, self.res_skip_layers)):
            a = cin(x)
            acts = _WNGateFn.apply(a) if _grad_on(a) else _wn_gate(a)
            rs = crs(acts)
            last = i == self.n_layers - 1
            if _grad_on(x, rs, skip):
                out = _WNUpdateFn.apply(x, rs, skip, mask, last)
            else:
                out = _wn_update(x, rs, skip, mask, last)
                out = out[1] if last else out
            if last:
                return out
            x, skip = out


class ResidualCouplingLayer(nn.Module):
    """VITS ResidualCouplingLayer with mean_only = True (``post`` zeroed at construction): x0, x1 = split(x);
    h = pre(x0) mask; h = WN(h, mask); m = post(h) mask; x1' = m + x1 mask (reverse: (x1 - m) mask); cat(x0, x1').
    The forward direction returns (x, logdet = 0), the reverse direction x, as VITS does."""

    def __init__(self, channels, hidden_channels, kernel_size, dilation_rate, n_layers, p_dropout=0, gin_channels=0,
                 mean_only=True):
        super().__init__()
        assert channels % 2 == 0, "channels should be divisible by 2"
        if not mean_only:
            raise NotImplementedError("ResidualCouplingLayer: mean_only=True only (the flow's coupling layers)")
        self.channels, self.hidden_channels, self.half_channels = channels, hidden_channels, channels // 2
        self.mean_only = True
        self.pre = _PlainConv1d(self.half_channels, hidden_channels, 1)
        self.enc = WN(hidden_channels, kernel_size, dilation_rate, n_layers, p_dropout=p_dropout,
                      gin_channels=gin_channels)
        self.post = _PlainConv1d(hidden_channels, self.half_channels, 1)
        self.post._parameters["weight"].data.zero_()
        self.post._parameters["bias"].data.zero_()

    def forward(self, x, x_mask, g=None, reverse=False):
        x, mask = _flow_inputs(x, x_mask, g, "ResidualCouplingLayer")
        if x.shape[1] != self.channels:
            raise ValueError(f"ResidualCouplingLayer: expected {self.channels} channels, got {x.shape[1]}")
        x, x0 = _FlowSplitFn.apply(x, False) if _grad_on(x) else _flow_split(x, False)
        y, _ = self._run(x, x0, mask, reverse, flip=False, want_y0=False)
        return y if reverse else (y, torch.zeros(x.size(0), dtype=x.dtype, device=x.device))

    def _run(self, x, x0, mask, reverse, flip, want_y0):
        """(y, y0): the layer on x with its first half x0 already split off; ``flip``: y with the following Flip
        applied; ``want_y0``: y's first half too (the next layer's x0)."""
        h = self.pre(x0)
        h = _FlowMaskFn.apply(h, mask) if _grad_on(h) else _flow_mask(h, mask)
        h = self.enc._run(h, mask)
        m = self.post(h)
        if _grad_on(x, m):
            return _FlowCouplingFn.apply(x, m, mask, flip, reverse, want_y0)
        return _flow_coupling(x, m, mask, flip, reverse, want_y0)


class ResidualCouplingBlock(nn.Module):
    """VITS ResidualCouplingBlock (flows.py:613-792): ``flows`` = [coupling layer, Flip] x n_flows.
    forward(x, x_mask, reverse=False): the layers in list order; reverse=True: in reversed order (each coupling layer
    then runs its inverse).  x [B, C, T] fp32 / bf16 (the result has x's dtype), x_mask [B, 1, T] (no gradient).
    Under autograd every coupling layer differentiates to x and its parameters (the WN convs' ``weight_g`` /
    ``weight_v`` / ``bias``, ``pre`` / ``post``'s ``weight`` / ``bias``); under ``torch.no_grad`` the same kernels run."""

    def __init__(self, channels, hidden_channels, kernel_size, dilation_rate, n_layers, n_flows=4, gin_channels=0):
        super().__init__()
        if gin_channels:
            raise NotImplementedError("ResidualCouplingBlock: conditioning (gin_channels > 0) is not supported")
        self.channels, self.hidden_channels, self.kernel_size = channels, hidden_channels, kernel_size
        self.dilation_rate, self.n_layers, self.n_flows, self.gin_channels = dilation_rate, n_layers, n_flows, 0
        self.flows = nn.ModuleList()
        for _ in range(n_flows):
            self.flows.append(ResidualCouplingLayer(channels, hidden_channels, kernel_size, dilation_rate, n_layers,
                                                    gin_channels=gin_channels, mean_only=True))
            self.flows.append(Flip())

    def forward(self, x, x_mask, g=None, reverse=False):
        x, mask = _flow_inputs(x, x_mask, g, "ResidualCouplingBlock")
        if x.shape[1] != self.channels:
            raise ValueError(f"ResidualCouplingBlock: expected {self.channels} channels, got {x.shape[1]}")
        layers = list(self.flows[0::2])
        if reverse:          # Flip, L_{n-1}^-1, Flip, ..., Flip, L_0^-1: each flip is applied by the kernel before it
            layers = layers[::-1]
        x, x0 = _FlowSplitFn.apply(x, reverse) if _grad_on(x) else _flow_split(x, reverse)
        for i, layer in enumerate(layers):
            more = i < len(layers) - 1
            x, x0 = layer._run(x, x0, mask, reverse, flip=more or not reverse, want_y0=more)
        return x


# ------------------------------------------------------------------------------------------------- layer descriptions
_AA_HALO = 5            # Activation1d: y[t] reads x[t - 5 .. t + 5] (12-tap x2 filters, bigvgan.cuh)


class _Geom:
    """Integer form of one op: how many output rows are final once ``R`` input rows have arrived.  A conv is the strided
    form with ``pl`` left and ``pr`` right zero rows (``padding`` on both sides, or on the left only when causal)."""

    def __init__(self, kind: str, K: int = 1, d: int = 1, s: int = 1, causal: bool = False, padding: int = 0):
        self.kind, self.K, self.d, self.s, self.causal = kind, K, d, s, causal
        if kind == "conv":
            self.span = d * (K - 1)
            self.pl = padding
            self.pr = 0 if causal else padding
        elif kind == "convT":
            self.span = K - 1
            self.p = 0 if causal else (K - s) // 2                       # flows.py:336-391
        elif kind == "act":
            self.span = 2 * _AA_HALO

    def total(self, R: int) -> int:
        """Output rows of the whole-utterance op on R input rows."""
        if self.kind == "conv":
            return (R + self.pl + self.pr - self.span - 1) // self.s + 1
        if self.kind == "convT":
            return R * self.s if self.causal else (R - 1) * self.s - 2 * self.p + self.K
        return R

    def avail(self, R: int, end: bool) -> int:
        if end:
            return max(0, self.total(R)) if R > 0 else 0
        if self.kind == "conv":                 # output o reads input rows o s - pl .. o s - pl + span
            return max(0, (R + self.pl - self.span - 1) // self.s + 1)
        if self.kind == "convT":
            return max(0, R * self.s - self.p)
        return max(0, R - _AA_HALO)

    def lookahead(self) -> int:
        """Rows after an output's own position that it reads (in output rows; a strided conv: input rows past the
        last of its own stride group)."""
        if self.kind == "conv":
            return self.span - self.pl - (self.s - 1)
        return self.p if self.kind == "convT" else _AA_HALO

    def reach(self) -> int:
        """Input rows before an output's own first row that it reads (a conv's left padding)."""
        if self.kind == "conv":
            return self.pl
        return 0 if self.kind == "convT" else _AA_HALO

    def first_read(self, e: int) -> int:
        """First input row that the outputs from row e on read (a conv: rounded down to a whole stride group)."""
        if self.kind == "conv":
            return max(0, e * self.s - self.pl) // self.s * self.s
        if self.kind == "convT":
            return max(0, -(-(e + self.p - self.K + 1) // self.s))
        return max(0, e - _AA_HALO)

    def origin(self, a: int) -> int:
        """Output row that a window starting at input row a (a conv: a multiple of the stride) numbers 0 when its rows
        are passed window-relative."""
        if self.kind == "conv":
            return a // self.s
        return a * self.s if self.kind == "convT" else a


class _Op(NamedTuple):
    """One op of a program over named streams.  ``kind``: conv, convT, act (``geom`` set), lrelu, tanh, or axpby
    (``coef`` = (alpha, beta): alpha * srcs[0] + beta * srcs[1]).  ``module``: the ``BigVGANFlowVAE`` attribute path
    of the layer that holds the weights, None for tanh / axpby."""
    kind: str
    module: Optional[str]
    srcs: Tuple[str, ...]
    dst: str
    geom: Optional[_Geom] = None
    coef: Optional[Tuple[float, float]] = None


def _program(h) -> Tuple[List[_Op], str]:
    """The inference path as a list of ops over named streams (flows.py:506-527 in execution order), from the input
    stream "z" to the returned output stream."""
    causal = bool(h["causal"])

    def conv(path, src, dst, K, d=1, causal=causal):
        pad = d * (K - 1) if causal else d * (K - 1) // 2                  # Conv1d (flows.py:607-608)
        return _Op("conv", path, (src,), dst, _Geom("conv", K, d, 1, causal, pad))

    def act(path, src, dst):
        return _Op("act", path, (src,), dst, _Geom("act"))

    def add(a, b, dst, alpha=1.0, beta=1.0):
        return _Op("axpby", None, (a, b), dst, coef=(alpha, beta))

    ops = [conv("conv_pre", "z", "x0", 7, causal=False)]
    nk = len(h["resblock_kernel_sizes"])
    x = "x0"
    for i, (u, ku) in enumerate(zip(h["upsample_rates"], h["upsample_kernel_sizes"])):
        up = f"u{i}"
        ops.append(_Op("convT", f"ups.{i}.0", (x,), up, _Geom("convT", int(ku), 1, int(u), causal)))
        xs = None
        for j, (k, dil) in enumerate(zip(h["resblock_kernel_sizes"], h["resblock_dilation_sizes"])):
            rb, cur, k = f"resblocks.{i * nk + j}", up, int(k)
            for q, d in enumerate(dil):
                t = f"{rb}.{q}"
                if h["resblock"] == "1":
                    ops += [act(f"{rb}.activations.{2 * q}", cur, t + "a1"),
                            conv(f"{rb}.convs1.{q}", t + "a1", t + "c1", k, int(d)),
                            act(f"{rb}.activations.{2 * q + 1}", t + "c1", t + "a2"),
                            conv(f"{rb}.convs2.{q}", t + "a2", t + "c2", k),
                            add(t + "c2", cur, t + "r")]
                else:
                    ops += [act(f"{rb}.activations.{q}", cur, t + "a"),
                            conv(f"{rb}.convs.{q}", t + "a", t + "c", k, int(d)),
                            add(t + "c", cur, t + "r")]
                cur = t + "r"
            if xs is None:
                xs = cur
            else:
                ops.append(add(xs, cur, f"s{i}.{j}"))
                xs = f"s{i}.{j}"
        x = f"x{i + 1}"
        ops.append(add(xs, xs, x, 1.0 / nk, 0.0))
    ops += [act("activation_post", x, "ap"), conv("conv_post", "ap", "cp", 7),
            _Op("tanh", None, ("cp",), "wav")]
    return ops, "wav"


def _encoder_program(h) -> Tuple[List[_Op], str]:
    """Encoder.generator (flows.py:191-241) as a list of ops over named streams, in execution order, from the input
    stream "x" to "lat".  Conv1d_S pads d (K - 1) // 2, so the strided conv (K = 2 f, stride f) maps L rows to
    (L - 2) // f + 1; the ResStack has 6 layers at dilations 1 .. 32 (``Encoder``'s stacks / stack_dilation_base)."""
    p = "audio_encoder.generator"

    def conv(path, src, dst, K, s=1, d=1):
        return _Op("conv", path, (src,), dst, _Geom("conv", K, d, s, padding=d * (K - 1) // 2))

    def lrelu(path, src, dst):
        return _Op("lrelu", path, (src,), dst)

    ops = [conv(f"{p}.0.layer", "x", "h", 3), lrelu(f"{p}.1", "h", "a0")]
    x, idx = "a0", 2
    for i, f in enumerate(h["downsample_rates"]):
        f = int(f)
        ops.append(conv(f"{p}.{idx}.layer", x, f"s{i}", 2 * f, f))
        x = f"s{i}"
        for j in range(6):
            rs, t = f"{p}.{idx + 1}.layers.{j}", f"s{i}.{j}"
            ops += [lrelu(f"{rs}.0", x, t + "a"), conv(f"{rs}.1", t + "a", t + "c", 3, d=2 ** j),
                    lrelu(f"{rs}.2", t + "c", t + "b"), conv(f"{rs}.3", t + "b", t + "d", 3),
                    _Op("axpby", None, (x, t + "d"), t + "r", coef=(1.0, 1.0))]
            x = t + "r"
        ops.append(lrelu(f"{p}.{idx + 2}", x, f"a{i + 1}"))
        x, idx = f"a{i + 1}", idx + 3
    ops.append(conv(f"{p}.{idx}.layer", x, "lat", 3))
    return ops, "lat"


def _lengths(h, encoder: bool, n: int, end: bool = True) -> Dict[str, int]:
    """Rows of every stream of the encoder's (``encoder``) or the decoder's op list for one clip of ``n`` input rows;
    0 from the first op on that would get no rows (the clip's own call raises there).  ``end=False``: the rows that are
    final while more input may follow (the streams' integer interpreter)."""
    ops, _ = _encoder_program(h) if encoder else _program(h)
    R = {"x" if encoder else "z": int(n)}
    for op in ops:
        rows = min(R[s] for s in op.srcs)
        R[op.dst] = op.geom.avail(rows, end) if op.geom else rows
    return R


def latent_length(h, n_samples: int) -> int:
    """Latent frames ``extract_latents`` returns for ``n_samples`` samples: the chained floors of the encoder's convs."""
    return _lengths(h, True, n_samples)["lat"]


def wav_length(h, n_frames: int) -> int:
    """Samples ``inference_from_latents`` returns for ``n_frames`` latent frames, from the decoder's layer arithmetic."""
    return _lengths(h, False, n_frames)[_program(h)[1]]


# ------------------------------------------------------------------------------------------------- ragged batches
def ragged_order(valid_len: Sequence[int]) -> Tuple[List[int], List[int]]:
    """(order, inverse): ``order`` lists the clips longest first (ties keep their index order), ``inverse[b]`` is clip
    b's position in it, so ``sorted_batch[inverse]`` restores the caller's order."""
    order = sorted(range(len(valid_len)), key=lambda b: -int(valid_len[b]))
    inverse = [0] * len(order)
    for i, b in enumerate(order):
        inverse[b] = i
    return order, inverse


def tc_split(rows: Sequence[int]) -> int:
    """Clips of a longest-first batch whose own call runs a tensor-core layer on the tensor cores: those with at least
    ``TC_MIN_ROWS`` input rows there, a prefix of the batch."""
    n = sum(1 for r in rows if r >= TC_MIN_ROWS)
    if any(r < TC_MIN_ROWS for r in rows[:n]):
        raise ValueError("tc_split: rows must be sorted longest first")
    return n


def _check_valid_len(valid_len, B: int, T: int, out_len, what: str) -> List[int]:
    if isinstance(valid_len, torch.Tensor):
        valid_len = valid_len.tolist()
    lens = [int(v) for v in valid_len]
    if len(lens) != B:
        raise ValueError(f"{what}: valid_len has {len(lens)} entries for a batch of {B}")
    if B > _RAGGED_MAX_CLIPS:
        raise ValueError(f"{what}: at most {_RAGGED_MAX_CLIPS} clips per ragged call, got {B}")
    for b, v in enumerate(lens):
        if not 1 <= v <= T:
            raise ValueError(f"{what}: valid_len[{b}] = {v} is outside 1 .. {T} (the padded length)")
        if out_len(v) < 1:
            raise ValueError(f"{what}: clip {b} ({v} rows) is too short to give any output row")
    return lens


def _zero_tail(x: torch.Tensor, rows: Sequence[int]) -> None:
    """x[b, :, rows[b]:] = 0 in place (x: a contiguous [B, C, T] tensor of fp32 or bf16)."""
    B, C, T = x.shape
    _lib.check(_lib.lib().kvae_zero_tail_cf(x.data_ptr(), B, C, T, T, (ctypes.c_int * B)(*rows),
                                            _lib.dtype_code(x.dtype), _lib.stream_ptr(x.device)))


def _conv_ragged(m, x: torch.Tensor, rows: Sequence[int]) -> torch.Tensor:
    """m(x) on a longest-first batch, each clip on the engine its own call picks: at most two launches."""
    n = tc_split(rows) if m.tc_layer() else 0
    if n in (0, x.shape[0]):
        return m(x, tc=n > 0)
    return torch.cat([m(x[:n], tc=True), m(x[n:], tc=False)], dim=0)


def _run_ragged(model, encoder: bool, x: torch.Tensor, lens: List[int]) -> torch.Tensor:
    """The encoder's or decoder's op list on the longest-first batch ``x`` (rows past each clip's end: anything), clip b
    holding lens[b] input rows.  Rows past a clip's end are zeroed where the next op reads them as padding: the input
    of every non-causal conv (the decoder's activations already store zeros there) and of a non-causal transposed
    conv, and the output."""
    h = model.h
    ops, out = _encoder_program(h) if encoder else _program(h)
    R = [_lengths(h, encoder, n) for n in lens]
    src = "x" if encoder else "z"
    last = {}                                     # stream -> index of the op that reads it last
    for i, op in enumerate(ops):
        for name in op.srcs:
            last[name] = i
    vals = {src: x}
    _zero_tail(x, [r[src] for r in R])
    for i, op in enumerate(ops):
        xin = vals[op.srcs[0]]
        if op.kind in ("conv", "convT"):
            rows = [r[op.srcs[0]] for r in R]
            if encoder and op.srcs[0] != src or op.kind == "convT" and not op.geom.causal:
                _zero_tail(xin, rows)
            vals[op.dst] = _conv_ragged(_module(model, op.module), xin, rows)
        elif op.kind == "act":
            vals[op.dst] = _module(model, op.module).ragged(xin, [r[op.srcs[0]] for r in R])
        elif op.kind == "lrelu":
            vals[op.dst] = _module(model, op.module)(xin)
        elif op.kind == "axpby":
            vals[op.dst] = _axpby(xin, vals[op.srcs[1]], *op.coef)
        else:
            vals[op.dst] = _unary(xin, 1)
        for name in [k for k, j in last.items() if j == i]:
            vals.pop(name, None)
    y = vals[out]
    _zero_tail(y, [r[out] for r in R])
    return y


def _module(model, path: str):
    m = model
    for p in path.split("."):
        m = m[int(p)] if p.isdigit() else getattr(m, p)
    return m


class BigVGANFlowVAE(nn.Module):
    def __init__(self, h):
        super().__init__()
        self.h = h
        causal = h.causal
        self.audio_encoder = Encoder(out_channels=h.latent_dim, use_vae=h.use_vae, channels=list(h.downsample_channels),
                                     down_sample_factors=list(h.downsample_rates))
        # VITS builds this block as ResidualCouplingBlock(inter, hidden, 5, 1, 4); the checkpoint fixes everything but the
        # dilation rate 1, which changes no parameter shape (DESIGN §4.10g)
        self.flow = ResidualCouplingBlock(h.latent_dim, h.flow_hidden_channels, 5, 1, 4)
        self.num_kernels = len(h.resblock_kernel_sizes)
        self.num_upsamples = len(h.upsample_rates)
        self.conv_pre = Conv1d(h.latent_dim, h.upsample_initial_channel, 7, 1, causal=False)
        resblock = AMPBlock1 if h.resblock == "1" else AMPBlock2
        self.ups = nn.ModuleList()
        for i, (u, k) in enumerate(zip(h.upsample_rates, h.upsample_kernel_sizes)):
            self.ups.append(nn.ModuleList([ConvTranspose1d(h.upsample_initial_channel // (2 ** i),
                                                           h.upsample_initial_channel // (2 ** (i + 1)), k, u, causal=causal)]))
        self.resblocks = nn.ModuleList()
        ch = h.upsample_initial_channel
        for i in range(len(self.ups)):
            ch = h.upsample_initial_channel // (2 ** (i + 1))
            for k, d in zip(h.resblock_kernel_sizes, h.resblock_dilation_sizes):
                self.resblocks.append(resblock(h, ch, k, d, activation=h.activation, causal=causal))
        self.activation_post = _make_act(h, ch)
        self.conv_post = Conv1d(ch, 1, 7, 1, causal=causal)
        self.set_precision("fp32")
        for m in self.modules():           # no-grad calls fold weight norm once per weight version (layers.py)
            if isinstance(m, _WNConvBase):
                m._cache_fold = True

    def set_precision(self, precision: Optional[str]):
        """Arithmetic of the convolutions whose channel counts are multiples of 64 (the wide stages, > 90 % of the
        FLOPs of a production-size model): "fp32" (default) = tensor cores through the bf16x3 operand split (<= 1e-5),
        "bf16" = bf16 tensor-core operands (<= 1e-3 class), None = fp32 CUDA-core kernels everywhere."""
        if precision not in (None, "fp32", "bf16"):
            raise ValueError("precision must be None, 'fp32' or 'bf16'")
        for m in self.modules():
            if isinstance(m, _WNConvBase):
                m.tc_precision = precision
        return self

    def forward(self, x):
        raise NotImplementedError("BigVGANFlowVAE.forward (the training pass through the flow, flows.py:454-492) is "
                                  "not built; use extract_latents / inference_from_latents, or compose encode_with_grad, "
                                  "flow and decode_with_grad for training")

    def latent_length(self, n_samples: int) -> int:
        """Latent frames ``extract_latents`` returns for a clip of ``n_samples`` samples (0: too short for any)."""
        return latent_length(self.h, n_samples)

    def wav_length(self, n_frames: int) -> int:
        """Samples ``inference_from_latents`` returns for ``n_frames`` latent frames."""
        return wav_length(self.h, n_frames)

    def _ragged(self, encoder: bool, x: torch.Tensor, valid_len, what: str) -> torch.Tensor:
        """Clips sorted longest first (so each conv splits into at most two engine groups), run, put back."""
        _lib.require_cuda(x, what)
        if x.dim() != 3 or x.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError(f"{what}: valid_len needs a float32 or bfloat16 [B, C, T] input")
        out_len = self.latent_length if encoder else self.wav_length
        lens = _check_valid_len(valid_len, x.shape[0], x.shape[2], out_len, what)
        order, inverse = ragged_order(lens)
        xs = x[torch.tensor(order, device=x.device)].contiguous()     # a copy: its padding rows are zeroed in place
        y = _run_ragged(self, encoder, xs, [lens[b] for b in order])
        return y if order == sorted(order) else y[torch.tensor(inverse, device=y.device)]

    @torch.no_grad()
    def extract_latents(self, x, valid_len=None):
        """``valid_len`` (host sequence of B ints, 1 <= valid_len[b] <= T, B <= 64): clip b is x[b, :, :valid_len[b]];
        what x holds past that is ignored.  out[b, :, :latent_length(valid_len[b])] then equals
        ``extract_latents(x[b:b+1, :, :valid_len[b]])`` bit for bit, and the rest of out[b] is 0."""
        if valid_len is not None:
            return self._ragged(True, x, valid_len, "extract_latents")
        return self.audio_encoder(x)

    def encode_with_grad(self, x, valid_len=None):
        """``extract_latents`` under autograd: the same kernels on the same engines, so the output is ``torch.equal`` to
        it under every ``set_precision``, and ``backward`` reaches the audio (when it requires grad) and every parameter
        of the encoder that requires grad (the convs' ``weight_g`` / ``weight_v`` / ``bias``).  The convs' data and
        weight gradients run on the engine their forward ran on: tensor cores for the wide layers, the strided
        downsampling convs included; no weight-gradient work for a frozen encoder.  ``decode_with_grad(
        encode_with_grad(x), noise=...)`` is the whole autoencoder under autograd.  Ragged batches and the streams are
        inference-only.  Under ``torch.no_grad`` it is ``extract_latents``."""
        if valid_len is not None:
            raise NotImplementedError("encode_with_grad: valid_len (ragged batches) has no backward; encode each clip "
                                      "on its own or pad the batch")
        return self.audio_encoder(x)

    @torch.no_grad()
    def inference_from_latents(self, x, do_sample=True, noise: Optional[torch.Tensor] = None, valid_len=None):
        """``valid_len`` (host sequence of B ints, frames, 1 <= valid_len[b] <= T, B <= 64): clip b is
        x[b, :, :valid_len[b]]; what x (and noise) hold past that is ignored.  out[b, :, :wav_length(valid_len[b])]
        then equals the call on x[b:b+1, :, :valid_len[b]] (noise[b:b+1, :, :valid_len[b]]) bit for bit, and the rest
        of out[b] is 0."""
        return self._decode(x, do_sample, noise, valid_len)

    def decode_with_grad(self, x, do_sample=True, noise: Optional[torch.Tensor] = None, valid_len=None):
        """``inference_from_latents`` under autograd: the same kernels on the same engines, so the output is
        ``torch.equal`` to it (same ``noise``) under every ``set_precision``, and ``backward`` reaches the latents (mean
        and log-scale when sampling) and every parameter of the decoder that requires grad -- the convs' ``weight_g`` /
        ``weight_v`` / ``bias`` and the activations' ``alpha`` / ``beta``.  Each backward step is a libkvae kernel: the
        fused anti-aliased activation backward, the convs' data and weight gradients on the engine their forward ran on
        (tensor cores for the wide layers), no weight-gradient work for a frozen decoder.  Ragged batches and the streams
        are inference-only.  Under ``torch.no_grad`` it is ``inference_from_latents``."""
        if valid_len is not None:
            raise NotImplementedError("decode_with_grad: valid_len (ragged batches) has no backward; decode each clip "
                                      "on its own or pad the batch")
        return self._decode(x, do_sample, noise, None)

    def _decode(self, x, do_sample, noise, valid_len):
        h = self.h
        if h.use_vae and do_sample:
            assert x.size(1) == h.latent_dim * 2, "Input must be like [B, D, H]"
            m_q, logs_q = torch.split(x, h.latent_dim, dim=1)
            if noise is None:
                noise = torch.randn_like(m_q)
            if _grad_on(x):
                x = _GaussSampleFn.apply(x, noise, h.latent_dim)
            else:
                x = _gauss_sample(m_q, logs_q, noise)
        else:
            assert x.size(1) == h.latent_dim, "Input must be like [B, D, H]"
        if valid_len is not None:
            return self._ragged(False, x, valid_len, "inference_from_latents")
        x = self.conv_pre(x)
        for i in range(self.num_upsamples):
            for up in self.ups[i]:
                x = up(x)
            xs = None
            for j in range(self.num_kernels):
                y = self.resblocks[i * self.num_kernels + j](x)
                xs = y if xs is None else _axpby(xs, y, 1.0, 1.0)
            x = _axpby(xs, xs, 1.0 / self.num_kernels, 0.0)
        x = self.activation_post(x)
        x = self.conv_post(x)
        return _unary(x, 1)

    def remove_weight_norm(self):
        for m in self.modules():
            if isinstance(m, (WNConv1d, WNConvTranspose1d)) and m.has_weight_norm:
                m.remove_weight_norm()
