"""Drop-in for the reference's Oobleck discriminator (the GAN half of the autoencoder's training losses).

Same class names, constructor arguments, module tree and ``state_dict`` keys as
``stable_audio_tools/models/discriminators.py``:
  * get_hinge_losses                                   :11-14
  * SharedDiscriminatorConvNet                         :62-116   (``net.{0,2,4,6}.{bias,weight_g,weight_v}``, ``net.8.{weight,bias}``)
  * MultiScaleDiscriminator / MultiPeriodDiscriminator :119-168
  * MultiDiscriminator                                 :171-238
  * OobleckDiscriminator (``loss(reals, fakes)``)      :240-297   wired at training/autoencoders.py:133-134, 288
Parameters are initialised through torch's own ``nn.Conv1d`` / ``nn.Conv2d`` constructors in the reference's order, so
the same ``torch.manual_seed`` gives the reference's random-init ``state_dict``.

Compute: every net is ONE autograd node (``_SharedNetFn``) whose forward and backward chain libkvae kernels -- the
strided convolutions on ``kvae_disc_conv15_fwd`` / ``kvae_disc_conv15_bwd`` (fp32 kernels written for the nets' k = 15 /
stride 4 geometry; any other geometry on ``kvae_conv1d_fwd`` / ``kvae_conv1d_win_bwd``), everything between them on the
other ``kvae_disc_*`` entry points (csrc/disc.cuh).  The multi-period nets' 15 x 15 ``Conv2d`` over ``[N, C, ceil(T / n), n]``
runs as a ``Conv1d`` over the folded channels ``(c, w)``: identical products, without the ones that only ever meet the
zero padding of the width axis (n <= 11 < 15).  ``EncodecDiscriminator`` and ``DACGANLoss`` wrap un-vendored packages
(``encodec.msstftd``, ``dac.model.discriminator`` / ``audiotools``) whose arithmetic is not in the reference tree; they
raise ``NotImplementedError``.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
import typing as tp
from functools import reduce

import numpy as np
import torch
from torch import nn

from . import _lib


def _f32c(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    return t.contiguous() if t.dtype == torch.float32 else t.float().contiguous()


# KVAE_DISC_GENERIC=1: development switch -- every conv on the generic layer kernels (kvae_conv1d_fwd / kvae_conv1d_win_bwd)
# instead of the kernels written for the nets' own k = 15 / stride 4 / padding 7 geometry (same results to fp32 rounding)
_GENERIC = os.environ.get("KVAE_DISC_GENERIC", "0") == "1"


def _conv_fwd(x, w, bias, Cin, Cout, K, stride, pad):
    """Conv1d on [N, Cin, T] fp32 with a folded weight [Cout, Cin, K]."""
    L = _lib.lib()
    N, _, T = x.shape
    T_out = (T + 2 * pad - K) // stride + 1
    if T_out <= 0:
        raise RuntimeError("Kernel size can't be greater than actual input size")
    y = torch.empty((N, Cout, T_out), dtype=torch.float32, device=x.device)
    if not _GENERIC and L.kvae_disc_conv1x1_supported(K, stride, pad, Cout):
        _lib.check(L.kvae_disc_conv1x1_fwd(x.data_ptr(), y.data_ptr(), w.data_ptr(), _lib.ptr(bias), N, Cin, Cout, T,
                                           _lib.stream_ptr(x.device)))
        return y
    ns = L.kvae_conv1d_scratch_bytes(Cin, Cout, K)
    scratch = torch.empty(ns, dtype=torch.uint8, device=x.device)
    if not _GENERIC and L.kvae_disc_conv15_supported(K, stride, pad):
        _lib.check(L.kvae_disc_conv15_fwd(x.data_ptr(), y.data_ptr(), w.data_ptr(), _lib.ptr(bias), N, Cin, Cout, T,
                                          scratch.data_ptr(), ns, _lib.stream_ptr(x.device)))
        return y
    _lib.check(L.kvae_conv1d_fwd(x.data_ptr(), y.data_ptr(), w.data_ptr(), _lib.ptr(bias), 0, N, Cin, Cout, T, K, stride, 1,
                                 pad, _lib.KVAE_F32, scratch.data_ptr(), ns, _lib.stream_ptr(x.device)))
    return y


def _conv_bwd(x, gy, w, Cin, Cout, K, stride, pad, want_gx, want_dw, want_db):
    L = _lib.lib()
    N, _, T = x.shape
    gx = torch.empty_like(x) if want_gx else None
    dw = torch.empty_like(w) if want_dw else None
    db = torch.empty(Cout, dtype=torch.float32, device=x.device) if want_db else None
    if gx is None and dw is None and db is None:
        return None, None, None
    if not _GENERIC and L.kvae_disc_conv1x1_supported(K, stride, pad, Cout):
        _lib.check(L.kvae_disc_conv1x1_bwd(x.data_ptr(), gy.data_ptr(), w.data_ptr(), _lib.ptr(gx), _lib.ptr(dw), _lib.ptr(db),
                                           N, Cin, Cout, T, _lib.stream_ptr(x.device)))
        return gx, dw, db
    if not _GENERIC and L.kvae_disc_conv15_supported(K, stride, pad):
        ns = L.kvae_conv1d_scratch_bytes(Cin, Cout, K)
        scratch = torch.empty(ns, dtype=torch.uint8, device=x.device)
        _lib.check(L.kvae_disc_conv15_bwd(x.data_ptr(), gy.data_ptr(), w.data_ptr(), _lib.ptr(gx), _lib.ptr(dw), _lib.ptr(db),
                                          N, Cin, Cout, T, scratch.data_ptr(), ns, _lib.stream_ptr(x.device)))
        return gx, dw, db
    T_gy = gy.shape[2]
    ns = L.kvae_conv1d_win_bwd_scratch_bytes(0, N, Cin, Cout, T, T_gy, K, stride, 0)
    scratch = torch.empty(ns, dtype=torch.uint8, device=x.device)
    _lib.check(L.kvae_conv1d_win_bwd(x.data_ptr(), gy.data_ptr(), T_gy, w.data_ptr(), None, None, _lib.ptr(gx), _lib.ptr(dw),
                                     None, _lib.ptr(db), 0, N, Cin, Cout, T, K, stride, 1, pad, _lib.KVAE_F32, 0,
                                     scratch.data_ptr(), ns, _lib.stream_ptr(x.device)))
    return gx, dw, db


class _DiscConv(nn.Module):
    """Parameter holder for one convolution of a SharedDiscriminatorConvNet: ``weight_norm(nn.ConvNd(...))`` (old-style
    ``bias`` / ``weight_g`` / ``weight_v``) or a plain ``nn.ConvNd`` (``weight`` / ``bias``), 1-D or 2-D with a square
    kernel, as discriminators.py:85-106 builds them.  The compute lives in ``_SharedNetFn``."""

    def __init__(self, two_d, in_channels, out_channels, kernel_size, stride=1, padding=0, weight_norm=True):
        super().__init__()
        conv = (nn.Conv2d if two_d else nn.Conv1d)(in_channels, out_channels, kernel_size, stride=stride, padding=padding)
        self.two_d, self.in_channels, self.out_channels = bool(two_d), in_channels, out_channels
        self.kernel_size, self.stride, self.padding = int(kernel_size), int(stride), int(padding)
        self.weight_normed = bool(weight_norm)
        w = conv.weight.detach()
        if weight_norm:     # torch registers bias first, then weight_g, weight_v
            self.bias = nn.Parameter(conv.bias.detach().clone())
            self.weight_g = nn.Parameter(torch.norm_except_dim(w, 2, 0).clone())
            self.weight_v = nn.Parameter(w.clone())
        else:
            self.weight = nn.Parameter(w.clone())
            self.bias = nn.Parameter(conv.bias.detach().clone())

    def params(self):
        return (self.bias, self.weight_g, self.weight_v) if self.weight_normed else (self.weight, self.bias)

    def extra_repr(self):
        k = (self.kernel_size,) * (2 if self.two_d else 1)
        return f"{self.in_channels}, {self.out_channels}, kernel_size={k}, stride={self.stride}, padding={self.padding}"

    def folded(self, W):
        """(conv weight [Cout', Cin', K] fp32, bias [Cout'], torch-layout folded weight, output width) for an input whose
        folded axis has width W (1-D nets: W = 1 and nothing is folded)."""
        L = _lib.lib()
        if self.weight_normed:
            v, g = _f32c(self.weight_v), _f32c(self.weight_g)
            _lib.require_cuda(v, "discriminator")
            w = torch.empty_like(v)
            _lib.check(L.kvae_weight_norm_fold(v.data_ptr(), g.data_ptr(), w.data_ptr(), v.shape[0], v[0].numel(),
                                               _lib.stream_ptr(v.device)))
        else:
            w = _f32c(self.weight)
            _lib.require_cuda(w, "discriminator")
        b = _f32c(self.bias)
        if not self.two_d:
            return w.view(self.out_channels, self.in_channels, self.kernel_size), b, w, 1
        K, s, p = self.kernel_size, self.stride, self.padding
        Wo = L.kvae_disc_folded_width(W, K, s, p)
        if Wo <= 0:
            raise RuntimeError("Kernel size can't be greater than actual input size")
        wf = torch.empty((self.out_channels * Wo, self.in_channels * W, K), dtype=torch.float32, device=w.device)
        bf = torch.empty(self.out_channels * Wo, dtype=torch.float32, device=w.device)
        _lib.check(L.kvae_disc_fold_weight2d(w.data_ptr(), b.data_ptr(), wf.data_ptr(), bf.data_ptr(), self.out_channels,
                                             self.in_channels, K, s, p, W, 0, _lib.stream_ptr(w.device)))
        return wf, bf, w, Wo


class _SharedNetFn(torch.autograd.Function):
    """SharedDiscriminatorConvNet.forward (:108-116) and its backward on the folded layout: x [N, Cin W, T] ->
    (score [N], feature_0 .. feature_L), feature_l [N, Cout_l W_l, T_l] being the l-th conv's output."""

    @staticmethod
    def forward(ctx, net, W_in, x, *params):
        L = _lib.lib()
        convs = net.convs()
        st = _lib.stream_ptr(x.device)
        a = _f32c(x)
        N = a.shape[0]
        saved, geoms, feats = [a], [], []
        W = int(W_in)
        for i, cv in enumerate(convs):
            wf, bf, w_torch, Wo = cv.folded(W)
            Cin, Cout = cv.in_channels * W, cv.out_channels * Wo
            f = _conv_fwd(a, wf, bf, Cin, Cout, cv.kernel_size, cv.stride, cv.padding)
            geoms.append((Cin, Cout, W, Wo))
            feats.append(f)
            saved.append(wf)
            if i + 1 < len(convs):
                a = torch.empty_like(f)
                _lib.check(L.kvae_disc_silu_fwd(f.data_ptr(), a.data_ptr(), f.numel(), st))
                saved.append(a)
            W = Wo
        score = torch.empty(N, dtype=torch.float32, device=a.device)
        last = feats[-1]
        _lib.check(L.kvae_disc_score(last.data_ptr(), score.data_ptr(), N, last[0].numel(), 0, st))
        ctx.net, ctx.geoms, ctx.n_saved = net, geoms, len(saved)
        ctx.param_dtypes = [p.dtype for p in params]
        ctx.save_for_backward(*saved, *feats, *[p.detach() for p in params])
        return (score, *feats)

    @staticmethod
    def backward(ctx, g_score, *g_feats):
        L = _lib.lib()
        net = ctx.net
        convs = net.convs()
        n_l = len(convs)
        tensors = ctx.saved_tensors
        saved, feats, params = tensors[:ctx.n_saved], tensors[ctx.n_saved:ctx.n_saved + n_l], tensors[ctx.n_saved + n_l:]
        # saved = [a_0 (= x), wf_0, a_1, wf_1, ..., a_{L-1}, wf_{L-1}]
        acts, wfs = saved[0::2], saved[1::2]
        dev = acts[0].device
        st = _lib.stream_ptr(dev)
        need = ctx.needs_input_grad      # (net, W_in, x, *params)
        want_params = any(need[3:])
        gf = [None if g is None else _f32c(g) for g in g_feats]
        gs = None if g_score is None else _f32c(g_score)
        last = feats[-1]
        N = last.shape[0]
        if gs is None and gf[-1] is None:
            g = None
        else:
            g = torch.empty_like(last)
            _lib.check(L.kvae_disc_score_bwd(_lib.ptr(gs), _lib.ptr(gf[-1]), g.data_ptr(), N, last[0].numel(), st))
        pgrads: tp.List[tp.Optional[torch.Tensor]] = [None] * len(params)
        g_x = None
        pi = len(params)
        for i in range(n_l - 1, -1, -1):     # g: gradient at the output of conv i (feature i), or None
            cv = convs[i]
            pi -= 3 if cv.weight_normed else 2
            Cin, Cout, W, Wo = ctx.geoms[i]
            if g is None:                    # nothing reaches feature i: feature i-1 only has its own gradient
                g = gf[i - 1] if i > 0 else None
                continue
            want_gx = i > 0 or need[2]
            gx, dwf, dbf = _conv_bwd(acts[i], g, wfs[i], Cin, Cout, cv.kernel_size, cv.stride, cv.padding, want_gx,
                                     want_params, want_params)
            if want_params:
                if cv.two_d:                 # folded-channel gradients -> torch's [Cout, Cin, K, K] / [Cout]
                    dw = torch.empty((cv.out_channels, cv.in_channels, cv.kernel_size, cv.kernel_size),
                                     dtype=torch.float32, device=dev)
                    db = torch.empty(cv.out_channels, dtype=torch.float32, device=dev)
                    _lib.check(L.kvae_disc_fold_weight2d(dw.data_ptr(), db.data_ptr(), dwf.data_ptr(), dbf.data_ptr(),
                                                         cv.out_channels, cv.in_channels, cv.kernel_size, cv.stride,
                                                         cv.padding, W, 1, st))
                else:
                    dw, db = dwf, dbf
                if cv.weight_normed:
                    gp, vp = params[pi + 1], params[pi + 2]
                    v, gg = _f32c(vp), _f32c(gp)
                    dv = torch.empty_like(v)
                    dg = torch.empty(v.shape[0], dtype=torch.float32, device=dev)
                    _lib.check(L.kvae_weight_norm_bwd(v.data_ptr(), gg.data_ptr(), dw.data_ptr(), dv.data_ptr(),
                                                      dg.data_ptr(), v.shape[0], v[0].numel(), st))
                    pgrads[pi] = db.to(ctx.param_dtypes[pi])
                    pgrads[pi + 1] = dg.view_as(gp).to(ctx.param_dtypes[pi + 1])
                    pgrads[pi + 2] = dv.view_as(vp).to(ctx.param_dtypes[pi + 2])
                else:
                    pgrads[pi] = dw.view_as(params[pi]).to(ctx.param_dtypes[pi])
                    pgrads[pi + 1] = db.to(ctx.param_dtypes[pi + 1])
            if i > 0:                        # through the SiLU, plus the gradient arriving at feature i-1 itself
                f_prev = feats[i - 1]
                _lib.check(L.kvae_disc_silu_bwd(f_prev.data_ptr(), gx.data_ptr(), _lib.ptr(gf[i - 1]), gx.data_ptr(),
                                                f_prev.numel(), st))
                g = gx
            else:
                g_x = gx
        return (None, None, g_x, *pgrads)


class SharedDiscriminatorConvNet(nn.Module):

    def __init__(
        self,
        in_size: int,
        convolution: tp.Union[nn.Conv1d, nn.Conv2d],
        out_size: int = 1,
        capacity: int = 32,
        n_layers: int = 4,
        kernel_size: int = 15,
        stride: int = 4,
        activation: tp.Optional[tp.Callable[[], nn.Module]] = None,
        normalization: tp.Optional[tp.Callable[[nn.Module], nn.Module]] = None,
    ) -> None:
        super().__init__()
        if convolution not in (nn.Conv1d, nn.Conv2d):
            raise NotImplementedError("SharedDiscriminatorConvNet: convolution must be nn.Conv1d or nn.Conv2d")
        if normalization is not None and normalization is not torch.nn.utils.weight_norm:
            raise NotImplementedError("SharedDiscriminatorConvNet: only the default normalization (weight_norm) is built")
        if not isinstance(kernel_size, int):
            raise NotImplementedError("SharedDiscriminatorConvNet: integer kernel_size only (every reference config)")
        self.two_d = convolution is nn.Conv2d
        channels = [in_size] + list(int(c) for c in capacity * 2 ** np.arange(n_layers))
        if isinstance(stride, int):
            stride = n_layers * [stride]
        net: tp.List[nn.Module] = []
        for i in range(n_layers):
            net.append(_DiscConv(self.two_d, channels[i], channels[i + 1], kernel_size, stride=stride[i],
                                 padding=kernel_size // 2, weight_norm=True))
            act = nn.SiLU() if activation is None else activation()
            if not isinstance(act, nn.SiLU):
                raise NotImplementedError("SharedDiscriminatorConvNet: only the default activation (nn.SiLU) is built")
            net.append(act)
        net.append(_DiscConv(self.two_d, channels[-1], out_size, 1, weight_norm=False))
        self.net = nn.ModuleList(net)

    def convs(self) -> tp.List[_DiscConv]:
        return [m for m in self.net if isinstance(m, _DiscConv)]

    def _params(self):
        return [p for cv in self.convs() for p in cv.params()]

    def forward_folded(self, xf: torch.Tensor, W: int):
        """xf [N, C W, H] (the width axis folded into the channels; W = 1 for the 1-D nets) -> (score [N], features in the
        reference's shapes: [N, C', T'] or [N, C', H', W'])."""
        _lib.require_cuda(xf, "SharedDiscriminatorConvNet.forward")
        if xf.dim() != 3 or xf.shape[1] != self.convs()[0].in_channels * W:
            raise ValueError(f"expected [N, {self.convs()[0].in_channels * W}, T], got {tuple(xf.shape)}")
        if xf.shape[0] == 0 or xf.shape[2] == 0:
            raise ValueError("empty input")
        score, *feats = _SharedNetFn.apply(self, W, xf, *self._params())
        if self.two_d:
            N = xf.shape[0]
            feats = [f.view(N, cv.out_channels, -1, f.shape[2]).transpose(2, 3) for f, cv in zip(feats, self.convs())]
        return score, feats

    def forward(self, x):
        if self.two_d:      # [N, C, H, W] -> [N, C W, H]
            if x.dim() != 4:
                raise ValueError("expected [N, C, H, W]")
            N, Cc, H, W = x.shape
            return self.forward_folded(x.permute(0, 1, 3, 2).reshape(N, Cc * W, H), W)
        return self.forward_folded(x, 1)


class _AvgPool2Fn(torch.autograd.Function):
    """nn.functional.avg_pool1d(x, 2) (:137)"""

    @staticmethod
    def forward(ctx, x):
        xin = _f32c(x)
        N, Cc, T = xin.shape
        if T < 2:
            raise RuntimeError("avg_pool1d(2): input shorter than the pooling window")
        y = torch.empty((N, Cc, T // 2), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib().kvae_disc_avg_pool2(xin.data_ptr(), y.data_ptr(), N * Cc, T, 0, _lib.stream_ptr(x.device)))
        ctx.shape, ctx.x_dtype = (N, Cc, T), x.dtype
        return y

    @staticmethod
    def backward(ctx, gy):
        N, Cc, T = ctx.shape
        g = _f32c(gy)
        gx = torch.empty((N, Cc, T), dtype=torch.float32, device=g.device)
        _lib.check(_lib.lib().kvae_disc_avg_pool2(g.data_ptr(), gx.data_ptr(), N * Cc, T, 1, _lib.stream_ptr(g.device)))
        return gx.to(ctx.x_dtype)


class _PeriodFoldFn(torch.autograd.Function):
    """MultiPeriodDiscriminator.fold (:164-168) straight into the folded-channel layout [N, C n, ceil(T / n)]"""

    @staticmethod
    def forward(ctx, x, n):
        xin = _f32c(x)
        N, Cc, T = xin.shape
        H = (T + n - 1) // n
        y = torch.empty((N, Cc * n, H), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib().kvae_disc_period_fold(xin.data_ptr(), y.data_ptr(), N, Cc, T, n, 0, _lib.stream_ptr(x.device)))
        ctx.shape, ctx.n, ctx.x_dtype = (N, Cc, T), n, x.dtype
        return y

    @staticmethod
    def backward(ctx, gy):
        N, Cc, T = ctx.shape
        g = _f32c(gy)
        gx = torch.empty((N, Cc, T), dtype=torch.float32, device=g.device)
        _lib.check(_lib.lib().kvae_disc_period_fold(g.data_ptr(), gx.data_ptr(), N, Cc, T, ctx.n, 1, _lib.stream_ptr(g.device)))
        return gx.to(ctx.x_dtype), None


IndividualDiscriminatorOut = tp.Tuple[torch.Tensor, tp.Sequence[torch.Tensor]]
TensorDict = tp.Dict[str, torch.Tensor]


class MultiScaleDiscriminator(nn.Module):

    def __init__(self, in_channels: int, n_scales: int, **conv_kwargs) -> None:
        super().__init__()
        self.layers = nn.ModuleList([SharedDiscriminatorConvNet(in_channels, nn.Conv1d, **conv_kwargs)
                                     for _ in range(n_scales)])

    def forward(self, x: torch.Tensor) -> IndividualDiscriminatorOut:
        _lib.require_cuda(x, "MultiScaleDiscriminator.forward")
        score = 0
        features = []
        for layer in self.layers:
            s, f = layer(x)
            score = score + s
            features.extend(f)
            x = _AvgPool2Fn.apply(x)
        return score, features


class MultiPeriodDiscriminator(nn.Module):

    def __init__(self, in_channels: int, periods: tp.Sequence[int], **conv_kwargs) -> None:
        super().__init__()
        self.periods = periods
        self.layers = nn.ModuleList([SharedDiscriminatorConvNet(in_channels, nn.Conv2d, **conv_kwargs) for _ in periods])

    def forward(self, x: torch.Tensor) -> IndividualDiscriminatorOut:
        _lib.require_cuda(x, "MultiPeriodDiscriminator.forward")
        score = 0
        features = []
        for layer, n in zip(self.layers, self.periods):
            s, f = layer.forward_folded(_PeriodFoldFn.apply(x, int(n)), int(n))
            score = score + s
            features.extend(f)
        return score, features

    def fold(self, x: torch.Tensor, n: int) -> torch.Tensor:
        """the reference's [N, C, ceil(T / n), n] view (host-side helper; ``forward`` folds on the device)"""
        pad = (n - (x.shape[-1] % n)) % n
        x = nn.functional.pad(x, (0, pad))
        return x.reshape(*x.shape[:2], -1, n)


class MultiDiscriminator(nn.Module):
    """Individual discriminators take one tensor (NxB C T) and return a score tensor (NxB) and a sequence of features."""

    def __init__(self, discriminator_list: tp.Sequence[nn.Module], keys: tp.Sequence[str]) -> None:
        super().__init__()
        self.discriminators = nn.ModuleList(discriminator_list)
        self.keys = keys

    def unpack_tensor_to_dict(self, features: torch.Tensor) -> TensorDict:
        features = features.chunk(len(self.keys), 0)
        return {k: features[i] for i, k in enumerate(self.keys)}

    @staticmethod
    def concat_dicts(dict_a, dict_b):
        out_dict = {}
        for k in set(list(dict_a.keys()) + list(dict_b.keys())):
            out_dict[k] = []
            for d in (dict_a, dict_b):
                if k in d:
                    if isinstance(d[k], list):
                        out_dict[k].extend(d[k])
                    else:
                        out_dict[k].append(d[k])
        return out_dict

    @staticmethod
    def sum_dicts(dict_a, dict_b):
        out_dict = {}
        for k in set(list(dict_a.keys()) + list(dict_b.keys())):
            out_dict[k] = 0.
            if k in dict_a:
                out_dict[k] = out_dict[k] + dict_a[k]
            if k in dict_b:
                out_dict[k] = out_dict[k] + dict_b[k]
        return out_dict

    def forward(self, inputs: TensorDict) -> TensorDict:
        discriminator_input = torch.cat([inputs[k] for k in self.keys], 0)
        all_scores = []
        all_features = []
        for discriminator in self.discriminators:
            score, features = discriminator(discriminator_input)
            scores = self.unpack_tensor_to_dict(score)
            all_scores.append({f"score_{k}": scores[k] for k in scores.keys()})
            features = reduce(self.concat_dicts, map(self.unpack_tensor_to_dict, features))
            all_features.append({f"features_{k}": features[k] for k in features.keys()})
        inputs.update(reduce(self.sum_dicts, all_scores))
        inputs.update(reduce(self.concat_dicts, all_features))
        return inputs


class _HingeFn(torch.autograd.Function):
    """get_hinge_losses on the batch-concatenated score [2B] = (reals | fakes): (dis_loss, gen_loss)"""

    @staticmethod
    def forward(ctx, score):
        s = _f32c(score)
        B = s.numel() // 2
        losses = torch.empty(2, dtype=torch.float32, device=s.device)
        _lib.check(_lib.lib().kvae_disc_hinge(s.data_ptr(), B, losses.data_ptr(), None, None, _lib.stream_ptr(s.device)))
        ctx.save_for_backward(s)
        ctx.s_dtype = score.dtype
        return losses[0], losses[1]

    @staticmethod
    def backward(ctx, g_dis, g_gen):
        (s,) = ctx.saved_tensors
        B = s.numel() // 2
        gl = torch.stack([torch.zeros((), device=s.device) if g is None else g.detach().float().reshape(())
                          for g in (g_dis, g_gen)]).contiguous()
        gs = torch.empty_like(s)
        _lib.check(_lib.lib().kvae_disc_hinge(s.data_ptr(), B, None, gl.data_ptr(), gs.data_ptr(), _lib.stream_ptr(s.device)))
        return gs.to(ctx.s_dtype)


class _FeatureMatchFn(torch.autograd.Function):
    """sum over the feature tensors of mean |real - fake| (:285-295), each tensor batch-concatenated (reals | fakes);
    one launch over all of them, one launch for all the gradients."""

    @staticmethod
    def _tables(feats, grads=None):
        n = len(feats)
        fp = (C.c_void_p * n)(*[f.data_ptr() for f in feats])
        half = (C.c_longlong * n)(*[f.numel() // 2 for f in feats])
        gp = None if grads is None else (C.c_void_p * n)(*[g.data_ptr() for g in grads])
        return fp, half, gp

    @staticmethod
    def forward(ctx, *feats):
        L = _lib.lib()
        fs = [_f32c(f) for f in feats]
        if any(f.shape[0] % 2 for f in fs):
            raise ValueError("feature tensors must hold the reals and the fakes on the batch axis")
        dev = fs[0].device
        fp, half, _ = _FeatureMatchFn._tables(fs)
        ns = L.kvae_disc_feature_match_scratch_bytes(half, len(fs))
        scratch = torch.empty(ns, dtype=torch.uint8, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        _lib.check(L.kvae_disc_feature_match(fp, half, len(fs), loss.data_ptr(), None, None, scratch.data_ptr(), ns,
                                             _lib.stream_ptr(dev)))
        ctx.save_for_backward(*fs)
        ctx.meta = [(f.dtype, f.shape) for f in feats]
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        L = _lib.lib()
        fs = ctx.saved_tensors
        dev = fs[0].device
        gl = g.detach().float().reshape(1).contiguous()
        grads = [torch.empty_like(f) for f in fs]
        fp, half, gp = _FeatureMatchFn._tables(fs, grads)
        _lib.check(L.kvae_disc_feature_match(fp, half, len(fs), gl.data_ptr(), gl.data_ptr(), gp, None, 0, _lib.stream_ptr(dev)))
        return tuple(gr.view(shape).to(dt) for gr, (dt, shape) in zip(grads, ctx.meta))


def get_hinge_losses(score_real, score_fake):
    _lib.require_cuda(score_real, "get_hinge_losses")
    dis_loss, gen_loss = _HingeFn.apply(torch.cat([score_real.reshape(-1), score_fake.reshape(-1)], 0))
    return dis_loss, gen_loss


class OobleckDiscriminator(nn.Module):

    def __init__(self, in_channels=1):
        super().__init__()
        multi_scale_discriminator = MultiScaleDiscriminator(in_channels=in_channels, n_scales=3)
        multi_period_discriminator = MultiPeriodDiscriminator(in_channels=in_channels, periods=[2, 3, 5, 7, 11])
        self.multi_discriminator = MultiDiscriminator([multi_scale_discriminator, multi_period_discriminator],
                                                      ["reals", "fakes"])

    def loss(self, reals, fakes):
        """(dis_loss, gen_loss, feature_matching_distance) of discriminators.py:269-297.  The nets run ONCE on the
        batch-concatenated input; the hinge losses and the distance read the scores / features as they lie in memory
        (first half reals, second half fakes), so nothing is split or copied between the nets and the losses."""
        _lib.require_cuda(reals, "OobleckDiscriminator.loss")
        _lib.require_cuda(fakes, "OobleckDiscriminator.loss")
        if reals.shape != fakes.shape:
            raise ValueError("reals and fakes must have the same shape")
        x = torch.cat([reals, fakes], 0)
        score, feats = 0, []
        for d in self.multi_discriminator.discriminators:
            s, f = d(x)
            score = score + s
            feats.extend(f)
        dis_loss, gen_loss = _HingeFn.apply(score)
        # the distance is invariant to the layout of a feature tensor: hand over the contiguous folded buffers
        fm = _FeatureMatchFn.apply(*[f.transpose(2, 3) if f.dim() == 4 else f for f in feats])
        return dis_loss, gen_loss, fm


class EncodecDiscriminator(nn.Module):
    def __init__(self, *args, **kwargs):
        super().__init__()
        raise NotImplementedError("EncodecDiscriminator wraps encodec.msstftd.MultiScaleSTFTDiscriminator, an un-vendored "
                                  "package whose arithmetic is not part of the reference tree (discriminators.py:16-23); "
                                  "use OobleckDiscriminator")


class DACGANLoss(nn.Module):
    def __init__(self, *args, **kwargs):
        super().__init__()
        raise NotImplementedError("DACGANLoss depends on the un-vendored audiotools / dac packages "
                                  "(discriminators.py:8-9, 300-545); use OobleckDiscriminator")
