"""Drop-in modules for the leaves of the Oobleck stack: SnakeBeta, WNConv1d, WNConvTranspose1d.

Same constructor arguments, attribute names, parameter names/shapes and ``state_dict`` keys as the
reference:
  * SnakeBeta                      stable_audio_tools/models/blocks.py:309-339
  * WNConv1d / WNConvTranspose1d   dac.nn.layers (un-vendored): ``weight_norm(nn.Conv1d(...))`` /
                                   ``weight_norm(nn.ConvTranspose1d(...))`` with old-style parameters
                                   ``weight_g`` / ``weight_v`` (call sites autoencoders.py:49-53,76,98)
Parameters are initialised through torch's own ``nn.Conv1d`` / ``nn.ConvTranspose1d`` constructors, so
the same ``torch.manual_seed`` yields the same random-init ``state_dict`` as the reference.

``forward`` / ``backward`` of a leaf run the layer-level C-ABI kernels (fp32 arithmetic by default, autograd nodes
``_SnakeFn`` / ``_ConvLayerFn``).  A conv with ``tc_precision`` set runs its forward on the tensor cores through
``packed_weight`` / ``conv_rows``, which the streaming BigVGAN decoder calls on its windows too.  ``engine`` picks the
engine of a call, and ``keep`` the output rows a layer keeps (BigVGANFlowVAE's causal layers keep the first ones).
Every conv layer, BigVGANFlowVAE's included, differentiates through ``_ConvLayerFn``: its forward is the no-grad call,
its backward ``kvae_conv1d_win_bwd`` on the same engine.  The fast path is not here: ``OobleckEncoder`` /
``OobleckDecoder`` hand the whole stack to a fused plan (see ``_plan.py``).
"""
from __future__ import annotations

import torch
from torch import nn

from . import _lib


class _SnakeFn(torch.autograd.Function):
    """SnakeBeta.forward / backward on [B, C, T] (blocks.py:331-339 and its autograd): kvae_snake_fwd / kvae_snake_bwd."""

    @staticmethod
    def forward(ctx, x, alpha, beta, logscale):
        a = alpha.detach().float().contiguous()
        b = beta.detach().float().contiguous()
        y = _snake_call(x.detach(), a, b, logscale)
        ctx.save_for_backward(x.detach(), a, b)
        ctx.logscale = bool(logscale)
        ctx.param_dtypes = (alpha.dtype, beta.dtype)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, a, b = ctx.saved_tensors
        B, Cc, T = x.shape
        # the kernel works on channels-last rows [B*T, C] (the layout of the fused plans)
        xr = x.float().transpose(1, 2).contiguous()
        gr = gy.detach().float().transpose(1, 2).contiguous()
        gx = torch.empty_like(xr)
        da = torch.empty(Cc, dtype=torch.float32, device=x.device)
        db = torch.empty(Cc, dtype=torch.float32, device=x.device)
        scratch = torch.empty(2 * Cc, dtype=torch.float32, device=x.device)
        if xr.numel():
            _lib.check(_lib.lib().kvae_snake_bwd(xr.data_ptr(), gr.data_ptr(), gx.data_ptr(), a.data_ptr(), b.data_ptr(),
                                                 int(ctx.logscale), da.data_ptr(), db.data_ptr(), B * T, Cc,
                                                 scratch.data_ptr(), _lib.stream_ptr(x.device)))
        else:
            da.zero_(); db.zero_()
        return (gx.transpose(1, 2).contiguous().to(x.dtype), da.to(ctx.param_dtypes[0]), db.to(ctx.param_dtypes[1]),
                None)


class _ConvLayerFn(torch.autograd.Function):
    """Every conv layer under autograd (WNConv1d / WNConvTranspose1d and BigVGANFlowVAE's layers built on them): the
    forward is the layer's no-grad call (grad mode is off inside), so it runs the same kernels on the same engine; the
    backward is kvae_conv1d_win_bwd on that engine (0 = CUDA cores fp32, 1 = tcgen05 bf16, 2 = tcgen05 bf16x3), with no
    weight-gradient work when no conv parameter requires grad.  A 'same' conv with an even kernel differentiates its
    padded input (one more zero row on the right) and returns the gradient of the first T rows."""

    @staticmethod
    def forward(ctx, mod, x, tc, bias, *wparams):
        T = x.shape[2]
        y = mod(x, tc)
        ctx.mod, ctx.engine, ctx.x_dtype, ctx.T, ctx.T_gy = mod, mod.engine(T, tc, mod.keep(T)), x.dtype, T, y.shape[2]
        ctx.has_bias = bias is not None
        xin = x.detach() if x.dtype in (torch.float32, torch.bfloat16) else x.detach().float()
        if mod._same_extra_right:
            xin = torch.nn.functional.pad(xin, (0, mod._same_extra_right))
        ctx.save_for_backward(xin.contiguous(), mod.folded_weight(), *[p.detach() for p in wparams])
        return y

    @staticmethod
    def backward(ctx, gy):
        mod = ctx.mod
        xin, w, *wparams = ctx.saved_tensors
        L = _lib.lib()
        B, Cin, T = xin.shape
        K, s, d, p = mod.kernel_size[0], mod.stride[0], mod.dilation[0], mod.padding[0]
        Cout, tr = mod.out_channels, int(mod.transposed)
        g = gy.detach().to(xin.dtype).contiguous()
        need = ctx.needs_input_grad
        gx = torch.empty_like(xin) if need[1] else None
        db = torch.empty(Cout, dtype=torch.float32, device=xin.device) if ctx.has_bias and need[3] else None
        dv = dg = vf = gf = None
        if any(need[4:]):
            if len(wparams) == 2:                  # (weight_g, weight_v): the weight norm's backward too
                gf, vf = (t.float().contiguous() for t in wparams)
                dg = torch.empty(vf.shape[0], dtype=torch.float32, device=vf.device)
            dv = torch.empty(w.shape, dtype=torch.float32, device=w.device)
        if gx is None and dv is None and db is None:
            return (None,) * (4 + len(wparams))
        ns = L.kvae_conv1d_win_bwd_scratch_bytes(tr, B, Cin, Cout, T, ctx.T_gy, K, s, ctx.engine)
        scratch = torch.empty(ns, dtype=torch.uint8, device=xin.device)
        _lib.check(L.kvae_conv1d_win_bwd(xin.data_ptr(), g.data_ptr(), ctx.T_gy, w.data_ptr(), _lib.ptr(vf), _lib.ptr(gf),
                                         _lib.ptr(gx), _lib.ptr(dv), _lib.ptr(dg), _lib.ptr(db), tr, B, Cin, Cout, T, K,
                                         s, d, p, _lib.dtype_code(xin.dtype), ctx.engine, scratch.data_ptr(), ns,
                                         _lib.stream_ptr(xin.device)))
        if dv is None:
            wgrads = (None,) * len(wparams)
        elif len(wparams) == 2:
            wgrads = (dg.view_as(wparams[0]).to(wparams[0].dtype), dv.to(wparams[1].dtype))
        else:
            wgrads = (dv.to(wparams[0].dtype),)
        return (None, None if gx is None else gx[:, :, :ctx.T].to(ctx.x_dtype), None, db, *wgrads)


def snake_beta(x, alpha, beta):
    """Functional form of blocks.py:301-302 (alpha, beta already exponentiated, broadcast [1,C,1])."""
    _lib.require_cuda(x, "snake_beta")
    a = alpha.reshape(-1).float().contiguous()
    b = beta.reshape(-1).float().contiguous()
    return _snake_call(x, a, b, logscale=False)


def _snake_call(x, alpha, beta, logscale):
    if x.dim() != 3:
        raise ValueError("SnakeBeta expects [B, C, T]")
    B, Cc, T = x.shape
    if alpha.numel() != Cc:
        raise ValueError(f"SnakeBeta has {alpha.numel()} channels, input has {Cc}")
    xin = x if x.dtype in (torch.float32, torch.bfloat16) else x.float()
    xin = xin.contiguous()
    y = torch.empty_like(xin)
    if xin.numel():
        _lib.check(_lib.lib().kvae_snake_fwd(xin.data_ptr(), y.data_ptr(), alpha.data_ptr(), beta.data_ptr(),
                                             int(logscale), B, Cc, T, _lib.dtype_code(xin.dtype),
                                             _lib.stream_ptr(x.device)))
    return y if y.dtype == x.dtype else y.to(x.dtype)


class SnakeBeta(nn.Module):
    def __init__(self, in_features, alpha=1.0, alpha_trainable=True, alpha_logscale=True):
        super().__init__()
        self.in_features = in_features
        self.alpha_logscale = alpha_logscale
        if self.alpha_logscale:
            self.alpha = nn.Parameter(torch.zeros(in_features) * alpha)
            self.beta = nn.Parameter(torch.zeros(in_features) * alpha)
        else:
            self.alpha = nn.Parameter(torch.ones(in_features) * alpha)
            self.beta = nn.Parameter(torch.ones(in_features) * alpha)
        self.alpha.requires_grad = alpha_trainable
        self.beta.requires_grad = alpha_trainable
        self.no_div_by_zero = 0.000000001

    def forward(self, x):
        _lib.require_cuda(x, "SnakeBeta.forward")
        if torch.is_grad_enabled() and (x.requires_grad or self.alpha.requires_grad or self.beta.requires_grad):
            return _SnakeFn.apply(x, self.alpha, self.beta, self.alpha_logscale)
        return _snake_call(x, self.alpha.detach().float().contiguous(), self.beta.detach().float().contiguous(),
                           self.alpha_logscale)


# Inputs shorter than this run on the CUDA cores even when ``tc_precision`` sends the layer to the tensor cores.
TC_MIN_ROWS = 64


def _single(v):
    if isinstance(v, (tuple, list)):
        if len(v) != 1:
            raise ValueError("1-D convolution arguments must be scalars or 1-tuples")
        return int(v[0])
    return int(v)


class _WNConvBase(nn.Module):
    transposed = False

    def _init_from(self, conv: nn.Module):
        # old-style weight_norm: bias stays first, then weight_g = ||v|| over all dims but 0, weight_v = v
        w = conv.weight.detach()
        if conv.bias is not None:
            self.bias = nn.Parameter(conv.bias.detach().clone())
        else:
            self.register_parameter("bias", None)
        self.weight_g = nn.Parameter(torch.norm_except_dim(w, 2, 0).clone())
        self.weight_v = nn.Parameter(w.clone())

    # --- weight-norm handling -------------------------------------------------------------------
    @property
    def has_weight_norm(self) -> bool:
        return "weight_g" in self._parameters

    def folded_weight(self) -> torch.Tensor:
        """fp32 folded weight w = v * g/||v|| computed on the device by libkvae (fold in fp32, round once)."""
        if not self.has_weight_norm:
            return self._parameters["weight"].detach().float().contiguous()
        # Inference-only models built from stand-alone layers (BigVGANFlowVAE) set ``_cache_fold``: the folded weight is
        # reused until weight_v / weight_g change (storage or torch version counter, i.e. .to(), load_state_dict and
        # in-place optimizer steps all invalidate it).  Read-only for the callers.
        key = None
        if getattr(self, "_cache_fold", False) and not torch.is_grad_enabled():
            key = (self.weight_v.data_ptr(), self.weight_v._version, self.weight_g.data_ptr(), self.weight_g._version)
            hit = self.__dict__.get("_fold_cache")
            if hit is not None and hit[0] == key:
                return hit[1]
        v = self.weight_v.detach().float().contiguous()
        g = self.weight_g.detach().float().contiguous()
        _lib.require_cuda(v, "weight-norm fold")
        w = torch.empty_like(v)
        _lib.check(_lib.lib().kvae_weight_norm_fold(v.data_ptr(), g.data_ptr(), w.data_ptr(), v.shape[0],
                                                    v[0].numel(), _lib.stream_ptr(v.device)))
        if key is not None:
            self.__dict__["_fold_cache"] = (key, w)
        return w

    @property
    def weight(self):
        if not self.has_weight_norm:
            return self._parameters["weight"]
        return self.folded_weight().to(self.weight_v.dtype)

    def remove_weight_norm(self):
        """torch.nn.utils.remove_weight_norm equivalent (reference models/utils.py:14-20): replaces
        weight_g / weight_v by a plain ``weight`` parameter."""
        if not self.has_weight_norm:
            raise ValueError("weight_norm already removed")
        w = self.folded_weight().to(self.weight_v.dtype)
        del self._parameters["weight_g"]
        del self._parameters["weight_v"]
        self.register_parameter("weight", nn.Parameter(w))
        return self

    def conv_params(self):
        return [p for p in self.parameters(recurse=False)]

    # --- layer-level forward -------------------------------------------------------------------
    def forward(self, x, tc=True):
        """``tc=False`` keeps the layer on the CUDA cores whatever ``tc_precision`` says (the short clips of a ragged
        BigVGANFlowVAE batch, which their own calls run there)."""
        _lib.require_cuda(x, type(self).__name__ + ".forward")
        if x.dim() != 3 or x.shape[1] != self.in_channels:
            raise ValueError(f"expected [B, {self.in_channels}, T], got {tuple(x.shape)}")
        if x.shape[0] == 0 or x.shape[2] == 0:
            raise ValueError("empty input")
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.conv_params())):
            wparams = (self.weight_g, self.weight_v) if self.has_weight_norm else (self._parameters["weight"],)
            return _ConvLayerFn.apply(self, x, tc, self.bias, *wparams)
        T = x.shape[2]
        keep = self.keep(T)
        engine = self.engine(T, tc, keep)
        xin = x if x.dtype in (torch.float32, torch.bfloat16) else x.float()
        if engine:       # the tensor cores truncate inside the kernel
            y = self.conv_rows(xin.contiguous(), *self.packed_weight(engine), engine, self.padding[0], 0, keep)
        else:
            y = self._forward_impl(xin)
            if keep < y.shape[2]:
                y = y[:, :, :keep].contiguous()
        return y if y.dtype == x.dtype else y.to(x.dtype)

    # Stand-alone layers run fp32 CUDA-core arithmetic by default.  ``tc_precision`` ("bf16" | "fp32") sends layers
    # whose channel counts are multiples of 64 through the tcgen05 conv instead ("fp32" = bf16x3 operand split,
    # <= 1e-5).
    tc_precision = None
    _same_extra_right = 0     # WNConv1d(padding='same') with an even kernel: one more zero row on the right

    def tc_layer(self) -> bool:
        """Whether inputs of >= TC_MIN_ROWS rows go to the tcgen05 conv."""
        return self.tc_precision is not None and not self._same_extra_right and \
            bool(_lib.lib().kvae_conv1d_tc_supported(self.in_channels, self.out_channels, self.kernel_size[0],
                                                     self.stride[0], self.dilation[0], int(self.transposed)))

    def out_len(self, T: int) -> int:
        """Output rows of the conv on an input of T rows."""
        K, s, d, p = self.kernel_size[0], self.stride[0], self.dilation[0], self.padding[0]
        T += self._same_extra_right
        return (T - 1) * s - 2 * p + d * (K - 1) + 1 if self.transposed else (T + 2 * p - d * (K - 1) - 1) // s + 1

    def keep(self, T: int) -> int:
        """Output rows the layer keeps of an input of T rows: all of them here; BigVGANFlowVAE's causal layers keep
        the first ones only."""
        return self.out_len(T)

    def engine(self, T: int, tc: bool, keep: int) -> int:
        """The engine the layer runs an input of T rows on (keeping ``keep`` output rows): 0 = CUDA cores fp32,
        1 = tcgen05 bf16, 2 = tcgen05 bf16x3.  The tensor cores take a ``tc_layer`` from TC_MIN_ROWS rows on, unless
        ``tc`` is False or the layer is a strided Conv1d whose output is truncated."""
        if not tc or T < TC_MIN_ROWS or not self.tc_layer():
            return 0
        if not self.transposed and self.stride[0] != 1 and keep != self.out_len(T):
            return 0
        return 1 if self.tc_precision == "bf16" else 2

    def packed_weight(self, engine: int):
        """(the folded weight packed by kvae_conv1d_pack for ``engine``: 0 = CUDA cores fp32, 1 = tcgen05 bf16,
        2 = tcgen05 bf16x3; the fp32 bias or None)"""
        L = _lib.lib()
        w = self.folded_weight()
        K = self.kernel_size[0]
        nb = L.kvae_conv1d_packed_bytes(self.in_channels, self.out_channels, K, engine)
        packed = torch.empty(nb, dtype=torch.uint8, device=w.device)
        _lib.check(L.kvae_conv1d_pack(w.data_ptr(), int(self.transposed), self.in_channels, self.out_channels, K,
                                      engine, packed.data_ptr(), nb, _lib.stream_ptr(w.device)))
        return packed, None if self.bias is None else self.bias.detach().float().contiguous()

    def conv_rows(self, x, packed, bias, engine: int, padding: int, o0: int, o1: int) -> torch.Tensor:
        """Output rows [o0, o1) of this layer's conv (padding ``padding``) of x [B, Cin, T] (fp32 / bf16, rows at any
        pitch) with the weights of ``packed_weight(engine)``: kvae_conv1d_win_fwd.  The tcgen05 engines emit whole
        stride groups of a transposed conv; rows outside [o0, o1) are sliced off."""
        L = _lib.lib()
        K, s, d = self.kernel_size[0], self.stride[0], self.dilation[0]
        B, Cin, T = x.shape
        if x.stride(2) != 1 or x.stride(0) != Cin * x.stride(1):
            x = x.contiguous()
        a0, a1 = o0, o1
        if engine and self.transposed:
            a0, a1 = o0 // s * s, -(-o1 // s) * s
        y = torch.empty((B, self.out_channels, a1 - a0), dtype=x.dtype, device=x.device)
        # a strided conv's input is staged rounded up to whole stride groups
        ns = L.kvae_conv1d_stream_scratch_bytes(B, Cin, T, 1 if self.transposed else s, engine)
        scratch = torch.empty(ns, dtype=torch.uint8, device=x.device) if ns else None
        _lib.check(L.kvae_conv1d_win_fwd(x.data_ptr(), x.stride(1), y.data_ptr(), a1 - a0, packed.data_ptr(),
                                         _lib.ptr(bias), int(self.transposed), B, Cin, self.out_channels, T, K, s, d,
                                         padding, a0, a1, _lib.dtype_code(x.dtype), engine, _lib.ptr(scratch), ns,
                                         _lib.stream_ptr(x.device)))
        return y if (a0, a1) == (o0, o1) else y[:, :, o0 - a0:o1 - a0]

    def conv_window(self, win, packed, bias, engine: int, x0: int, o0: int, o1: int, t_end: int) -> torch.Tensor:
        """Output rows [o0, o1) of this Conv1d (its own stride and padding) over a stream whose rows [x0, x0 + W) the
        window ``win`` [B, Cin, W] holds (fp32 / bf16, rows at any pitch; x0 a multiple of the stride), with the weights
        of ``packed_weight(engine)``: kvae_conv1d_stream_fwd.  Rows < 0 and, when t_end >= 0, rows >= t_end read as
        zero."""
        if self.transposed:
            raise ValueError("conv_window: a Conv1d only (transposed convs stream through conv_rows)")
        L = _lib.lib()
        K, s, d, p = self.kernel_size[0], self.stride[0], self.dilation[0], self.padding[0]
        B, Cin, W = win.shape
        if win.stride(2) != 1 or win.stride(0) != Cin * win.stride(1):
            win = win.contiguous()
        y = torch.empty((B, self.out_channels, o1 - o0), dtype=win.dtype, device=win.device)
        ns = L.kvae_conv1d_stream_scratch_bytes(B, Cin, W, s, engine)
        scratch = torch.empty(ns, dtype=torch.uint8, device=win.device) if ns else None
        _lib.check(L.kvae_conv1d_stream_fwd(win.data_ptr(), win.stride(1), x0, W, y.data_ptr(), o1 - o0, o0, o1, t_end,
                                            packed.data_ptr(), _lib.ptr(bias), B, Cin, self.out_channels, K, s, d, p,
                                            _lib.dtype_code(win.dtype), engine, _lib.ptr(scratch), ns,
                                            _lib.stream_ptr(win.device)))
        return y

    def _forward_impl(self, xin):
        """All output rows of the conv of xin (fp32 / bf16) on the CUDA cores (kvae_conv1d_fwd), in xin's dtype."""
        T_out = self.out_len(xin.shape[2])
        if T_out <= 0:
            raise RuntimeError("Kernel size can't be greater than actual input size")
        if self._same_extra_right:     # 'same' with an even kernel: one more zero on the right
            xin = torch.nn.functional.pad(xin, (0, self._same_extra_right))
        xin = xin.contiguous()
        w = self.folded_weight()
        bias = None if self.bias is None else self.bias.detach().float().contiguous()
        B, _, T = xin.shape
        K, s, d, p = self.kernel_size[0], self.stride[0], self.dilation[0], self.padding[0]
        L = _lib.lib()
        y = torch.empty((B, self.out_channels, T_out), dtype=xin.dtype, device=xin.device)
        nscratch = L.kvae_conv1d_scratch_bytes(self.in_channels, self.out_channels, K)
        scratch = torch.empty(nscratch, dtype=torch.uint8, device=xin.device)
        _lib.check(L.kvae_conv1d_fwd(xin.data_ptr(), y.data_ptr(), w.data_ptr(), _lib.ptr(bias), int(self.transposed),
                                     B, self.in_channels, self.out_channels, T, K, s, d, p,
                                     _lib.dtype_code(xin.dtype), scratch.data_ptr(), nscratch,
                                     _lib.stream_ptr(xin.device)))
        return y

    def extra_repr(self):
        return (f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, stride={self.stride}, "
                f"padding={self.padding}, dilation={self.dilation}, bias={self.bias is not None}")


class WNConv1d(_WNConvBase):
    """weight_norm(nn.Conv1d(...)): weight_v [Cout, Cin, K], weight_g [Cout, 1, 1] (norm per out-channel)."""
    transposed = False

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 bias=True, padding_mode="zeros", device=None, dtype=None):
        super().__init__()
        if groups != 1 or padding_mode != "zeros" or (isinstance(padding, str) and (padding != "same" or _single(stride) != 1)):
            raise NotImplementedError("kalle_audio_b200.WNConv1d: groups=1, zero padding with an integer amount or "
                                      "'same' at stride 1 only (the forms the Oobleck stack uses)")
        # padding='same' (the conv of DecoderBlock's use_nearest_upsample branch, autoencoders.py:90-95): torch pads
        # d(K-1) in total, the smaller half on the left
        self.same_padding = isinstance(padding, str)
        conv_padding = padding
        if self.same_padding:
            total = _single(dilation) * (_single(kernel_size) - 1)
            self._same_extra_right = total - 2 * (total // 2)
            padding = total // 2
        conv = nn.Conv1d(in_channels, out_channels, kernel_size, stride=stride, padding=conv_padding, dilation=dilation,
                         bias=bias, device=device, dtype=dtype)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size = (_single(kernel_size),)
        self.stride = (_single(stride),)
        self.padding = (_single(padding),)
        self.dilation = (_single(dilation),)
        self.groups = 1
        self._init_from(conv)


class WNConvTranspose1d(_WNConvBase):
    """weight_norm(nn.ConvTranspose1d(...)): weight_v [Cin, Cout, K], weight_g [Cin, 1, 1] -- the norm is
    taken per *in*-channel because dim 0 of a transposed-conv weight is Cin (SURVEY.md H4)."""
    transposed = True

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, output_padding=0, groups=1,
                 bias=True, dilation=1, padding_mode="zeros", device=None, dtype=None):
        super().__init__()
        if groups != 1 or padding_mode != "zeros" or _single(output_padding) != 0 or _single(dilation) != 1:
            raise NotImplementedError("kalle_audio_b200.WNConvTranspose1d: groups=1, output_padding=0, dilation=1 only")
        conv = nn.ConvTranspose1d(in_channels, out_channels, kernel_size, stride=stride, padding=padding, bias=bias,
                                  device=device, dtype=dtype)
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size = (_single(kernel_size),)
        self.stride = (_single(stride),)
        self.padding = (_single(padding),)
        self.dilation = (1,)
        self.output_padding = (0,)
        self.groups = 1
        self._init_from(conv)


def nearest_upsample_conv_taps(w: torch.Tensor, stride: int) -> torch.Tensor:
    """Folded taps of ``Upsample(scale_factor=stride, mode='nearest')`` followed by ``Conv1d(k = 2*stride, padding='same')``
    (DecoderBlock's use_nearest_upsample branch, autoencoders.py:87-96) as ONE transposed convolution: ``w`` [Cout, Cin,
    2s] -> ConvTranspose1d weight [Cin, Cout, 3s - 1] for stride s, padding s, output_padding 1, with
    ``w'[k'] = sum_{k = 2s-1-k'}^{3s-2-k'} w[k]`` (k clipped to 0 .. 2s-1): every group of s upsampled positions that
    reads the same input sample contributes the sum of the taps that land on it."""
    Cout, Cin, K = w.shape
    s = int(stride)
    if K != 2 * s:
        raise ValueError("the nearest-upsample conv has kernel_size == 2 * stride")
    wp = w.new_zeros(Cin, Cout, 3 * s - 1)
    for kp in range(3 * s - 1):
        lo, hi = max(0, 2 * s - 1 - kp), min(2 * s - 1, 3 * s - 2 - kp)
        wp[:, :, kp] = w[:, :, lo:hi + 1].sum(-1).t()
    return wp.contiguous()


class NearestUpsampleConv(nn.Sequential):
    """``nn.Sequential(nn.Upsample(scale_factor=stride, mode="nearest"), WNConv1d(k=2*stride, padding='same',
    bias=False))`` exactly as the reference builds it (same state_dict keys ``0`` / ``1.weight_g`` / ``1.weight_v``).
    Stand-alone it chains the two modules; inside an OobleckDecoder plan the pair runs as one tcgen05 transposed conv."""

    def __init__(self, in_channels, out_channels, stride):
        super().__init__(nn.Upsample(scale_factor=stride, mode="nearest"),
                         WNConv1d(in_channels=in_channels, out_channels=out_channels, kernel_size=2 * stride, stride=1,
                                  bias=False, padding="same"))
        self.upsample_stride = int(stride)
        self[1]._upsample_stride = int(stride)      # the plan folds this conv's weight into transposed-conv taps
