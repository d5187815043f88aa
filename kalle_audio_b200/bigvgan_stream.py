"""Stateful streaming decode for ``BigVGANFlowVAE.inference_from_latents`` (flows.py:498-529).

A speech LM emits one latent frame per step; ``BigVGANStreamingDecoder.push`` turns each batch of frames into the
waveform samples that became final, and ``flush`` returns the rest.  Every op of the decoder keeps the tail of its own
input between calls and runs in *valid form* on the window ``[carry | new rows]``, so each output row is computed
exactly once, and ``torch.cat(pushes + [flush])`` equals the whole-utterance decode bit for bit:

  * convolutions (``conv_pre``, the AMP-block convs, ``conv_post``): the window starts with the left zero padding and
    the stream end appends the right zero padding; the conv then runs with padding 0.  Per output the kernels sum the
    same taps in the same order as the padded whole-row call (a zero row contributes ``fma(0, w, acc) == acc``).
  * transposed convs (``ups``): the window holds the input rows the next outputs read, the kernel runs with the layer's
    own padding and the needed output rows are kept (a causal layer skips the first ``stride`` rows of its window).
  * ``Activation1d``: ``kvae_aa_act_win_fwd``, the whole-row kernel addressed in absolute stream rows, so its
    replicate padding happens only at the true stream start and end.
  * residual adds / the AMP average / tanh / the Gaussian sample: the library's elementwise kernels on rows that both
    operands have.

The op list comes from one description of the decoder (``_program``) that two interpreters read: the integer one
behind ``bigvgan_stream_geometry`` (rows available per op, lookahead) and the tensor one behind the decoder.

Pushes whose (size, start-up phase) was seen before replay one ``torch.cuda.CUDAGraph``; the op state lives in static
buffers per phase, so a constant-hop stream in steady state is one graph launch per push.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib
from .bigvgan import BigVGANFlowVAE, _axpby, _k, _unary

_AA_HALO = 5            # Activation1d: y[t] reads x[t - 5 .. t + 5] (12-tap x2 filters, bigvgan.cuh)


# ------------------------------------------------------------------------------------------------ the op list
def _program(h) -> Tuple[List[tuple], str]:
    """The inference path as a list of ops over named streams (flows.py:506-527 in execution order).

    ("conv", module, src, dst)  ("convT", module, src, dst)  ("act", module, src, dst)
    ("axpby", a, b, dst, alpha, beta)  ("tanh", src, dst).  Module paths are ``BigVGANFlowVAE`` attribute paths."""
    ops: List[tuple] = [("conv", "conv_pre", "z", "x0")]
    nk = len(h["resblock_kernel_sizes"])
    x = "x0"
    for i in range(len(h["upsample_rates"])):
        up = f"u{i}"
        ops.append(("convT", f"ups.{i}.0", x, up))
        xs = None
        for j, dil in enumerate(h["resblock_dilation_sizes"]):
            rb, cur = f"resblocks.{i * nk + j}", up
            if h["resblock"] == "1":
                for q in range(len(dil)):
                    t = f"{rb}.{q}"
                    ops += [("act", f"{rb}.activations.{2 * q}", cur, t + "a1"),
                            ("conv", f"{rb}.convs1.{q}", t + "a1", t + "c1"),
                            ("act", f"{rb}.activations.{2 * q + 1}", t + "c1", t + "a2"),
                            ("conv", f"{rb}.convs2.{q}", t + "a2", t + "c2"),
                            ("axpby", t + "c2", cur, t + "r", 1.0, 1.0)]
                    cur = t + "r"
            else:
                for q in range(len(dil)):
                    t = f"{rb}.{q}"
                    ops += [("act", f"{rb}.activations.{q}", cur, t + "a"),
                            ("conv", f"{rb}.convs.{q}", t + "a", t + "c"),
                            ("axpby", t + "c", cur, t + "r", 1.0, 1.0)]
                    cur = t + "r"
            if xs is None:
                xs = cur
            else:
                ops.append(("axpby", xs, cur, f"s{i}.{j}", 1.0, 1.0))
                xs = f"s{i}.{j}"
        x = f"x{i + 1}"
        ops.append(("axpby", xs, xs, x, 1.0 / nk, 0.0))
    ops += [("act", "activation_post", x, "ap"), ("conv", "conv_post", "ap", "cp"), ("tanh", "cp", "wav")]
    return ops, "wav"


def _conv_shape(h, path: str) -> Tuple[int, int, int, bool]:
    """(kernel, dilation, stride, causal) of a conv / transposed conv of the program, from ``h`` alone."""
    causal = bool(h["causal"])
    if path == "conv_pre":
        return 7, 1, 1, False
    if path == "conv_post":
        return 7, 1, 1, causal
    parts = path.split(".")
    if parts[0] == "ups":
        i = int(parts[1])
        return int(h["upsample_kernel_sizes"][i]), 1, int(h["upsample_rates"][i]), causal
    nk = len(h["resblock_kernel_sizes"])
    j = int(parts[1]) % nk
    k = int(h["resblock_kernel_sizes"][j])
    d = int(h["resblock_dilation_sizes"][j][int(parts[3])]) if parts[2] in ("convs1", "convs") else 1
    return k, d, 1, causal


class _Geom:
    """Integer form of one op: how many output rows are final once ``R`` input rows have arrived."""

    def __init__(self, kind: str, K: int = 1, d: int = 1, s: int = 1, causal: bool = False):
        self.kind, self.K, self.d, self.s, self.causal = kind, K, d, s, causal
        if kind == "conv":
            self.span = d * (K - 1)
            self.pl = self.span if causal else d * (K - 1) // 2        # left zero rows (flows.py:607-608)
            self.pr = 0 if causal else self.pl                           # right zero rows at the stream end
        elif kind == "convT":
            self.span = K - 1
            self.p = 0 if causal else (K - s) // 2                       # flows.py:336-391
        elif kind == "act":
            self.span = 2 * _AA_HALO

    def total(self, R: int) -> int:
        """Output rows of the whole-utterance op on R input rows."""
        if self.kind == "conv":
            return R + self.pl + self.pr - self.span
        if self.kind == "convT":
            return R * self.s if self.causal else (R - 1) * self.s - 2 * self.p + self.K
        return R

    def avail(self, R: int, end: bool) -> int:
        if end:
            return max(0, self.total(R)) if R > 0 else 0
        if self.kind == "conv":
            return max(0, R + self.pl - self.span)
        if self.kind == "convT":
            return max(0, R * self.s - self.p)
        if self.kind == "act":
            return max(0, R - _AA_HALO)
        return R

    def lookahead(self) -> int:
        """Rows after an output's own position that it reads (in output rows)."""
        if self.kind == "conv":
            return self.span - self.pl
        if self.kind == "convT":
            return self.p
        return _AA_HALO if self.kind == "act" else 0


def _geom_of(h, op) -> _Geom:
    if op[0] in ("conv", "convT"):
        K, d, s, causal = _conv_shape(h, op[1])
        return _Geom(op[0], K, d, s, causal)
    return _Geom(op[0])


def bigvgan_stream_geometry(h) -> Dict[str, object]:
    """Pure host arithmetic over the layer definitions: per op (execution order) its kind, module, row rate (input
    rows per latent frame), rows read per output, span, dilation, stride and lookahead (output rows), plus the
    decoder's total ``lookahead`` in samples: after n frames, ``max(0, n * ratio - lookahead)`` samples are final."""
    h = dict(h)
    ops, out = _program(h)
    ratio = int(math.prod(h["upsample_rates"]))
    rate = {"z": 1}
    rows = []
    n = 64 + 4 * ratio                       # far beyond any start-up effect
    R = {"z": n}
    for op in ops:
        if op[0] == "tanh":
            R[op[2]], rate[op[2]] = R[op[1]], rate[op[1]]
            continue
        if op[0] == "axpby":
            R[op[3]], rate[op[3]] = min(R[op[1]], R[op[2]]), rate[op[1]]
            continue
        g = _geom_of(h, op)
        r_in = rate[op[2]]
        R[op[3]] = g.avail(R[op[2]], False)
        rate[op[3]] = r_in * g.s
        rows.append({"op": op[0], "module": op[1], "rate": r_in, "rows_read": -(-(g.span + 1) // g.s),
                     "span": g.span, "dilation": g.d, "stride": g.s, "lookahead": g.lookahead()})
    return {"ops": rows, "ratio": ratio, "lookahead": n * ratio - R[out]}


# ------------------------------------------------------------------------------------------------ the decoder
def _module(model, path: str):
    m = model
    for p in path.split("."):
        m = m[int(p)] if p.isdigit() else getattr(m, p)
    return m


def _cat(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    if b.shape[2] == 0:
        return a
    if a.shape[2] == 0:
        return b
    return torch.cat([a, b], dim=2)


def _rows(t: torch.Tensor, lo: int, hi: Optional[int] = None) -> torch.Tensor:
    return t[:, :, lo:hi] if (lo, hi) != (0, None) else t


class BigVGANStreamingDecoder:
    """Feed latent frames as they arrive; get waveform back as soon as it is final.

        sd = BigVGANStreamingDecoder(model)          # model: BigVGANFlowVAE on a CUDA device
        for z in frames:                             # z: [B, D, n] (or [B, 2 D, n] with do_sample), any n >= 0
            wav = sd.push(z)                         # [B, 1, m]: the samples that became final
        wav = sd.flush()                             # the rest; the next push starts a new stream

    ``torch.cat`` of everything returned equals ``model.inference_from_latents(torch.cat(frames, -1), do_sample,
    noise=torch.cat(noises, -1))`` with ``torch.equal``, output length included.  ``lookahead`` samples of the pushed
    frames are held back until the frames after them arrive.

    Engines are fixed per layer when a stream starts: a conv runs on the tensor cores when the model's precision sends
    it there (``set_precision("fp32" | "bf16")`` and channel counts the tcgen05 kernel takes), whatever the window
    length.  ``inference_from_latents`` does so only for inputs of >= 64 rows, so with tensor-core precision the
    equality holds for utterances of >= 64 frames (every eligible layer then has >= 64 rows in the whole decode too).

    With ``do_sample`` and no ``noise``, noise is drawn per push with ``torch.randn``: the samples do not replay the
    RNG stream of one whole ``inference_from_latents`` call.  Pass ``noise`` for a reproducible stream."""

    def __init__(self, model: BigVGANFlowVAE, max_frames: int = 16, use_cuda_graphs: bool = True,
                 do_sample: bool = False):
        if not isinstance(model, BigVGANFlowVAE):
            raise TypeError("BigVGANStreamingDecoder wraps a kalle_audio_b200.BigVGANFlowVAE")
        if max_frames < 1:
            raise ValueError("max_frames must be >= 1")
        self.model = model
        self.max_frames = int(max_frames)
        self.use_cuda_graphs = bool(use_cuda_graphs)
        h = model.h
        self.do_sample = bool(do_sample)
        self.sample = bool(h.use_vae and do_sample)
        self.in_channels = h.latent_dim * (2 if self.sample else 1)
        self.ratio = int(math.prod(h.upsample_rates))
        self._ops, self._out = _program(h)
        self._geoms = [_geom_of(h, op) for op in self._ops]
        self.lookahead = int(bigvgan_stream_geometry(h)["lookahead"])
        self._convs = sorted({op[1] for op in self._ops if op[0] in ("conv", "convT")})
        self._params = [p for name in ("conv_pre", "ups", "resblocks", "activation_post", "conv_post")
                        for p in getattr(model, name).parameters()]
        self.graph_captures = 0         # CUDA graphs captured by this decoder
        self.graph_replays = 0          # pushes served by replaying one
        self._graphs: Dict[tuple, dict] = {}
        self._static: Dict[tuple, List[torch.Tensor]] = {}
        self._pool = None
        self._graph_key = None
        self.reset()

    # ------------------------------------------------------------------ stream state
    def reset(self) -> None:
        """Drops the stream; the next push starts a new one (captured graphs stay while the weights do)."""
        self._B = None
        self._ints: Optional[List[tuple]] = None
        self._tens: Optional[List[List[torch.Tensor]]] = None
        self._in_static = False
        self._weights = None

    def _weights_key(self) -> tuple:
        key = [(p.data_ptr(), p._version) for p in self._params]
        key += [_module(self.model, c).tc_precision for c in self._convs]
        return tuple(key)

    def _begin(self, z: torch.Tensor) -> None:
        B, dev, dt = z.shape[0], z.device, z.dtype
        key = self._weights_key()
        L = _lib.lib()
        if (key, B, dt, dev) != self._graph_key:
            # engines fixed and weights packed once per weight version; the captured graphs hold the packed weights'
            # addresses, so both are replaced together
            self._engine, self._packed = {}, {}
            for c in self._convs:
                m = _module(self.model, c)
                tc = m.tc_precision is not None and not getattr(m, "_same_extra_right", 0) and \
                    L.kvae_conv1d_tc_supported(m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0],
                                               m.dilation[0], int(m.transposed))
                self._engine[c] = m.tc_precision if tc else None
                code = {None: 0, "bf16": 1, "fp32": 2}[self._engine[c]]
                K = m.kernel_size[0]
                nb = L.kvae_conv1d_packed_bytes(m.in_channels, m.out_channels, K, code)
                packed = torch.empty(nb, dtype=torch.uint8, device=dev)
                _lib.check(L.kvae_conv1d_pack(m.folded_weight().data_ptr(), int(m.transposed), m.in_channels,
                                              m.out_channels, K, code, packed.data_ptr(), nb, _lib.stream_ptr(dev)))
                bias = None if m.bias is None else m.bias.detach().float().contiguous().clone()
                self._packed[c] = (packed, code, bias)
            self._graphs, self._static, self._graph_key = {}, {}, (key, B, dt, dev)
        self._weights = key
        self._B, self._dtype, self._dev = B, dt, dev
        self._ints, self._tens = [], []
        for op, g in zip(self._ops, self._geoms):
            if op[0] == "conv":
                ch = _module(self.model, op[1]).in_channels
                self._ints.append((0, 0))                               # (rows in, rows out)
                self._tens.append([torch.zeros((B, ch, g.pl), dtype=dt, device=dev)])
            elif op[0] == "convT":
                ch = _module(self.model, op[1]).in_channels
                self._ints.append((0, 0, 0))                            # (rows in, first carried row, rows out)
                self._tens.append([torch.zeros((B, ch, 0), dtype=dt, device=dev)])
            elif op[0] == "act":
                ch = _module(self.model, op[1]).act.alpha.numel()
                self._ints.append((0, 0))
                self._tens.append([torch.zeros((B, ch, 0), dtype=dt, device=dev)])
            elif op[0] == "axpby" and op[1] != op[2]:
                self._ints.append((0,))
                self._tens.append([None, None])                         # pending rows of each operand
            else:
                self._ints.append(())
                self._tens.append([])
        self._in_static = False

    # ------------------------------------------------------------------ one step of every op (functional)
    def _conv_call(self, path: str, x: torch.Tensor, padding: int, o0: int, o1: int) -> torch.Tensor:
        """Output rows [o0, o1) of the layer's conv (padding ``padding``) of the window ``x`` (pitched rows), with the
        weights packed at stream start."""
        m = _module(self.model, path)
        L = _lib.lib()
        packed, code, bias = self._packed[path]
        K, s, d = m.kernel_size[0], m.stride[0], m.dilation[0]
        B, Cin, T = x.shape
        if x.stride(2) != 1 or x.stride(0) != Cin * x.stride(1):
            x = x.contiguous()
        a0, a1 = o0, o1
        if code and m.transposed:             # the tcgen05 engine emits whole stride groups
            a0, a1 = o0 // s * s, -(-o1 // s) * s
        y = torch.empty((B, m.out_channels, a1 - a0), dtype=x.dtype, device=x.device)
        ns = L.kvae_conv1d_win_scratch_bytes(B, Cin, T, code)
        scratch = torch.empty(ns, dtype=torch.uint8, device=x.device) if ns else None
        _lib.check(L.kvae_conv1d_win_fwd(x.data_ptr(), x.stride(1), y.data_ptr(), a1 - a0, packed.data_ptr(),
                                         _lib.ptr(bias), int(m.transposed), B, Cin, m.out_channels, T, K, s, d, padding,
                                         a0, a1, _lib.dtype_code(x.dtype), code, _lib.ptr(scratch), ns,
                                         _lib.stream_ptr(x.device)))
        return y if (a0, a1) == (o0, o1) else y[:, :, o0 - a0:o1 - a0]

    def _act_call(self, path: str, win: torch.Tensor, x0: int, o0: int, o1: int, t_end: int) -> torch.Tensor:
        act = _module(self.model, path)
        B, C, W = win.shape
        y = torch.empty((B, C, o1 - o0), dtype=win.dtype, device=win.device)
        if win.stride(2) != 1 or win.stride(0) != C * win.stride(1):
            win = win.contiguous()
        beta = getattr(act.act, "beta", None)
        fu = act.upsample.filter.detach().float().reshape(-1).contiguous()
        fd = act.downsample.lowpass.filter.detach().float().reshape(-1).contiguous()
        alpha = act.act.alpha.detach().float().contiguous()
        beta = None if beta is None else beta.detach().float().contiguous()
        _lib.check(_lib.lib().kvae_aa_act_win_fwd(win.data_ptr(), win.stride(1), x0, W, y.data_ptr(), o1 - o0, o0, o1,
                                                  t_end, alpha.data_ptr(), _lib.ptr(beta), int(act.act.alpha_logscale),
                                                  fu.data_ptr(), fd.data_ptr(), B, C, _lib.dtype_code(win.dtype),
                                                  _lib.stream_ptr(win.device)))
        return y

    def _step(self, ints, tens, z: torch.Tensor, end: bool):
        """Runs every op once on its new input rows.  Pure: returns (waveform rows, new ints, new tensors)."""
        vals = {"z": z}
        new_ints, new_tens = [], []
        for op, g, st, ts in zip(self._ops, self._geoms, ints, tens):
            kind = op[0]
            if kind == "conv":
                R, e = st
                x = vals[op[2]]
                win = _cat(ts[0], x)
                R += x.shape[2]
                if end and g.pr:
                    win = _cat(win, win.new_zeros((win.shape[0], win.shape[1], g.pr)))
                n_out = win.shape[2] - g.span
                if n_out > 0:
                    y = self._conv_call(op[1], win, 0, 0, n_out)
                    e += n_out
                    win = _rows(win, n_out)
                else:
                    y = win.new_zeros((win.shape[0], _module(self.model, op[1]).out_channels, 0))
                vals[op[3]] = y
                new_ints.append((R, e))
                new_tens.append([win])
            elif kind == "convT":
                R, j0, e = st
                x = vals[op[2]]
                win = _cat(ts[0], x)
                R += x.shape[2]
                o_max = g.avail(R, end)
                m = _module(self.model, op[1])
                if o_max > e:
                    # only the rows not emitted yet: a causal layer skips the first `stride` rows of its window
                    y = self._conv_call(op[1], win, g.p, e - g.s * j0, o_max - g.s * j0)
                    e = o_max
                else:
                    y = win.new_zeros((win.shape[0], m.out_channels, 0))
                j1 = max(0, -(-(e + g.p - g.K + 1) // g.s))
                vals[op[3]] = y
                new_ints.append((R, j1, e))
                new_tens.append([_rows(win, j1 - j0)])
            elif kind == "act":
                R, e = st
                x = vals[op[2]]
                a = max(0, e - _AA_HALO)
                win = _cat(ts[0], x)
                R += x.shape[2]
                o_max = g.avail(R, end)
                if o_max > e:
                    # a window away from the stream start (its outputs at o >= 5) is addressed window-relative
                    # (include/kvae.h), so a captured graph's kernel arguments hold for every later push of a phase
                    off = a
                    y = self._act_call(op[1], win, a - off, e - off, o_max - off, R - off if end else -1)
                    e = o_max
                else:
                    y = win.new_zeros((win.shape[0], win.shape[1], 0))
                a1 = max(0, e - _AA_HALO)
                vals[op[3]] = y
                new_ints.append((R, e))
                new_tens.append([_rows(win, a1 - a)])
            elif kind == "axpby":
                a_in, b_in = vals[op[1]], vals[op[2]]
                if op[1] == op[2]:                                      # the AMP average: stateless
                    vals[op[3]] = _axpby(a_in, b_in, op[4], op[5]) if a_in.shape[2] else a_in
                    new_ints.append(())
                    new_tens.append([])
                    continue
                pa = a_in if ts[0] is None else _cat(ts[0], a_in)
                pb = b_in if ts[1] is None else _cat(ts[1], b_in)
                n = min(pa.shape[2], pb.shape[2])
                if n:
                    y = _axpby(_rows(pa, 0, n), _rows(pb, 0, n), op[4], op[5])
                else:
                    y = pa[:, :, :0]
                vals[op[3]] = y
                new_ints.append((st[0] + n,))
                new_tens.append([_rows(pa, n), _rows(pb, n)])
            else:                                                       # tanh
                x = vals[op[1]]
                vals[op[2]] = _unary(x, 1) if x.shape[2] else x
                new_ints.append(())
                new_tens.append([])
        return vals[self._out], new_ints, new_tens

    def _head(self, z: torch.Tensor, noise: Optional[torch.Tensor]) -> torch.Tensor:
        """The Gaussian sample of the do_sample branch (flows.py:500-501) on the pushed frames."""
        if not self.sample:
            return _k(z)
        D = self.model.h.latent_dim
        m, lg = _k(z[:, :D]), _k(z[:, D:])
        nz = _k(noise).to(m.dtype)
        out = torch.empty_like(m)
        if m.numel():
            _lib.check(_lib.lib().kvae_gauss_sample(m.data_ptr(), lg.to(m.dtype).data_ptr(), nz.data_ptr(),
                                                    out.data_ptr(), m.numel(), _lib.dtype_code(m.dtype),
                                                    _lib.stream_ptr(z.device)))
        return out

    # ------------------------------------------------------------------ graphs
    def _sig(self) -> tuple:
        return tuple(tuple(t.shape[2] if t is not None else -1 for t in ts) for ts in self._tens)

    def _static_for(self, tens: List[List[torch.Tensor]]) -> List[List[torch.Tensor]]:
        """The static buffers of the phase whose state has the shapes of ``tens`` (allocated on first use)."""
        sig = tuple(tuple(t.shape[2] if t is not None else -1 for t in ts) for ts in tens)
        buf = self._static.get(sig)
        if buf is None:
            buf = [[None if t is None else torch.empty_like(t, memory_format=torch.contiguous_format) for t in ts]
                   for ts in tens]
            self._static[sig] = buf
        return buf

    def _phase(self) -> tuple:
        """What a step depends on besides the carried row counts: the position of the next output inside the window
        and whether the window still touches the stream start."""
        ph = []
        for op, g, st in zip(self._ops, self._geoms, self._ints):
            if op[0] == "convT":
                ph.append((st[2] - g.s * st[1], st[1] == 0))
            elif op[0] == "act":
                a = max(0, st[1] - _AA_HALO)
                ph.append((st[1] - a, a == 0))
        return tuple(ph)

    def _run_graph(self, z: torch.Tensor, noise: Optional[torch.Tensor]) -> torch.Tensor:
        n = z.shape[2]
        key = (n, self._phase(), self._sig())
        G = self._graphs.get(key)
        if G is None:
            # eager run (also warms every kernel), then capture the same step from static copies of the input state
            out, ints1, tens1 = self._step(self._ints, self._tens, self._head(z, noise), False)
            src = self._static_for(self._tens)
            if not self._in_static:
                for dst_l, src_l in zip(src, self._tens):
                    for dst, t in zip(dst_l, src_l):
                        if dst is not None:
                            dst.copy_(t)
            dst_state = self._static_for(tens1)
            zin = torch.empty_like(z)
            nin = None if noise is None else torch.empty_like(noise)
            if self._pool is None:
                self._pool = torch.cuda.graph_pool_handle()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=self._pool):
                gout, _, gtens = self._step(list(self._ints), src, self._head(zin, nin), False)
                static_ptrs = {t.untyped_storage().data_ptr() for ts in src for t in ts if t is not None}
                moved = []
                for dst_l, src_l in zip(dst_state, gtens):
                    for dst, t in zip(dst_l, src_l):
                        if dst is None or t is dst:
                            continue
                        if t.untyped_storage().data_ptr() in static_ptrs:
                            t = t.clone()                      # never copy a static buffer onto another in place
                        moved.append((dst, t))
                for dst, t in moved:
                    dst.copy_(t)
            dints = [tuple(b - a for a, b in zip(i0, i1)) for i0, i1 in zip(self._ints, ints1)]
            self._graphs[key] = {"graph": g, "z": zin, "noise": nin, "out": gout, "dints": dints, "state": dst_state}
            self.graph_captures += 1
            self._ints, self._tens, self._in_static = ints1, tens1, False
            return out
        if not self._in_static:
            src = self._static[key[2]]
            for dst_l, src_l in zip(src, self._tens):
                for dst, t in zip(dst_l, src_l):
                    if dst is not None and dst is not t:
                        dst.copy_(t)
        G["z"].copy_(z)
        if G["noise"] is not None:
            G["noise"].copy_(noise)
        G["graph"].replay()
        self.graph_replays += 1
        self._ints = [tuple(a + d for a, d in zip(i0, di)) for i0, di in zip(self._ints, G["dints"])]
        self._tens, self._in_static = G["state"], True
        return G["out"].clone()

    # ------------------------------------------------------------------ public surface
    def _check(self, z: torch.Tensor, noise: Optional[torch.Tensor]) -> None:
        _lib.require_cuda(z, "BigVGANStreamingDecoder.push")
        if z.dim() != 3 or z.shape[1] != self.in_channels:
            raise ValueError(f"expected latents [B, {self.in_channels}, n], got {tuple(z.shape)}")
        if z.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("latents must be float32 or bfloat16")
        if self._B is not None:
            if z.shape[0] != self._B:
                raise ValueError("batch size changed inside a stream")
            if z.dtype != self._dtype or z.device != self._dev:
                raise ValueError("dtype or device changed inside a stream")
            if self._weights_key() != self._weights:
                raise RuntimeError("BigVGANStreamingDecoder: the model's weights or precision changed inside a stream; "
                                   "call reset() to start a new stream with the new weights")
        if noise is not None:
            if not self.sample:
                raise ValueError("noise is only used with do_sample on a use_vae model")
            _lib.require_cuda(noise, "BigVGANStreamingDecoder.push")
            if tuple(noise.shape) != (z.shape[0], self.model.h.latent_dim, z.shape[2]):
                raise ValueError("noise must be [B, D, n] like the mean half of the latents")

    @torch.no_grad()
    def push(self, latents: torch.Tensor, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """latents [B, D, n] (or [B, 2 D, n] with do_sample), n >= 0 -> the [B, 1, m] samples that became final."""
        self._check(latents, noise)
        if self._B is None:
            self._begin(latents)
        if self.sample and noise is None:
            noise = torch.randn((latents.shape[0], self.model.h.latent_dim, latents.shape[2]), dtype=latents.dtype,
                                device=latents.device)
        pieces = []
        for i in range(0, latents.shape[2], self.max_frames):
            z = latents[:, :, i:i + self.max_frames]
            nz = None if noise is None else noise[:, :, i:i + self.max_frames].contiguous()
            if self.use_cuda_graphs:
                pieces.append(self._run_graph(z.contiguous(), nz))
            else:
                out, self._ints, self._tens = self._step(self._ints, self._tens, self._head(z, nz), False)
                pieces.append(out)
        if not pieces:
            return latents.new_zeros((latents.shape[0], 1, 0))
        return pieces[0] if len(pieces) == 1 else torch.cat(pieces, dim=2)

    @torch.no_grad()
    def flush(self) -> torch.Tensor:
        """The samples still held back (right edge as in the whole decode); then resets the stream."""
        if self._B is None:
            raise ValueError("nothing was pushed")
        if self._weights_key() != self._weights:
            raise RuntimeError("BigVGANStreamingDecoder: the model's weights or precision changed inside a stream; "
                               "call reset() to start a new stream with the new weights")
        D = self.in_channels
        z = torch.zeros((self._B, D, 0), dtype=self._dtype, device=self._dev)
        nz = None if not self.sample else torch.zeros((self._B, self.model.h.latent_dim, 0), dtype=self._dtype,
                                                      device=self._dev)
        out, _, _ = self._step(self._ints, self._tens, self._head(z, nz), True)
        self.reset()
        return out
