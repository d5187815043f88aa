"""Stateful streaming decode and encode for ``BigVGANFlowVAE.inference_from_latents`` (flows.py:498-529) and
``extract_latents`` (:494-496).

A speech LM emits one latent frame per step; ``BigVGANStreamingDecoder.push`` turns each batch of frames into the
waveform samples that became final, and ``flush`` returns the rest.  ``BigVGANStreamingEncoder`` does the same from
audio to latent frames.  Both are one interpreter of an op list, the decoder's (``bigvgan._program``) or the
encoder's (``bigvgan._encoder_program``).  Every op keeps the tail of its own input between calls and runs in *valid
form* on the window ``[carry | new rows]``, so each output row is computed exactly once, and
``torch.cat(pushes + [flush])`` equals the whole call bit for bit:

  * convolutions (any stride): the carry holds whole stride groups from a stream row = 0 (mod stride) on, and
    ``kvae_conv1d_stream_fwd`` runs on ``[carry | new rows]`` with the layer's own padding.  Rows below 0 read as zero,
    and so do rows at or past the stream end, which is given only at ``flush``.  Per output the kernels sum the same
    taps in the same order as the whole-layer call.
  * transposed convs (``ups``): the window holds the input rows the next outputs read, the kernel runs with the layer's
    own padding and the needed output rows are kept (a causal layer skips the first ``stride`` rows of its window).
  * ``Activation1d``: ``kvae_aa_act_win_fwd``, the whole-row kernel addressed in absolute stream rows, so its
    replicate padding happens only at the true stream start and end.
  * LeakyReLU / tanh / the AMP average: stateless on the new rows; residual adds: the library's elementwise kernel on
    the rows that both operands have; the decoder's Gaussian sample: on the pushed frames.

The same op lists are read by the integer interpreters behind ``bigvgan_stream_geometry`` /
``bigvgan_encode_stream_geometry`` (rows available per op, lookahead) and by the ragged whole-clip calls of
``BigVGANFlowVAE``.

Pushes whose (size, start-up phase) was seen before replay one ``torch.cuda.CUDAGraph``; the op state lives in static
buffers per phase, so a constant-hop stream in steady state is one graph launch per push.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch

from . import _lib
from .bigvgan import BigVGANFlowVAE, _axpby, _encoder_program, _gauss_sample, _k, _lengths, _module, _program, _unary


def bigvgan_stream_geometry(h) -> Dict[str, object]:
    """Pure host arithmetic over the layer definitions: per op (execution order) its kind, module, row rate (input
    rows per latent frame), rows read per output, span, dilation, stride and lookahead (output rows), plus the
    decoder's total ``lookahead`` in samples: after n frames, ``max(0, n * ratio - lookahead)`` samples are final."""
    h = dict(h)
    ops, out = _program(h)
    ratio = int(math.prod(h["upsample_rates"]))
    rate = {"z": 1}
    rows = []
    for op in ops:
        g, r_in = op.geom, rate[op.srcs[0]]
        rate[op.dst] = r_in * (g.s if g else 1)
        if g:
            rows.append({"op": op.kind, "module": op.module, "rate": r_in, "rows_read": -(-(g.span + 1) // g.s),
                         "span": g.span, "dilation": g.d, "stride": g.s, "lookahead": g.lookahead()})
    n = 64 + 4 * ratio                       # far beyond any start-up effect
    return {"ops": rows, "ratio": ratio, "lookahead": n * ratio - _lengths(h, False, n, end=False)[out]}


def bigvgan_encode_stream_geometry(h) -> Dict[str, object]:
    """Pure host arithmetic over the encoder's layer definitions: per conv (execution order) its module, row rate (input
    samples per input row), span, dilation, stride, padding and lookahead, plus the encoder's ``lookahead`` and
    ``context`` in samples: after n samples, ``max(0, (n - lookahead) // ratio)`` frames are final, and frame t reads
    the samples ``t * ratio - context .. t * ratio + ratio - 1 + lookahead``."""
    h = dict(h)
    ops, out = _encoder_program(h)
    ratio = int(math.prod(h["downsample_rates"]))
    rate = {"x": 1}
    first = {"x": 0}                          # row o of a stream reads the samples from o * rate + first on
    rows = []
    bound = 0
    for op in ops:
        g, r_in = op.geom, rate[op.srcs[0]]
        if g is None:
            rate[op.dst], first[op.dst] = r_in, min(first[s] for s in op.srcs)
            continue
        rate[op.dst] = r_in * g.s
        first[op.dst] = first[op.srcs[0]] - g.reach() * r_in
        bound += g.span * r_in
        rows.append({"module": op.module, "rate": r_in, "span": g.span, "dilation": g.d, "stride": g.s,
                     "padding": g.pl, "lookahead": g.lookahead()})
    # the fewest samples after which F frames are final (the stream's integer interpreter) is F * ratio + lookahead
    F = bound // ratio + 2
    lo, hi = 0, F * ratio + bound
    while lo < hi:
        mid = (lo + hi) // 2
        if _lengths(h, True, mid, end=False)[out] >= F:
            hi = mid
        else:
            lo = mid + 1
    return {"ops": rows, "ratio": ratio, "lookahead": lo - F * ratio, "context": -first[out]}


def _cat(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    if b.shape[2] == 0:
        return a
    if a.shape[2] == 0:
        return b
    return torch.cat([a, b], dim=2)


def _rows(t: torch.Tensor, lo: int, hi: Optional[int] = None) -> torch.Tensor:
    return t[:, :, lo:hi] if (lo, hi) != (0, None) else t


class _OpStream:
    """The stream interpreter of the decoder's or the encoder's op list: per-op state, one step per op kind, engines
    fixed and weights packed per weight version, the check that the weights did not change inside a stream, and the
    CUDA graphs (static state buffers per phase, capture, replay).  ``push`` takes [B, ``in_channels``, n] and returns
    [B, ``out_channels``, m].  A subclass sets ``in_channels``, ``out_channels`` and ``_noun`` (what it is fed, for the
    error messages) and may override ``_head``, the step on the pushed rows before the first op."""

    _noun = ""

    def __init__(self, model: BigVGANFlowVAE, encoder: bool, use_cuda_graphs: bool):
        if not isinstance(model, BigVGANFlowVAE):
            raise TypeError(f"{type(self).__name__} wraps a kalle_audio_b200.BigVGANFlowVAE")
        self.model = model
        self.use_cuda_graphs = bool(use_cuda_graphs)
        self._ops, self._out = _encoder_program(model.h) if encoder else _program(model.h)
        self._src = self._ops[0].srcs[0]
        # each op's module, resolved once: looking paths up per op and push cost an eager push more host time than
        # the rest of its interpreter
        self._mods = [op.module and _module(model, op.module) for op in self._ops]
        self._convs = {op.module: m for op, m in zip(self._ops, self._mods) if op.kind in ("conv", "convT")}
        self._params = [p for m in self._mods if m is not None for p in m.parameters()]
        self.graph_captures = 0         # CUDA graphs captured by this stream
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
        key += [m.tc_precision for m in self._convs.values()]
        return tuple(key)

    def _begin(self, x: torch.Tensor) -> None:
        """Starts a stream of B clips: engines fixed per layer (``tc_layer()``) and weights packed once per weight
        version; the captured graphs hold the packed weights' addresses, so both are replaced together."""
        B, dt, dev = x.shape[0], x.dtype, x.device
        key = self._weights_key()
        if (key, B, dt, dev) != self._graph_key:
            self._engine, self._packed = {}, {}
            for c, m in self._convs.items():
                self._engine[c] = m.tc_precision if m.tc_layer() else None
                code = {None: 0, "bf16": 1, "fp32": 2}[self._engine[c]]
                packed, bias = m.packed_weight(code)
                self._packed[c] = (packed, None if bias is None else bias.clone(), code)
            self._graphs, self._static, self._graph_key = {}, {}, (key, B, dt, dev)
        self._weights = key
        self._B, self._dtype, self._dev = B, dt, dev
        self._ints, self._tens = [], []
        for op, m in zip(self._ops, self._mods):
            if op.geom is not None:                     # (rows in, first carried row, rows out), the carry
                ch = m.act.alpha.numel() if op.kind == "act" else m.in_channels
                self._ints.append((0, 0, 0))
                self._tens.append([torch.zeros((B, ch, 0), dtype=dt, device=dev)])
            else:                                       # stateless; a residual add keeps the pending rows of both operands
                self._ints.append(())
                self._tens.append([None, None] if op.kind == "axpby" and op.srcs[0] != op.srcs[1] else [])
        self._in_static = False

    def _check_weights(self) -> None:
        if self._weights_key() != self._weights:
            raise RuntimeError(f"{type(self).__name__}: the model's weights or precision changed inside a stream; "
                               "call reset() to start a new stream with the new weights")

    # ------------------------------------------------------------------ one step of every op (functional)
    def _step(self, ints, tens, x: torch.Tensor, end: bool):
        """Runs every op once on its new input rows.  Pure: returns (output rows, new ints, new tensors)."""
        vals = {self._src: x}
        new_ints, new_tens = [], []
        for op, m, st, ts in zip(self._ops, self._mods, ints, tens):
            g, xin = op.geom, vals[op.srcs[0]]
            st1, ts1 = (), []
            if g is not None:
                R, a, e = st
                win = _cat(ts[0], xin)
                R += xin.shape[2]
                o_max = g.avail(R, end)
                if o_max > e:
                    # window-relative rows (include/kvae.h): no output reads a row below the window except at the
                    # stream start, where the window starts at row 0, so a captured graph's kernel arguments hold
                    # for every later push of a phase
                    q = g.origin(a)
                    o0, o1, t_end = e - q, o_max - q, R - a if end else -1
                    if op.kind == "conv":
                        y = m.conv_window(win, *self._packed[op.module], 0, o0, o1, t_end)
                    elif op.kind == "convT":
                        y = m.conv_rows(win, *self._packed[op.module], g.p, o0, o1)
                    else:
                        y = m.window(win, 0, o0, o1, t_end)
                    e = o_max
                else:
                    y = win.new_zeros((win.shape[0], win.shape[1] if op.kind == "act" else m.out_channels, 0))
                a1 = g.first_read(e)
                st1, ts1 = (R, a1, e), [_rows(win, a1 - a)]
            elif op.kind == "axpby" and op.srcs[0] != op.srcs[1]:     # a residual add: rows both operands have
                pa = xin if ts[0] is None else _cat(ts[0], xin)
                b_in = vals[op.srcs[1]]
                pb = b_in if ts[1] is None else _cat(ts[1], b_in)
                n = min(pa.shape[2], pb.shape[2])
                y = _axpby(_rows(pa, 0, n), _rows(pb, 0, n), *op.coef) if n else pa[:, :, :0]
                ts1 = [_rows(pa, n), _rows(pb, n)]
            elif not xin.shape[2]:
                y = xin
            elif op.kind == "axpby":                    # the AMP average
                y = _axpby(xin, xin, *op.coef)
            elif op.kind == "lrelu":
                y = m(xin)
            else:                                       # tanh
                y = _unary(xin, 1)
            vals[op.dst] = y
            new_ints.append(st1)
            new_tens.append(ts1)
        return vals[self._out], new_ints, new_tens

    def _head(self, x: torch.Tensor, noise: Optional[torch.Tensor]) -> torch.Tensor:
        return _k(x)

    def _phase(self) -> tuple:
        """What a step depends on besides the carried row counts: per op with a window, the position of the next output
        in it and whether the window still starts at the stream start."""
        return tuple((st[2] - op.geom.origin(st[1]), st[1] == 0) for op, st in zip(self._ops, self._ints) if op.geom)

    # ------------------------------------------------------------------ CUDA graphs
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

    def _run_graph(self, *inputs: Optional[torch.Tensor]) -> torch.Tensor:
        """One push of ``inputs`` (the arguments of ``_head``; the first one is [B, C, n]): replays the graph of its
        (size, phase, state shapes), or runs it eagerly and captures it."""
        n = inputs[0].shape[2]
        key = (n, self._phase(), self._sig())
        G = self._graphs.get(key)
        if G is None:
            # eager run (also warms every kernel), then capture the same step from static copies of the input state
            out, ints1, tens1 = self._step(self._ints, self._tens, self._head(*inputs), False)
            src = self._static_for(self._tens)
            if not self._in_static:
                for dst_l, src_l in zip(src, self._tens):
                    for dst, t in zip(dst_l, src_l):
                        if dst is not None:
                            dst.copy_(t)
            dst_state = self._static_for(tens1)
            gin = [None if t is None else torch.empty_like(t) for t in inputs]
            if self._pool is None:
                self._pool = torch.cuda.graph_pool_handle()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=self._pool):
                gout, _, gtens = self._step(list(self._ints), src, self._head(*gin), False)
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
            self._graphs[key] = {"graph": g, "inputs": gin, "out": gout, "dints": dints, "state": dst_state}
            self.graph_captures += 1
            self._ints, self._tens, self._in_static = ints1, tens1, False
            return out
        if not self._in_static:
            src = self._static[key[2]]
            for dst_l, src_l in zip(src, self._tens):
                for dst, t in zip(dst_l, src_l):
                    if dst is not None and dst is not t:
                        dst.copy_(t)
        for dst, t in zip(G["inputs"], inputs):
            if dst is not None:
                dst.copy_(t)
        G["graph"].replay()
        self.graph_replays += 1
        self._ints = [tuple(a + d for a, d in zip(i0, di)) for i0, di in zip(self._ints, G["dints"])]
        self._tens, self._in_static = G["state"], True
        return G["out"].clone()

    # ------------------------------------------------------------------ public surface
    def _check(self, x: torch.Tensor) -> None:
        _lib.require_cuda(x, f"{type(self).__name__}.push")
        if x.requires_grad:
            raise ValueError(f"{type(self).__name__}.push: streams are inference-only and return no gradient; use "
                             "BigVGANFlowVAE.encode_with_grad / decode_with_grad for gradients (or pass a tensor that does not "
                             "require grad)")
        if x.dim() != 3 or x.shape[1] != self.in_channels:
            raise ValueError(f"expected {self._noun} [B, {self.in_channels}, n], got {tuple(x.shape)}")
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError(f"{self._noun} must be float32 or bfloat16")
        if self._B is not None:
            if x.shape[0] != self._B:
                raise ValueError("batch size changed inside a stream")
            if x.dtype != self._dtype or x.device != self._dev:
                raise ValueError("dtype or device changed inside a stream")
            self._check_weights()

    def _push(self, x: torch.Tensor, noise: Optional[torch.Tensor], chunk: int) -> torch.Tensor:
        """x [B, in_channels, n] (and the noise of the decoder's head) in steps of at most ``chunk`` rows."""
        if self._B is None:
            self._begin(x)
        pieces = []
        for i in range(0, x.shape[2], chunk):
            xi = x[:, :, i:i + chunk]
            nz = None if noise is None else noise[:, :, i:i + chunk].contiguous()
            if self.use_cuda_graphs:
                pieces.append(self._run_graph(xi.contiguous(), nz))
            else:
                out, self._ints, self._tens = self._step(self._ints, self._tens, self._head(xi, nz), False)
                pieces.append(out)
        if not pieces:
            return x.new_zeros((x.shape[0], self.out_channels, 0))
        return pieces[0] if len(pieces) == 1 else torch.cat(pieces, dim=2)

    @torch.no_grad()
    def flush(self) -> torch.Tensor:
        """The output rows still held back (right edge as in the whole call); then resets the stream."""
        if self._B is None:
            raise ValueError("nothing was pushed")
        self._check_weights()
        x = torch.zeros((self._B, self.in_channels, 0), dtype=self._dtype, device=self._dev)   # no new rows
        out, _, _ = self._step(self._ints, self._tens, x, True)
        self.reset()
        return out


class BigVGANStreamingDecoder(_OpStream):
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

    _noun = "latents"

    def __init__(self, model: BigVGANFlowVAE, max_frames: int = 16, use_cuda_graphs: bool = True,
                 do_sample: bool = False):
        super().__init__(model, False, use_cuda_graphs)
        if max_frames < 1:
            raise ValueError("max_frames must be >= 1")
        self.max_frames = int(max_frames)
        h = model.h
        self.do_sample = bool(do_sample)
        self.sample = bool(h.use_vae and do_sample)
        self.in_channels = h.latent_dim * (2 if self.sample else 1)
        self.out_channels = 1
        self.ratio = int(math.prod(h.upsample_rates))
        self.lookahead = int(bigvgan_stream_geometry(h)["lookahead"])

    def _head(self, z: torch.Tensor, noise: Optional[torch.Tensor]) -> torch.Tensor:
        """The Gaussian sample of the do_sample branch (flows.py:500-501) on the pushed frames."""
        if not self.sample:
            return _k(z)
        D = self.model.h.latent_dim
        return _gauss_sample(z[:, :D], z[:, D:], noise)

    @torch.no_grad()
    def push(self, latents: torch.Tensor, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """latents [B, D, n] (or [B, 2 D, n] with do_sample), n >= 0 -> the [B, 1, m] samples that became final."""
        self._check(latents)
        if noise is not None:
            if not self.sample:
                raise ValueError("noise is only used with do_sample on a use_vae model")
            _lib.require_cuda(noise, "BigVGANStreamingDecoder.push")
            if tuple(noise.shape) != (latents.shape[0], self.model.h.latent_dim, latents.shape[2]):
                raise ValueError("noise must be [B, D, n] like the mean half of the latents")
        if self.sample and noise is None:
            noise = torch.randn((latents.shape[0], self.model.h.latent_dim, latents.shape[2]), dtype=latents.dtype,
                                device=latents.device)
        return self._push(latents, noise, self.max_frames)


class BigVGANStreamingEncoder(_OpStream):
    """Feed audio as it arrives; get latent frames back as soon as they are final.

        se = BigVGANStreamingEncoder(model)          # model: BigVGANFlowVAE on a CUDA device
        for x in chunks:                             # x: [B, 1, n] audio, any n >= 0, fp32 or bf16
            lat = se.push(x)                         # [B, C_lat, m]: the frames that became final
        lat = se.flush()                             # the rest; the next push starts a new stream

    C_lat is ``2 * latent_dim`` for a ``use_vae`` model, as ``extract_latents`` returns.  ``torch.cat`` of everything
    returned equals ``model.extract_latents(torch.cat(chunks, -1))`` with ``torch.equal``, frame count included
    (``latent_length``).  Frame t is final once sample ``t * ratio + ratio - 1 + lookahead`` has arrived, and reads
    samples from ``t * ratio - context`` on; ``frames(n)`` counts the frames final after n samples.  Each sample is
    encoded once: the stream keeps per-op carries, not the clip.

    Engines are fixed per layer when a stream starts, as in ``BigVGANStreamingDecoder``: ``extract_latents`` puts a
    conv on the tensor cores only for inputs of >= 64 rows.  Clips that are not whole frames need nothing more: a
    strided tensor-core conv of the whole call stages its input rounded up to whole stride groups with zero rows, as
    the stream does."""

    _noun = "audio"

    def __init__(self, model: BigVGANFlowVAE, max_samples: Optional[int] = None, use_cuda_graphs: bool = True):
        super().__init__(model, True, use_cuda_graphs)
        h = model.h
        self.ratio = int(math.prod(h.downsample_rates))
        max_samples = 16 * self.ratio if max_samples is None else int(max_samples)
        if max_samples < 1:
            raise ValueError("max_samples must be >= 1")
        self.max_samples = max_samples
        geo = bigvgan_encode_stream_geometry(h)
        self.lookahead, self.context = int(geo["lookahead"]), int(geo["context"])
        self.in_channels = 1
        self.out_channels = self._mods[-1].out_channels

    def frames(self, n_samples: int, end: bool = False) -> int:
        """Latent frames final after ``n_samples`` samples; with ``end``, the frames of the whole clip
        (``latent_length``)."""
        return _lengths(self.model.h, True, n_samples, end)[self._out]

    @torch.no_grad()
    def push(self, audio: torch.Tensor) -> torch.Tensor:
        """audio [B, 1, n], n >= 0 -> the [B, C_lat, m] latent frames that became final."""
        self._check(audio)
        return self._push(audio, None, self.max_samples)
