"""Stateful streaming decode and encode for ``BigVGANFlowVAE.inference_from_latents`` (flows.py:498-529) and
``extract_latents`` (:494-496).

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

The op list comes from one description of the decoder (``bigvgan._program``) that three interpreters read: the integer
one behind ``bigvgan_stream_geometry`` (rows available per op, lookahead), the tensor one behind the decoder, and the
ragged whole-clip decode of ``BigVGANFlowVAE.inference_from_latents(valid_len=...)``.

``BigVGANStreamingEncoder`` runs the encoder's op list (``bigvgan._encoder_program``) the same way: every conv keeps a
carry of whole stride groups from a stream row = 0 (mod stride) on and runs ``kvae_conv1d_stream_fwd`` on
``[carry | new rows]`` with the layer's own padding, the stream end given only at ``flush``; LeakyReLU is stateless on
the new rows; the residual adds keep the pending rows of both operands.

Pushes whose (size, start-up phase) was seen before replay one ``torch.cuda.CUDAGraph``; the op state lives in static
buffers per phase, so a constant-hop stream in steady state is one graph launch per push.  Both streams share that
machinery (``_GraphedStream``).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch

from . import _lib
from .bigvgan import (_AA_HALO, BigVGANFlowVAE, _axpby, _encoder_program, _gauss_sample, _geom_of, _k, _lengths,
                      _module, _program, _unary)


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
        if op[0] == "lrelu":
            rate[op[3]], first[op[3]] = rate[op[2]], first[op[2]]
            continue
        if op[0] == "add":
            rate[op[3]], first[op[3]] = rate[op[1]], min(first[op[1]], first[op[2]])
            continue
        g = _geom_of(h, op)
        r_in = rate[op[2]]
        rate[op[3]] = r_in * g.s
        first[op[3]] = first[op[2]] - g.reach() * r_in
        bound += g.span * r_in
        rows.append({"module": op[1], "rate": r_in, "span": g.span, "dilation": g.d, "stride": g.s,
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


# ------------------------------------------------------------------------------------------------ the decoder
def _cat(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    if b.shape[2] == 0:
        return a
    if a.shape[2] == 0:
        return b
    return torch.cat([a, b], dim=2)


def _rows(t: torch.Tensor, lo: int, hi: Optional[int] = None) -> torch.Tensor:
    return t[:, :, lo:hi] if (lo, hi) != (0, None) else t


class _GraphedStream:
    """What both streams share: engines fixed and weights packed per weight version, the check that the weights did not
    change inside a stream, and the CUDA graphs (static state buffers per phase, capture, replay).  A subclass sets
    ``model``, ``_params`` (the parameters its ops read) and ``_convs`` (their conv module paths), calls
    ``_init_graphs``, and defines ``_step``, ``_head`` and ``_phase``."""

    def _init_graphs(self) -> None:
        self.graph_captures = 0         # CUDA graphs captured by this stream
        self.graph_replays = 0          # pushes served by replaying one
        self._graphs: Dict[tuple, dict] = {}
        self._static: Dict[tuple, List[torch.Tensor]] = {}
        self._pool = None
        self._graph_key = None

    def _weights_key(self) -> tuple:
        key = [(p.data_ptr(), p._version) for p in self._params]
        key += [_module(self.model, c).tc_precision for c in self._convs]
        return tuple(key)

    def _fix_engines(self, B: int, dt: torch.dtype, dev: torch.device) -> None:
        """Starts a stream of B clips: engines fixed per layer (``tc_layer()``) and weights packed once per weight
        version; the captured graphs hold the packed weights' addresses, so both are replaced together."""
        key = self._weights_key()
        if (key, B, dt, dev) != self._graph_key:
            self._engine, self._packed = {}, {}
            for c in self._convs:
                m = _module(self.model, c)
                self._engine[c] = m.tc_precision if m.tc_layer() else None
                code = {None: 0, "bf16": 1, "fp32": 2}[self._engine[c]]
                packed, bias = m.packed_weight(code)
                self._packed[c] = (packed, None if bias is None else bias.clone(), code)
            self._graphs, self._static, self._graph_key = {}, {}, (key, B, dt, dev)
        self._weights = key
        self._B, self._dtype, self._dev = B, dt, dev

    def _check_weights(self) -> None:
        if self._weights_key() != self._weights:
            raise RuntimeError(f"{type(self).__name__}: the model's weights or precision changed inside a stream; "
                               "call reset() to start a new stream with the new weights")

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


class BigVGANStreamingDecoder(_GraphedStream):
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
        self._init_graphs()
        self.reset()

    # ------------------------------------------------------------------ stream state
    def reset(self) -> None:
        """Drops the stream; the next push starts a new one (captured graphs stay while the weights do)."""
        self._B = None
        self._ints: Optional[List[tuple]] = None
        self._tens: Optional[List[List[torch.Tensor]]] = None
        self._in_static = False
        self._weights = None

    def _begin(self, z: torch.Tensor) -> None:
        B, dev, dt = z.shape[0], z.device, z.dtype
        self._fix_engines(B, dt, dev)
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
                    y = _module(self.model, op[1]).conv_rows(win, *self._packed[op[1]], 0, 0, n_out)
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
                    y = m.conv_rows(win, *self._packed[op[1]], g.p, e - g.s * j0, o_max - g.s * j0)
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
                    y = _module(self.model, op[1]).window(win, a - off, e - off, o_max - off, R - off if end else -1)
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
        return _gauss_sample(z[:, :D], z[:, D:], noise)

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
            self._check_weights()
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
        self._check_weights()
        D = self.in_channels
        z = torch.zeros((self._B, D, 0), dtype=self._dtype, device=self._dev)
        nz = None if not self.sample else torch.zeros((self._B, self.model.h.latent_dim, 0), dtype=self._dtype,
                                                      device=self._dev)
        out, _, _ = self._step(self._ints, self._tens, self._head(z, nz), True)
        self.reset()
        return out


# ------------------------------------------------------------------------------------------------ the encoder
class BigVGANStreamingEncoder(_GraphedStream):
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

    Engines are fixed per layer when a stream starts, as in ``BigVGANStreamingDecoder``.  ``extract_latents`` puts a
    conv on the tensor cores only for inputs of >= 64 rows, and a strided tensor-core conv of the whole call needs an
    input length divisible by its stride; for other clips the stream equals the ragged call
    ``extract_latents(x_padded, valid_len=[L])[..., :latent_length(L)]`` on the clip padded to whole frames."""

    def __init__(self, model: BigVGANFlowVAE, max_samples: Optional[int] = None, use_cuda_graphs: bool = True):
        if not isinstance(model, BigVGANFlowVAE):
            raise TypeError("BigVGANStreamingEncoder wraps a kalle_audio_b200.BigVGANFlowVAE")
        h = model.h
        self.ratio = int(math.prod(h.downsample_rates))
        max_samples = 16 * self.ratio if max_samples is None else int(max_samples)
        if max_samples < 1:
            raise ValueError("max_samples must be >= 1")
        self.model = model
        self.max_samples = max_samples
        self.use_cuda_graphs = bool(use_cuda_graphs)
        self._ops, self._out = _encoder_program(h)
        self._geoms = [_geom_of(h, op) for op in self._ops]
        geo = bigvgan_encode_stream_geometry(h)
        self.lookahead, self.context = int(geo["lookahead"]), int(geo["context"])
        self._convs = sorted({op[1] for op in self._ops if op[0] == "conv"})
        self.out_channels = _module(model, self._ops[-1][1]).out_channels
        self._params = list(model.audio_encoder.parameters())
        self._init_graphs()
        self.reset()

    def frames(self, n_samples: int, end: bool = False) -> int:
        """Latent frames final after ``n_samples`` samples; with ``end``, the frames of the whole clip
        (``latent_length``)."""
        return _lengths(self.model.h, True, n_samples, end)[self._out]

    # ------------------------------------------------------------------ stream state
    def reset(self) -> None:
        """Drops the stream; the next push starts a new one (captured graphs stay while the weights do)."""
        self._B = None
        self._ints: Optional[List[tuple]] = None
        self._tens: Optional[List[List[torch.Tensor]]] = None
        self._in_static = False
        self._weights = None

    def _begin(self, x: torch.Tensor) -> None:
        B, dev, dt = x.shape[0], x.device, x.dtype
        self._fix_engines(B, dt, dev)
        self._ints, self._tens = [], []
        for op in self._ops:
            if op[0] == "conv":
                ch = _module(self.model, op[1]).in_channels
                self._ints.append((0, 0, 0))                            # (rows in, first carried row, rows out)
                self._tens.append([torch.zeros((B, ch, 0), dtype=dt, device=dev)])
            elif op[0] == "add":
                self._ints.append((0,))
                self._tens.append([None, None])                         # pending rows of each operand
            else:
                self._ints.append(())
                self._tens.append([])
        self._in_static = False

    # ------------------------------------------------------------------ one step of every op (functional)
    def _step(self, ints, tens, x: torch.Tensor, end: bool):
        """Runs every op once on its new input rows.  Pure: returns (latent rows, new ints, new tensors)."""
        vals = {"x": x}
        new_ints, new_tens = [], []
        for op, g, st, ts in zip(self._ops, self._geoms, ints, tens):
            kind = op[0]
            if kind == "conv":
                R, a, e = st
                xin = vals[op[2]]
                win = _cat(ts[0], xin)
                R += xin.shape[2]
                o_max = g.avail(R, end)
                m = _module(self.model, op[1])
                if o_max > e:
                    # window-relative rows (include/kvae.h): the window starts at a row = 0 (mod stride), and no
                    # output reads a row below it except at the stream start, where the window starts at row 0
                    q = a // g.s
                    y = m.conv_window(win, *self._packed[op[1]], 0, e - q, o_max - q, R - a if end else -1)
                    e = o_max
                else:
                    y = win.new_zeros((win.shape[0], m.out_channels, 0))
                a1 = max(0, e * g.s - g.pl) // g.s * g.s                # first row the next output reads, whole groups
                vals[op[3]] = y
                new_ints.append((R, a1, e))
                new_tens.append([_rows(win, a1 - a)])
            elif kind == "lrelu":
                xin = vals[op[2]]
                vals[op[3]] = _module(self.model, op[1])(xin) if xin.shape[2] else xin
                new_ints.append(())
                new_tens.append([])
            else:                                                       # add: rows both operands have
                a_in, b_in = vals[op[1]], vals[op[2]]
                pa = a_in if ts[0] is None else _cat(ts[0], a_in)
                pb = b_in if ts[1] is None else _cat(ts[1], b_in)
                n = min(pa.shape[2], pb.shape[2])
                vals[op[3]] = _axpby(_rows(pa, 0, n), _rows(pb, 0, n), 1.0, 1.0) if n else pa[:, :, :0]
                new_ints.append((st[0] + n,))
                new_tens.append([_rows(pa, n), _rows(pb, n)])
        return vals[self._out], new_ints, new_tens

    def _head(self, x: torch.Tensor) -> torch.Tensor:
        return _k(x)

    def _phase(self) -> tuple:
        """What a step depends on besides the carried row counts: per conv, the next output's position in its window
        and whether the window still starts at the stream start."""
        return tuple((st[2] - st[1] // g.s, st[1] == 0) for op, g, st in zip(self._ops, self._geoms, self._ints)
                     if op[0] == "conv")

    # ------------------------------------------------------------------ public surface
    def _check(self, x: torch.Tensor) -> None:
        _lib.require_cuda(x, "BigVGANStreamingEncoder.push")
        if x.dim() != 3 or x.shape[1] != 1:
            raise ValueError(f"expected audio [B, 1, n], got {tuple(x.shape)}")
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("audio must be float32 or bfloat16")
        if self._B is not None:
            if x.shape[0] != self._B:
                raise ValueError("batch size changed inside a stream")
            if x.dtype != self._dtype or x.device != self._dev:
                raise ValueError("dtype or device changed inside a stream")
            self._check_weights()

    @torch.no_grad()
    def push(self, audio: torch.Tensor) -> torch.Tensor:
        """audio [B, 1, n], n >= 0 -> the [B, C_lat, m] latent frames that became final."""
        self._check(audio)
        if self._B is None:
            self._begin(audio)
        pieces = []
        for i in range(0, audio.shape[2], self.max_samples):
            x = audio[:, :, i:i + self.max_samples]
            if self.use_cuda_graphs:
                pieces.append(self._run_graph(x.contiguous()))
            else:
                out, self._ints, self._tens = self._step(self._ints, self._tens, self._head(x), False)
                pieces.append(out)
        if not pieces:
            return audio.new_zeros((audio.shape[0], self.out_channels, 0))
        return pieces[0] if len(pieces) == 1 else torch.cat(pieces, dim=2)

    @torch.no_grad()
    def flush(self) -> torch.Tensor:
        """The frames still held back (right edge as in the whole encode); then resets the stream."""
        if self._B is None:
            raise ValueError("nothing was pushed")
        self._check_weights()
        x = torch.zeros((self._B, 1, 0), dtype=self._dtype, device=self._dev)
        out, _, _ = self._step(self._ints, self._tens, x, True)
        self.reset()
        return out
