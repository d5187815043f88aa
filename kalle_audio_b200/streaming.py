"""Incremental latent -> waveform decoding, and incremental waveform -> latent encoding (``StreamingEncoder``).

Two engines behind one class:

* **stateful** (default wherever the decoder's layers all have tensor-core kernels -- the graded architectures):
  ``kvae_decode_stream_begin / push / end``.  Every layer keeps the tail of its own input between calls (persistent
  per-layer halo state inside libkvae), so each row of each layer is computed exactly once -- 0 % recompute -- and
  the concatenated output equals ``decoder(latents)`` bit for bit.  A constant-hop stream is one CUDA-graph launch
  per hop.  Samples come out as soon as they are final, i.e. ``lookahead`` samples behind the pushed latents.
* **exact-context windows** (other architectures): described below.

Exact-context windows:

The reference streams by ``decode_audio(chunked=True, chunk_size=128, overlap=32)``
(stable_audio_tools/models/autoencoders.py:499-560; infer_stream-style callers): overlapping windows, the middle of
each pasted into the output -- 1.33x recompute, and only approximately equal to the unchunked decode (the overlap is
a guess at the receptive field).  ``StreamingDecoder`` computes the decoder's receptive field from its constructor
arguments instead (``decoder_context_frames``), so every window carries exactly the latent frames its emitted samples
depend on: the concatenated stream equals ``decoder(latents)`` of the whole sequence, the recompute is
(hop + left + right) / hop (1.21x at hop 96 for the SAO / 12.5 Hz strides), and a frame is emitted as soon as its
right context has arrived.  Windows of one shape replay as one CUDA graph (``enable_cuda_graphs``).

This is SURVEY.md section 8(f) item 1 built on the existing fused plan; it adds no kernels.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib


def decoder_context_frames(strides: Sequence[int]) -> Tuple[int, int]:
    """(left, right) latent frames an OobleckDecoder output block depends on beyond its own frames.

    Walks the stack backwards with interval arithmetic (autoencoders.py:150-191): final conv k7 pad 3; per
    DecoderBlock three ResidualUnits (k7, dilation 9 / 3 / 1) and a ConvTranspose1d(k = 2s + s % 2, stride s,
    pad ceil(s / 2)); first conv k7 pad 3.  ``strides`` in constructor (encoder) order."""
    ratio = int(math.prod(strides))
    f0, f1 = 1000, 1001                      # one frame far from the edges
    lo, hi = f0 * ratio, f1 * ratio - 1      # output sample range of that frame
    lo, hi = lo - 3, hi + 3                  # final conv
    for s in strides:                        # decoder blocks in reverse execution order = encoder stride order
        lo, hi = lo - 39, hi + 39            # ResidualUnits: 3 * (1 + 3 + 9)
        k, p = 2 * s + s % 2, math.ceil(s / 2)
        lo = -((-(lo + p - k + 1)) // s)     # ceil((lo + p - k + 1) / s)
        hi = (hi + p) // s
    lo, hi = lo - 3, hi + 3                  # first conv
    return f0 - lo, hi - (f1 - 1)


def encoder_context_samples(strides: Sequence[int]) -> Tuple[int, int]:
    """(left, right) input samples an OobleckEncoder latent frame depends on beyond its own ``ratio`` samples.

    Walks the stack backwards with interval arithmetic (autoencoders.py:64-81, 130-141): final conv k3 pad 1; per
    EncoderBlock, in reverse, the strided Conv1d(k = 2s, stride s, pad ceil(s / 2)) and three ResidualUnits (k7,
    dilation 9 / 3 / 1: 39 rows each way at that block's rate); head conv k7 pad 3.  ``strides`` in constructor order."""
    ratio = int(math.prod(strides))
    f0 = 1000                                # one frame far from the edges
    lo, hi = f0 - 1, f0 + 1                  # final conv
    for s in reversed(strides):
        p = math.ceil(s / 2)
        lo, hi = lo * s - p, hi * s + 2 * s - 1 - p   # output t reads rows t*s - p .. t*s + 2s - 1 - p
        lo, hi = lo - 39, hi + 39            # ResidualUnits: 3 * (1 + 3 + 9)
    lo, hi = lo - 3, hi + 3                  # head conv
    return f0 * ratio - lo, hi - ((f0 + 1) * ratio - 1)


class StreamingEncoder:
    """Feed audio as it arrives; get latent frames back as soon as they are final.

        se = StreamingEncoder(autoencoder.encoder)
        for x in audio_chunks:               # x: [B, io_channels, n], any n >= 0
            z = se.push(x)                   # [B, latent_dim, m], m = frames that became final (possibly 0)
        tail = se.flush()                    # the last frames (right edge zero-padded like the whole-clip encode)

    ``torch.cat`` of everything returned equals ``encoder(torch.cat(audio_chunks, -1))`` bit for bit when the total
    length is a multiple of ``ratio``; otherwise it is the ``kvae_plan_out_length(L)`` frames the reference's floor
    arithmetic gives (``encoder(x, valid_len=...)``).  Every layer keeps the tail of its own input inside libkvae
    (``kvae_encode_stream_*``), so no sample is encoded twice; a frame comes out once ``lookahead`` samples past its
    last sample have arrived.  Needs an encoder whose every layer has a tensor-core kernel (channels and latent_dim
    multiples of 64, a 128-channel head): other architectures raise ``KvaeError`` on the first push."""

    def __init__(self, encoder, max_samples: Optional[int] = None, use_cuda_graphs: bool = True):
        """``max_samples``: the longest push the stream takes in one library call (longer pushes are split)."""
        if not hasattr(encoder, "_arch") or encoder._direction != _lib.KVAE_ENCODER:
            raise TypeError("StreamingEncoder wraps a kalle_audio_b200.OobleckEncoder")
        self.encoder = encoder
        strides = [encoder._arch.strides[i] for i in range(encoder._arch.n_stages)]
        self.ratio = int(math.prod(strides))
        self.max_samples = int(max_samples or max(65536, 4 * self.ratio))
        if self.max_samples < 1:
            raise ValueError("max_samples must be >= 1")
        self._use_graphs = bool(use_cuda_graphs)
        self._native = None            # (handle, finalizer, runner, batch) once the first push fixes device and batch
        self._last_dtype = None
        self.lookahead: Optional[int] = None   # samples; set by the library when the first push starts the stream

    def reset(self) -> None:
        """Drops the stream and its state; the next push starts a new one."""
        if self._native is not None:
            self._native[1]()
            self._native = None

    def _stream(self, audio: torch.Tensor):
        import ctypes as C
        import weakref
        if self._native is not None:
            if self._native[3] != audio.shape[0]:
                raise ValueError("batch size changed inside a stream")
            return self._native
        L = _lib.lib()
        r = self.encoder.runner(audio.device)
        r.sync_weights()
        h = C.c_void_p()
        _lib.check(L.kvae_encode_stream_begin(r.handle, audio.shape[0], self.max_samples, int(self._use_graphs),
                                              C.byref(h)))
        fin = weakref.finalize(self, L.kvae_encode_stream_destroy, h)
        self._native = (h, fin, r, audio.shape[0])
        self.lookahead = int(L.kvae_encode_stream_lookahead(h))
        return self._native

    def _call(self, x: Optional[torch.Tensor], end: bool) -> torch.Tensor:
        import ctypes as C
        L = _lib.lib()
        h, _, r, B = self._native
        r.sync_weights()
        dev = r.device
        out_dt = self.encoder._out_dtype(x) if x is not None else self._last_dtype
        self._last_dtype = out_dt
        kdt = out_dt if out_dt in (torch.float32, torch.bfloat16) else torch.float32
        n = 0 if x is None else x.shape[2]
        nf = int(L.kvae_encode_stream_frames(h, n, int(end)))
        if nf < 0:
            raise _lib.KvaeError(L.kvae_last_error().decode())
        lat = torch.empty((B, self.encoder._out_channels_for_plan, nf), dtype=kdt, device=dev)
        got = C.c_longlong(0)
        if end:
            _lib.check(L.kvae_encode_stream_end(h, lat.data_ptr(), _lib.dtype_code(kdt), nf, C.byref(got),
                                                _lib.stream_ptr(dev)))
        else:
            xin = x if x.dtype in (torch.float32, torch.bfloat16) else x.float()
            xin = xin.contiguous()
            _lib.check(L.kvae_encode_stream_push(h, xin.data_ptr(), _lib.dtype_code(xin.dtype), n, lat.data_ptr(),
                                                 _lib.dtype_code(kdt), nf, C.byref(got), _lib.stream_ptr(dev)))
        assert got.value == nf
        return lat if lat.dtype == out_dt else lat.to(out_dt)

    def push(self, audio: torch.Tensor) -> torch.Tensor:
        """audio [B, io_channels, n] -> the latent frames [B, latent_dim, m] that became final."""
        _lib.require_cuda(audio, "StreamingEncoder.push")
        if audio.dim() != 3:
            raise ValueError("expected [B, C, n]")
        self._stream(audio)
        pieces = [self._call(audio[:, :, i:i + self.max_samples], False)
                  for i in range(0, audio.shape[2], self.max_samples)]
        if not pieces:
            return audio.new_zeros((audio.shape[0], self.encoder._out_channels_for_plan, 0),
                                   dtype=self.encoder._out_dtype(audio))
        return pieces[0] if len(pieces) == 1 else torch.cat(pieces, dim=2)

    def flush(self) -> torch.Tensor:
        """Everything not yet emitted (end of stream).  The stream starts over with the next push."""
        if self._native is None:
            raise ValueError("nothing was pushed")
        return self._call(None, True)


class StreamingDecoder:
    """Feed latent frames as they arrive; get waveform back as soon as it is final.

        sd = StreamingDecoder(autoencoder.decoder, hop=96)
        for z in latent_chunks:              # z: [B, D, n], any n >= 0
            wav = sd.push(z)                 # [B, C, m * ratio], m = frames that became final (possibly 0)
        tail = sd.flush()                    # the last frames (right edge zero-padded like the unchunked decode)

    ``torch.cat`` of everything returned equals ``decoder(torch.cat(latent_chunks, -1))``."""

    def __init__(self, decoder, hop: int = 96, use_cuda_graphs: bool = True, stateful: Optional[bool] = None,
                 max_frames: Optional[int] = None):
        """``stateful``: None = the stateful engine when the plan supports it, else exact-context windows; True =
        stateful or raise; False = windows.  ``hop``: window mode emits in multiples of ``hop`` frames; the stateful
        engine takes pushes of any size up to ``max_frames`` (default ``max(hop, 128)``) and splits longer ones."""
        if not hasattr(decoder, "_arch") or decoder._direction != _lib.KVAE_DECODER:
            raise TypeError("StreamingDecoder wraps a kalle_audio_b200.OobleckDecoder")
        if hop < 1:
            raise ValueError("hop must be >= 1")
        self.decoder = decoder
        self.hop = int(hop)
        strides = [decoder._arch.strides[i] for i in range(decoder._arch.n_stages)]
        self.ratio = int(math.prod(strides))
        self.left, self.right = decoder_context_frames(strides)
        self.max_frames = int(max_frames or max(self.hop, 128))
        self._use_graphs = bool(use_cuda_graphs)
        self._want_stateful = stateful
        self._native = None            # (handle, finalizer, runner, batch) once the first push fixes device and batch
        self.stateful = False
        if use_cuda_graphs and stateful is False:
            decoder.enable_cuda_graphs(True)
        self.reset()

    def reset(self) -> None:
        self._buf: Optional[torch.Tensor] = None   # frames [emitted - left_available, received)
        self._emitted = 0                          # frames already returned
        self._start = 0                            # absolute index of _buf[..., 0]
        if self._native is not None:
            self._native[1]()                      # destroy the stream: a fresh one starts with zeroed halo state
            self._native = None

    @property
    def recompute_factor(self) -> float:
        return 1.0 if self.stateful else (self.hop + self.left + self.right) / self.hop

    # ------------------------------------------------------------------ stateful engine (libkvae)
    def _native_stream(self, latents: torch.Tensor):
        import ctypes as C
        import weakref
        if self._native is not None:
            if self._native[3] != latents.shape[0]:
                raise ValueError("batch size changed inside a stream")
            return self._native
        if self._want_stateful is False:
            return None
        L = _lib.lib()
        r = self.decoder.runner(latents.device)
        r.sync_weights()
        h = C.c_void_p()
        rc = L.kvae_decode_stream_begin(r.handle, latents.shape[0], self.max_frames, int(self._use_graphs), C.byref(h))
        if rc != 0:
            if self._want_stateful:
                raise _lib.KvaeError(L.kvae_last_error().decode())
            self._want_stateful = False            # this architecture streams by windows
            if self._use_graphs:
                self.decoder.enable_cuda_graphs(True)
            return None
        fin = weakref.finalize(self, L.kvae_decode_stream_destroy, h)
        self._native = (h, fin, r, latents.shape[0])
        self.stateful = True
        self.lookahead = int(L.kvae_decode_stream_lookahead(h))
        return self._native

    def _native_call(self, nat, z: Optional[torch.Tensor], end: bool) -> torch.Tensor:
        import ctypes as C
        L = _lib.lib()
        h, _, r, B = nat
        r.sync_weights()
        dev = r.device
        out_dt = self.decoder._out_dtype(z) if z is not None else self._last_dtype
        self._last_dtype = out_dt
        kdt = out_dt if out_dt in (torch.float32, torch.bfloat16) else torch.float32
        n = 0 if z is None else z.shape[2]
        ns = int(L.kvae_decode_stream_samples(h, n, int(end)))
        if ns < 0:
            raise _lib.KvaeError(L.kvae_last_error().decode())
        wav = torch.empty((B, self.decoder._out_channels_for_plan, ns), dtype=kdt, device=dev)
        got = C.c_longlong(0)
        if end:
            _lib.check(L.kvae_decode_stream_end(h, wav.data_ptr(), _lib.dtype_code(kdt), ns, C.byref(got),
                                                _lib.stream_ptr(dev)))
        else:
            zin = z if z.dtype in (torch.float32, torch.bfloat16) else z.float()
            zin = zin.contiguous()
            _lib.check(L.kvae_decode_stream_push(h, zin.data_ptr(), _lib.dtype_code(zin.dtype), n, wav.data_ptr(),
                                                 _lib.dtype_code(kdt), ns, C.byref(got), _lib.stream_ptr(dev)))
        assert got.value == ns
        return wav if wav.dtype == out_dt else wav.to(out_dt)

    def _decode_window(self, first: int, last: int, end_of_stream: bool) -> torch.Tensor:
        """Decodes frames [first, last) with whatever context exists and returns exactly their samples."""
        buf, start = self._buf, self._start
        w0 = max(first - self.left, start)
        w1 = last if end_of_stream else last + self.right
        win = buf[:, :, w0 - start:w1 - start]
        with torch.no_grad():
            y = self.decoder(win)
        return y[:, :, (first - w0) * self.ratio:(last - w0) * self.ratio]

    def _trim(self) -> None:
        keep_from = max(self._emitted - self.left, self._start)
        if keep_from > self._start:
            self._buf = self._buf[:, :, keep_from - self._start:]
            self._start = keep_from

    def push(self, latents: torch.Tensor) -> torch.Tensor:
        _lib.require_cuda(latents, "StreamingDecoder.push")
        if latents.dim() != 3:
            raise ValueError("expected [B, D, n]")
        nat = self._native_stream(latents)
        if nat is not None:
            self._pushed = getattr(self, "_pushed", 0) + latents.shape[2]
            pieces = [self._native_call(nat, latents[:, :, i:i + self.max_frames], False)
                      for i in range(0, latents.shape[2], self.max_frames)]
            if not pieces:
                return latents.new_zeros((latents.shape[0], self.decoder._out_channels_for_plan, 0))
            return pieces[0] if len(pieces) == 1 else torch.cat(pieces, dim=2)
        self._buf = latents if self._buf is None else torch.cat([self._buf, latents], dim=2)
        received = self._start + self._buf.shape[2]
        out: List[torch.Tensor] = []
        # a frame is final once `right` frames after it have arrived; emit in hop-sized windows
        while received - self.right - self._emitted >= self.hop:
            out.append(self._decode_window(self._emitted, self._emitted + self.hop, False))
            self._emitted += self.hop
            self._trim()
        if out:
            return torch.cat(out, dim=2)
        B = latents.shape[0]
        return latents.new_zeros((B, self.decoder._out_channels_for_plan, 0))

    def flush(self) -> torch.Tensor:
        """Everything not yet emitted (end of stream).  Resets the state."""
        if self._native is not None:
            res = self._native_call(self._native, None, True)
            self._pushed = 0
            return res                  # the library has reset the stream: the next push starts a new one
        if self._buf is None:
            raise ValueError("nothing was pushed")
        received = self._start + self._buf.shape[2]
        out: List[torch.Tensor] = []
        while received - self._emitted > 0:
            n = min(self.hop, received - self._emitted)
            last = self._emitted + n
            end = last + self.right >= received       # no full right context left: this window ends the stream
            if end:
                last = received
            out.append(self._decode_window(self._emitted, last, end))
            self._emitted = last
            self._trim()
        res = torch.cat(out, dim=2) if out else self._buf.new_zeros((self._buf.shape[0],
                                                                     self.decoder._out_channels_for_plan, 0))
        self.reset()
        return res
