// Stateful streaming decoder (included by kvae.cu inside its anonymous-namespace context).
//
// The reference streams with decode_audio(chunked=True, chunk_size=128, overlap=32)
// (stable_audio_tools/models/autoencoders.py:499-560): overlapping windows are decoded from scratch and the middle
// of each is pasted into the output -- 1.33x the work, and every window pays the zero-padded edges.  Here every layer
// keeps the tail of its own input between calls instead (persistent per-layer halo state), so each output row of
// each layer is computed exactly once: 0 % recompute, and the stream equals the unchunked decode bit for bit.
//
// Mechanics.  Every convolution is run in its "valid" form on a window buffer [carry rows | new rows]:
//   * a layer whose taps read input rows q + d, d in [dmin, dmax], keeps span = dmax - dmin rows between calls and
//     produces out = rows - span new outputs per call, trailing its input by dmax rows (that accumulated lag is the
//     decoder's look-ahead, 10 latent frames for the SAO / 12.5 Hz strides);
//   * the kernels are the ones of the batch path: the window is just another tensor map, all tap offsets are shifted
//     by -dmin so they are non-negative (StreamGeom::row_bias), outputs are appended to the consumer's window buffer;
//   * at the start of a stream a buffer holds -dmin rows of zeros (the conv's left padding); at the end
//     (kvae_decode_stream_end) every layer emits dmax more rows, reading past its last row, where TMA's out-of-bounds
//     zero fill is the conv's right padding;
//   * after a call the last `span` rows of every buffer move to its front (one batched copy kernel).
// A call with the same buffer fill and frame count as an earlier one re-uses its prepared launches, and (optionally)
// replays them as one CUDA graph: the steady state of a constant-hop stream is one graph launch per hop.
//
// The encoder (kvae_encode_stream_*) runs the same engine in the other direction: the input is a channels-first fp32
// sample window [B, io, cap] (its carry: the head's 6-sample halo), the rates go down by each strided conv's stride s,
// and the last conv writes channels-first latents into a staging buffer.  A strided conv keeps the phase assignment of
// the batch path, which views its input as [T/s, s, C]: its window starts at an absolute row = 0 (mod s), its carry is
// a whole number of s-row groups and its bias counts groups; it emits output q once every row q reads has arrived
// (rows of a partly filled group feed only outputs that are not stored).  At the end of the stream the rows of the
// last partial group past the true end are zeroed by a memset in the prepared launch list, so every layer's output
// count follows the reference's floor arithmetic (ConvGeom::out_len).

struct StreamOut {            // geometry shared by the raw (stream) and act (operand) tensors one step produces
  long long rows = 0;         // valid rows per clip currently in the buffers
  long long abs_base = 0;     // absolute index (at this tensor's rate) of buffer row 0
  long long cap = 0;          // rows per clip the buffers can hold (= pitch)
  int keep = 0;               // rows the consumer needs between calls (its span)
  int init_rows = 0;          // zero rows at the start of a stream (the consumer's -dmin)
  size_t off_raw = 0, off_act = 0;
  int raw_row_bytes = 0, act_row_bytes = 0;   // 0: tensor not produced
  int cf = 0;                 // > 0: channels-first fp32 [B, cf, cap] (the encoder's sample window; raw_row_bytes = 4)
};

struct StreamStep {
  StepKind kind = kTcConv;
  int bias = 0;               // in input groups of P_in rows: added to every tap offset
  int span = 0;               // last window row output 0 reads (input rows): the rows kept between calls
  int dmax = 0;               // last input row output q reads, relative to row q * P_in
  int P_in = 1, P_out = 1;
  int in_out = -1;            // index of the StreamOut this step reads (-1: the stream's input buffer, slot 0 of `outs`)
};

struct StreamCarry { uint8_t* dst; const uint8_t* src; unsigned long long bytes; unsigned long long pitch; };

__global__ void stream_carry_kernel(const StreamCarry* d, int n_desc) {
  const StreamCarry c = d[blockIdx.y];
  uint8_t* dst = c.dst + static_cast<size_t>(blockIdx.z) * c.pitch;
  const uint8_t* src = c.src + static_cast<size_t>(blockIdx.z) * c.pitch;
  const size_t n16 = c.bytes / 16;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n16; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(src)[i];
  (void)n_desc;
}

// one clip-strided 2D region: `height` rows of `width` bytes, `pitch` bytes apart
struct StreamRegion { uint8_t* dst; const uint8_t* src; size_t width, pitch, height; };

__global__ void stream_append_cf_kernel(const void* x, int x_f32, float* y, long long n, long long y_pitch) {
  const size_t row = blockIdx.y;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
    y[row * y_pitch + i] = ld_elem(x, row * n + i, x_f32);
}

struct PreparedPush {
  std::vector<StepLaunch> steps;           // the steps that run in this call, in order
  long long n_out = 0;                     // rows the call emits (samples / latent frames)
  int in_rows0 = 0;                        // row of the input buffer where the new rows go
  std::vector<StreamRegion> zero;          // end of stream: rows of a strided conv's last partial group past the end
  std::vector<StreamCarry> carry;          // non-overlapping moves (one kernel)
  std::vector<StreamCarry> carry_overlap;  // overlapping moves (through scratch)
  std::vector<StreamRegion> carry_cf;      // the channels-first sample window (through scratch)
  StreamCarry* carry_dev = nullptr;
  std::vector<StreamOut> after;            // state after this call
  cudaGraphExec_t graph = nullptr;
  bool eager_done = false;
  ~PreparedPush() {
    if (graph) cudaGraphExecDestroy(graph);
    if (carry_dev) cudaFree(carry_dev);
  }
};

}  // namespace

struct kvae_stream {
  kvae_plan* plan = nullptr;
  bool enc = false;                 // encoder: samples in, latent frames out
  int B = 0, max_frames = 0;
  bool use_graphs = false;
  uint8_t* ws = nullptr;
  size_t ws_bytes = 0;
  std::vector<StreamOut> outs;      // [0] = the input window (decoder: channels-last latents, encoder: channels-first
                                    // samples), [1 + k] = outputs of step k
  std::vector<StreamStep> ss;
  uint8_t* z_stage = nullptr;       // [B, latent, max_frames] in the caller's dtype (4 bytes per element reserved)
  float* wav_stage = nullptr;       // [B, io, max_samples] (the encoder's input: caller's dtype)
  __nv_bfloat16* col = nullptr;     // encoder head on the tensor cores: im2col operand [B, rows, 64] (inside ws)
  uint8_t* scratch = nullptr;       // overlapping carry moves
  size_t scratch_bytes = 0;
  long long max_samples = 0;
  long long max_in = 0;             // input rows one call takes (max_frames / max_samples)
  long long ratio = 1;
  bool stream_f16 = false;
  std::map<std::vector<long long>, std::unique_ptr<PreparedPush>> cache;
  long long frames_in = 0, samples_out = 0;
  bool needs_zero = false;          // the carry regions must be zeroed before the next stream starts
  cudaStream_t cap_stream = nullptr;   // graph capture happens here (the caller's stream may be the legacy default)
};

namespace {

void stream_reset(kvae_stream* s) {
  for (StreamOut& o : s->outs) {
    o.rows = o.init_rows;
    o.abs_base = -static_cast<long long>(o.init_rows);
  }
  s->frames_in = 0;
  s->samples_out = 0;
}

// per-step tap statistics: input groups (of P_in rows; rows for stride-1 and transposed convs) and input rows read
bool stream_step_geometry(const ConvGeom& g, StreamStep& st, std::string& err) {
  TapPlan tp;
  if (!build_taps(g, tp, err)) return false;
  int dmin = 1 << 30, dmax = -(1 << 30), rmax = -(1 << 30);
  for (const Tap& t : tp.taps) {
    dmin = std::min(dmin, t.a_row + t.shift);
    dmax = std::max(dmax, t.a_row + t.shift);
    rmax = std::max(rmax, (t.a_row + t.shift) * tp.P_in + t.a_phase);
  }
  st.bias = -dmin;
  st.dmax = rmax;
  st.span = rmax + st.bias * tp.P_in;
  st.P_in = tp.P_in;
  st.P_out = tp.P_out;
  if (dmin > 0 || dmax < 0) { err = "streaming: one-sided receptive field unsupported"; return false; }
  return true;
}

// Lays out one call: how many rows every step produces, the launches, the carry moves and the state afterwards.
bool stream_prepare(kvae_stream* s, int n_in, bool flush, int out_dtype, PreparedPush& P, std::string& err) {
  kvae_plan* p = s->plan;
  const std::vector<Step>& steps = p->steps;
  const int n = static_cast<int>(steps.size());
  const int B = s->B;
  std::vector<StreamOut> cur = s->outs;
  P.in_rows0 = static_cast<int>(cur[0].rows);
  cur[0].rows += n_in;
  if (cur[0].rows > cur[0].cap) { err = "streaming: input buffer overflow"; return false; }
  uint8_t* base = s->ws;
  auto raw_ptr = [&](const StreamOut& o, long long row) -> uint8_t* { return base + o.off_raw + static_cast<size_t>(row) * o.raw_row_bytes; };
  auto act_ptr = [&](const StreamOut& o, long long row) -> uint8_t* { return base + o.off_act + static_cast<size_t>(row) * o.act_row_bytes; };
  P.n_out = 0;
  std::vector<long long> consumed(cur.size(), 0);   // rows of each buffer its consumer is done with after this call
  for (int k = 0; k < n; ++k) {
    const StreamStep& st = s->ss[k];
    if (st.kind == kRuSecond) continue;
    const ConvLayer& c = p->convs[steps[k].conv];
    StreamOut& in = cur[st.in_out + 1];
    const int ko = (st.kind == kRuFused) ? k + 1 : k;       // the step whose tensors receive the result
    StreamOut& out = cur[ko + 1];
    const bool last = (ko == n - 1);
    // every output whose input rows have all arrived; at the end of the stream, all the conv's output rows (its
    // right zero padding lies past the window).  in.abs_base is a multiple of P_in.
    const long long out_q = flush ? c.g.out_len(static_cast<int>(in.rows)) / st.P_out - st.bias
                                  : (in.rows > st.span ? (in.rows - 1 - st.span) / st.P_in + 1 : 0);
    if (out_q <= 0) continue;
    const long long out_rows = out_q * st.P_out;
    const long long out_abs = (in.abs_base / st.P_in + st.bias) * st.P_out;
    if (!last) {
      if (out.abs_base + out.rows != out_abs) { err = "internal: streaming row bookkeeping at step " + std::to_string(k); return false; }
      if (out.rows + out_rows > out.cap) { err = "streaming: window buffer overflow at step " + std::to_string(k); return false; }
    } else {
      // decoder: the tail writes the waveform staging [B, io, max_samples] (fp32); encoder: the output conv writes
      // channels-first latents [B, latent, max_frames] in the caller's dtype
      if (out_rows > (s->enc ? s->max_frames : s->max_samples)) {
        err = s->enc ? "streaming: latent staging overflow" : "streaming: waveform staging overflow";
        return false;
      }
      P.n_out = out_rows;
    }
    StreamGeom sg;
    sg.in_rows = static_cast<int>((in.rows + st.P_in - 1) / st.P_in * st.P_in);   // whole phase groups
    if (sg.in_rows > in.cap) { err = "internal: strided window exceeds its buffer"; return false; }
    if (flush && sg.in_rows > in.rows) {
      // rows of the last partial group past the end of the stream are the conv's zero padding
      if (!in.act_row_bytes) { err = "internal: strided conv without operand tensor"; return false; }
      P.zero.push_back({act_ptr(in, in.rows), nullptr, static_cast<size_t>(sg.in_rows - in.rows) * in.act_row_bytes,
                        static_cast<size_t>(in.cap) * in.act_row_bytes, static_cast<size_t>(B)});
    }
    sg.out_q = static_cast<int>(out_q);
    sg.row_bias = st.bias;
    sg.in_pitch = in.cap;
    sg.raw_pitch = out.cap;
    sg.act_pitch = out.cap;
    StepIO io;
    // skip connection: rows of the residual-source stream aligned with this step's output rows
    const Step& so = steps[ko];
    if (so.residual_from >= 0) {
      const StreamOut& r = cur[so.residual_from + 1];
      const long long rel = out_abs - r.abs_base;
      if (!r.raw_row_bytes || rel < 0 || rel + out_rows > r.rows) { err = "internal: streaming skip rows unavailable at step " + std::to_string(k); return false; }
      io.res = raw_ptr(r, rel);
      sg.res_pitch = r.cap;
    }
    if (st.kind == kWaveInTc && out_rows > in.cap) { err = "internal: head operand overflow"; return false; }
    io.in_act = in.act_row_bytes ? act_ptr(in, 0) : nullptr;
    io.in_raw = in.raw_row_bytes ? raw_ptr(in, 0) : nullptr;
    io.in_rows = in.rows;
    io.in_pitch = in.cap;
    io.in_row0 = 0;                                          // edge kernels: the clip's -3 plus the window's bias of 3
    io.out_rows = out_rows;
    io.out_pitch = out.cap;
    io.out_raw = out.raw_row_bytes ? raw_ptr(out, out.rows) : nullptr;
    io.out_act = out.act_row_bytes ? reinterpret_cast<__nv_bfloat16*>(act_ptr(out, out.rows)) : nullptr;
    io.ext = s->enc ? static_cast<void*>(s->z_stage) : static_cast<void*>(s->wav_stage);
    io.ext_f32 = s->enc ? (out_dtype == KVAE_F32) : 1;
    io.cf_ld = s->max_frames;
    io.col = s->col;
    io.sg = &sg;
    P.steps.emplace_back();
    if (!prepare_step(p, steps, k, false, B, io, P.steps.back(), err)) return false;
    consumed[st.in_out + 1] = out_q * st.P_in;
    if (!last) out.rows += out_rows;
  }
  // carry: keep the last `keep` rows of every buffer (all of them while a layer is still starved)
  for (size_t j = 0; j < cur.size(); ++j) {
    StreamOut& o = cur[j];
    if (!o.cap) continue;
    const long long keep = flush ? 0 : o.rows - consumed[j];
    const long long drop = o.rows - keep;
    if (drop > 0 && keep > 0 && o.cf) {
      uint8_t* b0 = base + o.off_raw;
      P.carry_cf.push_back({b0, b0 + static_cast<size_t>(drop) * 4, static_cast<size_t>(keep) * 4, static_cast<size_t>(o.cap) * 4,
                            static_cast<size_t>(B) * o.cf});
    } else if (drop > 0 && keep > 0) {
      for (int which = 0; which < 2; ++which) {
        const int rb = which ? o.act_row_bytes : o.raw_row_bytes;
        if (!rb) continue;
        uint8_t* b0 = base + (which ? o.off_act : o.off_raw);
        StreamCarry cdesc{b0, b0 + static_cast<size_t>(drop) * rb, static_cast<unsigned long long>(keep) * rb,
                          static_cast<unsigned long long>(o.cap) * rb};
        if (cdesc.bytes % 16) { err = "internal: carry size not a multiple of 16 bytes"; return false; }
        (keep <= drop ? P.carry : P.carry_overlap).push_back(cdesc);
      }
    }
    o.abs_base += drop;
    o.rows = keep;
  }
  for (const StreamCarry& c : P.carry_overlap)
    if (c.bytes * static_cast<size_t>(B) > s->scratch_bytes) { err = "internal: carry scratch too small"; return false; }
  for (const StreamRegion& c : P.carry_cf)
    if (c.width * c.height > s->scratch_bytes) { err = "internal: carry scratch too small"; return false; }
  if (!P.carry.empty()) {
    if (cudaMalloc(&P.carry_dev, P.carry.size() * sizeof(StreamCarry)) != cudaSuccess) { err = "cudaMalloc(carry table) failed"; return false; }
    if (cudaMemcpy(P.carry_dev, P.carry.data(), P.carry.size() * sizeof(StreamCarry), cudaMemcpyHostToDevice) != cudaSuccess) {
      err = "cudaMemcpy(carry table) failed";
      return false;
    }
  }
  P.after = cur;
  return true;
}

cudaError_t stream_launch_all(kvae_stream* s, PreparedPush& P, int n_frames, int z_f32, cudaStream_t st) {
  kvae_plan* p = s->plan;
  const ConvLayer& c0 = p->convs[p->steps[0].conv];
  for (const StreamRegion& z : P.zero) {
    cudaError_t e = cudaMemset2DAsync(z.dst, z.pitch, 0, z.width, z.height, st);
    if (e != cudaSuccess) return e;
  }
  if (n_frames > 0 && s->enc) {
    // [B, io, n] staging (caller's dtype) -> fp32 rows appended to the sample window
    const StreamOut& o = s->outs[0];
    dim3 grid(std::min(ceil_div(n_frames, 256), 16), s->B * o.cf);
    stream_append_cf_kernel<<<grid, 256, 0, st>>>(s->wav_stage, z_f32, reinterpret_cast<float*>(s->ws + o.off_raw) + P.in_rows0,
                                                  n_frames, o.cap);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ++g_launches;
  } else if (n_frames > 0) {
    // [B, D, n_frames] (staging) -> channels-last rows appended to the input window
    const StreamOut& o = s->outs[0];
    dim3 grid(ceil_div(n_frames, 32), ceil_div(c0.g.Cin, 32), s->B), block(32, 8);
    cf_to_cl_bf16_kernel<<<grid, block, 0, st>>>(s->z_stage, z_f32,
                                                 reinterpret_cast<__nv_bfloat16*>(s->ws + o.off_act + static_cast<size_t>(P.in_rows0) * o.act_row_bytes),
                                                 c0.g.Cin, n_frames, c0.umma ? 0 : 1, o.cap);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ++g_launches;
  }
  for (StepLaunch& S : P.steps) {
    cudaError_t e = launch_step(S, p->convs[p->steps[S.k].conv].g, s->B, s->stream_f16, st);
    if (e != cudaSuccess) return e;
  }
  if (!P.carry.empty()) {
    size_t maxb = 0;
    for (const StreamCarry& c : P.carry) maxb = std::max<size_t>(maxb, c.bytes);
    const int bx = static_cast<int>(std::max<size_t>(1, std::min<size_t>((maxb / 16 + 255) / 256, 8)));
    stream_carry_kernel<<<dim3(bx, static_cast<unsigned>(P.carry.size()), s->B), 256, 0, st>>>(P.carry_dev, static_cast<int>(P.carry.size()));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    ++g_launches;
  }
  for (const StreamCarry& c : P.carry_overlap) {           // rare (pushes shorter than a layer's halo): through scratch
    cudaError_t e = cudaMemcpy2DAsync(s->scratch, c.bytes, c.src, c.pitch, c.bytes, s->B, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(c.dst, c.pitch, s->scratch, c.bytes, c.bytes, s->B, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return e;
  }
  for (const StreamRegion& c : P.carry_cf) {               // a few samples per channel row: through scratch
    cudaError_t e = cudaMemcpy2DAsync(s->scratch, c.width, c.src, c.pitch, c.width, c.height, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(c.dst, c.pitch, s->scratch, c.width, c.width, c.height, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

void stream_zero_initial_rows(kvae_stream* s, cudaStream_t st);

// out_dtype: the encoder's latent dtype (its output conv writes it); the decoder converts its fp32 staging instead
PreparedPush* stream_get(kvae_stream* s, int n_frames, bool flush, int z_dtype, int out_dtype) {
  std::vector<long long> key;
  key.push_back(n_frames); key.push_back(flush ? 1 : 0); key.push_back(z_dtype);
  if (s->enc) key.push_back(out_dtype);
  for (const StreamOut& o : s->outs) key.push_back(o.rows);
  auto it = s->cache.find(key);
  if (it == s->cache.end()) {
    auto P = std::make_unique<PreparedPush>();
    std::string err;
    if (!stream_prepare(s, n_frames, flush, out_dtype, *P, err)) { fail(err); return nullptr; }
    if (s->cache.size() > 64) s->cache.clear();
    it = s->cache.emplace(key, std::move(P)).first;
  }
  return it->second.get();
}

// in: [B, C_in, n_in] (decoder: latents, encoder: samples); out: [B, C_out, *n_out] (decoder: samples, encoder: frames)
int stream_run(kvae_stream* s, const void* in, int in_dtype, int n_in, bool flush, void* out, int out_dtype,
               long long out_capacity, long long* n_out, cudaStream_t st) {
  kvae_plan* p = s->plan;
  for (const ConvLayer& c : p->convs)
    if (!c.set) return fail("plan weights not set (kvae_plan_set_conv / kvae_plan_load_params)");
  for (const SnakeLayer& sn : p->snakes)
    if (!sn.set) return fail("plan SnakeBeta parameters not set");
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail("cannot select device");
  if (n_in < 0 || n_in > s->max_in)
    return fail(s->enc ? "streaming: n_samples out of range (0 .. max_samples)" : "streaming: n_frames out of range (0 .. max_frames)");
  PreparedPush* Pp = stream_get(s, n_in, flush, in_dtype, out_dtype);
  if (!Pp) return -1;
  PreparedPush& P = *Pp;
  if (s->needs_zero) {
    stream_zero_initial_rows(s, st);
    s->needs_zero = false;
  }
  if (P.n_out > out_capacity)
    return fail(s->enc ? "latent buffer too small for this call (kvae_encode_stream_frames tells the size)"
                       : "wav buffer too small for this call (kvae_decode_stream_samples tells the size)");
  const int io = p->arch.io_channels;
  const int D = p->arch.latent_dim;
  const size_t ies = in_dtype == KVAE_F32 ? 4 : 2, oes = out_dtype == KVAE_F32 ? 4 : 2;
  if (n_in > 0)
    KV_CUDA(cudaMemcpyAsync(s->enc ? static_cast<void*>(s->wav_stage) : static_cast<void*>(s->z_stage), in,
                            static_cast<size_t>(s->B) * (s->enc ? io : D) * n_in * ies, cudaMemcpyDeviceToDevice, st));
  if (s->use_graphs) {
    if (!P.graph) {
      // the first call with this geometry runs eagerly (sets kernel attributes, fills caches), the second is captured
      // (captured on a stream of our own: the caller's may be the legacy default stream, which cannot capture)
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      if (st) KV_CUDA(cudaStreamIsCapturing(st, &cs));
      // (the encoder's short pushes move overlapping carries at every deep stage: 2D copies through scratch, which a
      // graph captures like any other copy; the decoder stream runs such calls eagerly, as it always has)
      if (cs == cudaStreamCaptureStatusNone && P.eager_done && (s->enc || P.carry_overlap.empty())) {
        if (!s->cap_stream) KV_CUDA(cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking));
        cudaGraph_t g = nullptr;
        KV_CUDA(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
        cudaError_t e = stream_launch_all(s, P, n_in, in_dtype == KVAE_F32, s->cap_stream);
        cudaError_t e2 = cudaStreamEndCapture(s->cap_stream, &g);
        if (e != cudaSuccess) { if (g) cudaGraphDestroy(g); return cuda_fail(e, "stream capture"); }
        KV_CUDA(e2);
        e = cudaGraphInstantiate(&P.graph, g, 0);
        cudaGraphDestroy(g);
        KV_CUDA(e);
      }
    }
    if (P.graph) {
      KV_CUDA(cudaGraphLaunch(P.graph, st));
    } else {
      KV_CUDA(stream_launch_all(s, P, n_in, in_dtype == KVAE_F32, st));
      P.eager_done = true;
    }
  } else {
    KV_CUDA(stream_launch_all(s, P, n_in, in_dtype == KVAE_F32, st));
  }
  if (P.n_out > 0 && s->enc) {
    // staging [B, D, max_frames] (already in the caller's dtype) -> the caller's buffer [B, D, n]
    KV_CUDA(cudaMemcpy2DAsync(out, P.n_out * oes, s->z_stage, static_cast<size_t>(s->max_frames) * oes, P.n_out * oes,
                              static_cast<size_t>(s->B) * D, cudaMemcpyDeviceToDevice, st));
  } else if (P.n_out > 0) {
    // staging [B, io, n] fp32 -> the caller's buffer [B, io, n] (dtype conversion included)
    const size_t cnt = static_cast<size_t>(s->B) * io * P.n_out;
    if (out_dtype == KVAE_F32) {
      KV_CUDA(cudaMemcpyAsync(out, s->wav_stage, cnt * 4, cudaMemcpyDeviceToDevice, st));
    } else {
      const int blocks = static_cast<int>(std::min<size_t>((cnt + 255) / 256, 148 * 8));
      f32_to_bf16_kernel<<<blocks, 256, 0, st>>>(s->wav_stage, static_cast<__nv_bfloat16*>(out), cnt);
      KV_CUDA(cudaGetLastError());
      ++g_launches;
    }
  }
  s->outs = P.after;
  s->frames_in += n_in;
  s->samples_out += P.n_out;
  if (n_out) *n_out = P.n_out;
  if (flush) {
    stream_reset(s);
    s->needs_zero = true;
  }
  return 0;
}

// decides which kernels serve the steps and sizes the persistent window buffers; max_in: input rows one call takes
// (decoder: latent frames, encoder: samples)
int stream_create(kvae_plan* p, int B, long long max_in, int use_graphs, kvae_stream** out) {
  if (!p || !out) return fail("null argument");
  const bool enc = p->direction == KVAE_ENCODER;
  if (B <= 0 || max_in <= 0) return fail(enc ? "streaming: bad batch / max_samples" : "streaming: bad batch / max_frames");
  if (max_in > (1 << 26)) return fail("streaming: too many input rows per call");
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail("cannot select device");
  const std::vector<Step>& steps = p->steps;
  const int n = static_cast<int>(steps.size());
  auto s = std::make_unique<kvae_stream>();
  s->plan = p; s->enc = enc; s->B = B; s->max_in = max_in; s->use_graphs = use_graphs != 0;
  s->stream_f16 = p->stream_f16;
  s->ratio = p->ratio;
  // output staging: decoder samples, encoder latent frames (the stream's lag is far below 24 frames)
  if (enc) {
    s->max_samples = max_in;
    s->max_frames = static_cast<int>((max_in + 24 * p->ratio) / p->ratio + 1);
  } else {
    s->max_frames = static_cast<int>(max_in);
    s->max_samples = static_cast<long long>(max_in + 24) * p->ratio;
  }
  s->ss.resize(n);
  s->outs.assign(n + 1, StreamOut());
  std::string err;
  const int split = (p->precision == KVAE_PREC_F32) ? 2 : 1;
  const ConvLayer& c0 = p->convs[steps[0].conv];
  if (!enc && !conv_tc(c0, false)) return fail("streaming: needs a tensor-core first layer (latent_dim and channels multiples of 64)");
  // step kinds and geometry
  for (int k = 0; k < n; ++k) {
    const ConvLayer& c = p->convs[steps[k].conv];
    StreamStep& st = s->ss[k];
    st.in_out = k - 1;
    st.kind = step_kind(p, steps, k, false);
    if (st.kind == kRuSecond) continue;
    if (!stream_step_geometry(c.g, st, err)) return fail(err);
    if (st.kind == kDirect)
      return fail("streaming: step " + std::to_string(k) + " has no tensor-core kernel (channels must be multiples of 64; "
                  "the 128-channel tail is required)");
    if (st.kind == kWaveOut && (c.g.Cin != 128)) return fail("streaming: CUDA-core tail needs 128 input channels");
    if (!enc && k == n - 1 && st.kind == kTcConv) return fail("streaming: tensor-core output conv unsupported");
  }
  // rate of every tensor relative to the input rate, keep / init rows from the consumer
  std::vector<double> rates(n + 1, 1.0);
  for (int k = 0; k < n; ++k) rates[k + 1] = static_cast<double>(steps[k].len_num) / steps[k].len_den;
  const long long in_slack = enc ? 24 * p->ratio : 24;
  size_t off = 0;
  auto consumer_of = [&](int j) -> int {   // first step that reads StreamOut j (j = -1: the input)
    for (int k = j + 1; k < n; ++k)
      if (s->ss[k].kind != kRuSecond && s->ss[k].in_out == j) return k;
    return -1;
  };
  // a fused unit at step k writes the tensors of step k+1; its consumer is step k+2 reading StreamOut k+1
  for (int k = 0; k < n; ++k)
    if (s->ss[k].kind != kRuSecond && k > 0 && s->ss[k - 1].kind == kRuSecond) s->ss[k].in_out = k - 1;
  for (int j = -1; j < n - 1; ++j) {
    StreamOut& o = s->outs[j + 1];
    if (j >= 0 && s->ss[j].kind == kRuFused) continue;         // the k7 half of a fused unit produces no tensor
    const int cons = consumer_of(j);
    if (cons < 0) return fail("internal: streaming tensor without consumer");
    const StreamStep& cs = s->ss[cons];
    o.keep = cs.span;
    o.init_rows = cs.bias * cs.P_in;
    const double r = rates[j + 1];
    o.cap = static_cast<long long>(std::ceil(r * (max_in + in_slack))) + o.keep + 64;
    o.cap = (o.cap + 8 * cs.P_in - 1) / (8 * cs.P_in) * (8 * cs.P_in);   // whole phase groups of a strided consumer
    if (enc && j < 0) {
      // channels-first fp32 sample window [B, io, cap]
      o.cf = c0.g.Cin;
      o.raw_row_bytes = 4;
      o.off_raw = off;
      off += align_up(static_cast<size_t>(B) * o.cf * o.cap * 4, 1024);
      continue;
    }
    const int C = (j < 0) ? c0.g.Cin : p->convs[steps[j].conv].g.Cout;
    const bool needs_raw = j >= 0 && steps[j].needs_raw;
    const bool needs_act = j < 0 || steps[j].needs_act;
    if (needs_raw) {
      o.raw_row_bytes = C * (s->stream_f16 ? 2 : 4);
      o.off_raw = off;
      off += align_up(static_cast<size_t>(B) * o.cap * o.raw_row_bytes, 1024);
    }
    if (needs_act) {
      o.act_row_bytes = C * 2 * split;
      o.off_act = off;
      off += align_up(static_cast<size_t>(B) * o.cap * o.act_row_bytes, 1024);
    }
  }
  size_t off_col = 0;
  if (enc && s->ss[0].kind == kWaveInTc) {                      // im2col operand of the head: at most a window of rows
    off_col = off;
    off += align_up(static_cast<size_t>(B) * s->outs[0].cap * 64 * 2, 1024);
  }
  s->ws_bytes = std::max<size_t>(off, 1024);
  size_t max_carry = 1024;
  for (const StreamOut& o : s->outs)
    max_carry = std::max<size_t>(max_carry, static_cast<size_t>(o.keep) * std::max(o.raw_row_bytes, o.act_row_bytes) * std::max(o.cf, 1));
  s->scratch_bytes = max_carry * B;
  KV_CUDA(cudaMalloc(&s->ws, s->ws_bytes));
  KV_CUDA(cudaMemset(s->ws, 0, s->ws_bytes));            // the initial carry rows are zeros (conv left padding)
  if (off_col) s->col = reinterpret_cast<__nv_bfloat16*>(s->ws + off_col);
  KV_CUDA(cudaMalloc(&s->z_stage, static_cast<size_t>(B) * p->arch.latent_dim * s->max_frames * 4));
  KV_CUDA(cudaMalloc(&s->wav_stage, static_cast<size_t>(B) * p->arch.io_channels * s->max_samples * 4));
  KV_CUDA(cudaMalloc(&s->scratch, s->scratch_bytes));
  stream_reset(s.get());
  *out = s.release();
  return 0;
}

void stream_zero_initial_rows(kvae_stream* s, cudaStream_t st) {
  // the carry region of every buffer becomes the conv's left zero padding again
  for (const StreamOut& o : s->outs) {
    if (!o.cap || !o.init_rows) continue;
    if (o.raw_row_bytes)
      cudaMemset2DAsync(s->ws + o.off_raw, static_cast<size_t>(o.cap) * o.raw_row_bytes, 0, static_cast<size_t>(o.init_rows) * o.raw_row_bytes,
                        static_cast<size_t>(s->B) * std::max(o.cf, 1), st);
    if (o.act_row_bytes)
      cudaMemset2DAsync(s->ws + o.off_act, static_cast<size_t>(o.cap) * o.act_row_bytes, 0, static_cast<size_t>(o.init_rows) * o.act_row_bytes, s->B, st);
  }
}
