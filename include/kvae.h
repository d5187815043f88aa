/* kvae.h -- C ABI of libkvae.so, the B200 (sm_100a) implementation of kalle-audio's
 * sigmaVAE / Oobleck autoencoder hot path.
 *
 * The reference (18281818221/kalle-audio) is pure Python and has no FFI of its own; its boundary for
 * this path is the nn.Module surface of stable_audio_tools/models/autoencoders.py.  Each entry point
 * below names the reference interface it stands in for; kalle_audio_b200/ (Python, ctypes) mirrors the
 * module surface on top of these calls.  INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); the library owns only opaque
 *     plan handles (packed weights, per-shape launch descriptors);
 *   - tensors cross the boundary in the reference's layout: [B, C, T], T contiguous; `dtype` is
 *     KVAE_F32 or KVAE_BF16;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy stream);
 *   - return 0 on success, negative on error; kvae_last_error() returns the message for this thread;
 *   - a plan is not thread-safe: one plan per module instance per device (the reference's callers are
 *     single-threaded, SURVEY.md section 8b).
 *   - there is no CPU path: with no sm_100 device every compute entry point fails with an error.
 */
#ifndef KVAE_H_
#define KVAE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KVAE_F32 0
#define KVAE_BF16 1

#define KVAE_ENCODER 0
#define KVAE_DECODER 1

/* precision of the convolution arithmetic inside a plan */
/* KVAE_PREC_BF16: bf16 tensor-core operands (tcgen05 kind::f16), fp32 accumulation in TMEM.  The residual stream is
 *   fp32 in registers / TMEM and stored as fp16 in HBM by inference plans (fp32 in training plans); the decoder's
 *   tail conv multiplies in fp16 with fp32 accumulation.  Waveform error <= 1e-3 against the reference's fp32 output.
 * KVAE_PREC_F32: still on the tensor cores for every conv whose channel counts are multiples of 64 -- both operands
 *   are stored as bf16 (hi | lo) halves and each K chunk is multiplied three times (hi*hi + lo*hi + hi*lo), fp32
 *   accumulation, fp32 residual stream in HBM, fp32 SnakeBeta (range-reduced sine); the io-channel convs and
 *   architectures with other channel counts use fp32 CUDA-core FMAs.  Waveform error <= 1e-5. */
#define KVAE_PREC_BF16 0
#define KVAE_PREC_F32 1

#define KVAE_MAX_STAGES 8

/* Architecture of one OobleckEncoder / OobleckDecoder: the constructor arguments of
 * autoencoders.py:117-125 (encoder) and :151-160 (decoder).  use_snake must be true and
 * antialias_activation false (the only combination the reference's configs use); the Python layer
 * raises NotImplementedError for the others. */
typedef struct kvae_arch {
  int io_channels;                /* in_channels (encoder) / out_channels (decoder)            */
  int channels;                   /* base width, 128                                           */
  int latent_dim;                 /* encoder: channels emitted; decoder: channels consumed     */
  int n_stages;                   /* len(c_mults) == len(strides)                              */
  int c_mults[KVAE_MAX_STAGES];   /* as passed to the constructor (without the implicit 1)     */
  int strides[KVAE_MAX_STAGES];
  int final_tanh;                 /* decoder only                                              */
  int use_nearest_upsample;       /* decoder only: DecoderBlock's Upsample(nearest, x stride) + WNConv1d(k = 2*stride,
                                     padding 'same', bias=False) branch (autoencoders.py:87-96).  Nearest upsampling
                                     followed by a stride-1 conv IS a transposed conv: the plan runs it as
                                     ConvTranspose1d(k = 3*stride - 1, stride, padding = stride, output_padding = 1)
                                     whose taps are sums of the conv's taps (w'[k'] = sum of w[k] over
                                     k = 2s-1-k' .. 3s-2-k' clipped to 0 .. 2s-1), which kvae_plan_conv_info reports
                                     and kvae_plan_set_conv expects ([Cin, Cout, 3*stride - 1]).  Inference only. */
} kvae_arch;

typedef struct kvae_plan kvae_plan;

int kvae_version(void);
const char* kvae_last_error(void);
/* number of CUDA devices with compute capability 10.x visible to the library (0 => no compute). */
int kvae_device_count(void);
/* kernels launched by this thread through the library since the last reset (bench.py's gpu_launches). */
long long kvae_launch_count(int reset);

/* ---- plans: replace OobleckEncoder.__init__/forward (:116-147) and OobleckDecoder (:150-191) ---- */
int kvae_plan_create(const kvae_arch* arch, int direction, int precision, int device, kvae_plan** out);
void kvae_plan_destroy(kvae_plan* plan);
/* Layers are indexed in the reference's module (= state_dict) order. */
int kvae_plan_num_convs(const kvae_plan* plan);
int kvae_plan_num_snakes(const kvae_plan* plan);
/* shape of conv `idx`: kind (0 Conv1d / 1 ConvTranspose1d), Cin, Cout, K, stride, dilation, padding, has_bias */
int kvae_plan_conv_info(const kvae_plan* plan, int idx, int info[8]);
int kvae_plan_snake_channels(const kvae_plan* plan, int idx);
/* Folded (weight-norm removed) fp32 weight in torch layout -- Conv1d [Cout,Cin,K], ConvTranspose1d
 * [Cin,Cout,K] -- and optional bias [Cout].  Replaces the per-forward torch._weight_norm hook of
 * dac.nn.layers.WNConv1d / WNConvTranspose1d (call sites autoencoders.py:49,52,76,98,133,141,168,184):
 * the fold happens once at load time and the library re-packs for its kernels. */
int kvae_plan_set_conv(kvae_plan* plan, int idx, const float* w_folded, const float* bias, void* stream);
/* SnakeBeta parameters (blocks.py:313-329): alpha, beta [C] fp32; logscale as in the module. */
int kvae_plan_set_snake(kvae_plan* plan, int idx, const float* alpha, const float* beta, int logscale,
                        void* stream);

/* Scratch the caller must provide for a (B, T) problem; T is the INPUT length (latent frames for a
 * decoder, audio samples for an encoder). */
size_t kvae_workspace_bytes(kvae_plan* plan, int B, long long T);
/* OobleckDecoder.forward (:190): z [B, latent_dim, T] -> wav [B, io_channels, T*prod(strides)]. */
int kvae_decode(kvae_plan* plan, const void* z, int z_dtype, void* wav, int wav_dtype, int B, long long T,
                void* workspace, size_t workspace_bytes, void* stream);
/* OobleckEncoder.forward (:146): wav [B, io_channels, L] -> lat [B, latent_dim, L/prod(strides)]. */
int kvae_encode(kvae_plan* plan, const void* wav, int wav_dtype, void* lat, int lat_dtype, int B, long long L,
                void* workspace, size_t workspace_bytes, void* stream);
/* Ragged batches -- what the reference gets by calling the module once per clip (pretransform iterate_batch,
 * autoencoders.py:287-300; the per-item encode of twj_dataset.py:239): clip b holds valid_len[b] <= T valid input
 * positions and is zero-padded to T by the caller; valid_len is a HOST array of B ints.  The library re-creates the
 * reference's end-of-clip zero padding per clip inside every layer, so the first kvae_plan_out_length(valid_len[b])
 * output positions of clip b equal the stand-alone call on that clip -- including audio lengths that are not
 * multiples of the ratio, where the reference's strided convs floor; the rest of its output row is unspecified.
 * For the encoder T must still be a multiple of prod(strides) (pad up); valid_len need not be. */
int kvae_decode_ragged(kvae_plan* plan, const void* z, int z_dtype, void* wav, int wav_dtype, int B, long long T,
                       const int* valid_len, void* workspace, size_t workspace_bytes, void* stream);
int kvae_encode_ragged(kvae_plan* plan, const void* wav, int wav_dtype, void* lat, int lat_dtype, int B, long long L,
                       const int* valid_len, void* workspace, size_t workspace_bytes, void* stream);
/* Output length of a pass over an input of length T by the reference's own arithmetic (every conv floors,
 * L_out = (L + 2p - d(K-1) - 1)/s + 1): T*prod(strides) for a decoder; for an encoder floor-ish, and not simply
 * T / prod(strides) when a stride is odd (the stride-5 stage of the 12.5 Hz models maps 159 rows to 32). */
long long kvae_plan_out_length(const kvae_plan* plan, long long T);
/* Dataset-side preprocessing of twj_dataset.py:231-235 for a batch: B mono fp32 clips stored back to back in `wav`
 * (clip b = wav[offsets[b] .. +lens[b]); offsets / lens are DEVICE arrays) -> out [B, channels, L_pad] fp32 =
 * librosa.util.normalize(clip) * gain (peak normalisation; gain 0.95 there) copied to every channel (the stereo
 * duplication of :235) and zero-padded.  scratch: >= 4*B bytes. */
int kvae_prep_mono_clips(const float* wav, const long long* offsets, const int* lens, int B, long long L_pad,
                         int channels, float gain, float* out, void* scratch, void* stream);
/* ---- stateful streaming decode: replaces decode_audio(chunked=True, chunk_size, overlap) (autoencoders.py:499-560)
 * for callers that receive latents incrementally (infer_stream-style).  The reference re-decodes overlapping windows
 * (1.33x the work at 128/32); a kvae_stream keeps every layer's input tail between calls instead (persistent
 * per-layer halo state), so every row of every layer is computed once and the concatenated output equals
 * kvae_decode of the whole sequence bit for bit.  One stream = B clips advancing in lockstep; not thread-safe.
 *   begin   allocates the window buffers for pushes of up to max_frames latent frames; use_graphs != 0 replays
 *           calls of a geometry seen before as one CUDA graph (constant-hop streams: one graph launch per hop)
 *   samples how many samples per channel the next push of n_frames (or, end != 0, the end call) will emit
 *   push    z [B, latent_dim, n_frames] -> wav [B, io_channels, *n_samples] (packed with that length); the output
 *           trails the input by kvae_decode_stream_lookahead samples (the decoder's receptive field, 10 latent
 *           frames for the SAO / 12.5 Hz strides), so early pushes may emit nothing
 *   end     emits the remaining samples (right edge zero-padded like the unchunked decode) and resets the stream
 * Decoder plans whose layers all run on the tensor-core kernels (latent_dim / channels multiples of 64, 128-channel
 * tail), bf16 or fp32 mode; other architectures get an error (the Python layer then streams by exact-context windows). */
typedef struct kvae_stream kvae_stream;
int kvae_decode_stream_begin(kvae_plan* plan, int B, int max_frames, int use_graphs, kvae_stream** out);
long long kvae_decode_stream_samples(kvae_stream* s, int n_frames, int end);
long long kvae_decode_stream_lookahead(const kvae_stream* s);
int kvae_decode_stream_push(kvae_stream* s, const void* z, int z_dtype, int n_frames, void* wav, int wav_dtype,
                            long long wav_capacity, long long* n_samples, void* stream);
int kvae_decode_stream_end(kvae_stream* s, void* wav, int wav_dtype, long long wav_capacity, long long* n_samples,
                           void* stream);
void kvae_decode_stream_destroy(kvae_stream* s);
/* ---- stateful streaming encode: the same engine in the encoder's direction, for callers that receive audio
 * incrementally (live input to a speech LM) or encode long recordings in bounded memory.  Every layer keeps the tail
 * of its own input; the strided convs keep whole groups of `stride` rows, so the emitted latents equal kvae_encode of
 * the whole clip bit for bit, and for a length L that is not a multiple of the ratio they are the
 * kvae_plan_out_length(L) frames of the reference's floor arithmetic (kvae_encode_ragged).
 *   begin      window buffers for pushes of up to max_samples samples; use_graphs as for the decoder stream
 *   frames     how many latent frames the next push of n_samples (or, end != 0, the end call) will emit
 *   lookahead  samples past a frame's last sample that must have arrived before the frame is emitted (the encoder's
 *              right receptive field: 14 885 for the SAO strides, 9 925 for the 12.5 Hz strides)
 *   push       wav [B, io_channels, n_samples] -> lat [B, latent_dim, *n_frames] (packed with that length)
 *   end        emits the remaining frames (right edge zero-padded like the whole-clip encode) and resets the stream
 *   destroy    frees the stream
 * Encoder plans whose every step has a tensor-core kernel (channels / latent_dim multiples of 64, a 128-channel head),
 * bf16 or fp32 mode; other architectures get an error from begin. */
int kvae_encode_stream_begin(kvae_plan* plan, int B, long long max_samples, int use_graphs, kvae_stream** out);
long long kvae_encode_stream_frames(kvae_stream* s, long long n_samples, int end);
long long kvae_encode_stream_lookahead(const kvae_stream* s);
int kvae_encode_stream_push(kvae_stream* s, const void* wav, int wav_dtype, long long n_samples, void* lat,
                            int lat_dtype, long long lat_capacity, long long* n_frames, void* stream);
int kvae_encode_stream_end(kvae_stream* s, void* lat, int lat_dtype, long long lat_capacity, long long* n_frames,
                           void* stream);
void kvae_encode_stream_destroy(kvae_stream* s);
/* kvae_encode with the sigma-VAE sample fused into the last conv's epilogue: lat [B, latent_dim, T] as kvae_encode,
 * and z [B, D, T] = lat[:, :D] + std * noise (sample(mean, 'fix') of model_sigmaVAE.py:187-213 applied to the mean
 * half of the encoder output, D = latent_dim / 2 for the mean | scale layout of twj_dataset.py:251), evaluated on the
 * STORED latents with torch's two roundings, so z is bit-identical to the two-step form.  noise, z and lat share
 * lat_dtype.  Tensor-core encoder plans only (kvae_plan_fused_sample_supported). */
int kvae_encode_sample(kvae_plan* plan, const void* wav, int wav_dtype, void* lat, void* z, const void* noise,
                       int lat_dtype, int D, float std, int B, long long L, void* workspace, size_t workspace_bytes,
                       void* stream);
int kvae_plan_fused_sample_supported(const kvae_plan* plan);
/* algorithmic FLOPs of one pass (2*MACs of every conv, all taps counted; SURVEY.md section 8d) */
double kvae_plan_flops(const kvae_plan* plan, int B, long long T);

/* Per-step device timing for the roofline report: after kvae_plan_profile(plan, 1) every run records a CUDA
 * event between steps on the launching stream; kvae_plan_step_profile waits for the last recorded run and
 * returns, per convolution step, its duration (ms), algorithmic FLOPs and whether it ran on tcgen05.
 * Returns the number of steps (> 0) or a negative error. */
int kvae_plan_profile(kvae_plan* plan, int enable);
int kvae_plan_step_profile(kvae_plan* plan, float* ms, double* flops, int* tensor_core, int max_steps);

/* ---- layer-level entry points (module-level drop-ins and tests) ---- */
/* SnakeBeta.forward (blocks.py:331-339) on [B, C, T]. */
int kvae_snake_fwd(const void* x, void* y, const float* alpha, const float* beta, int logscale, int B, int C,
                   long long T, int dtype, void* stream);
/* torch.nn.utils.weight_norm fold, dim=0: w[i,:] = v[i,:] * g[i] / ||v[i,:]||  (fp32). */
int kvae_weight_norm_fold(const float* v, const float* g, float* w, int dim0, int inner, void* stream);
/* WNConv1d.forward / WNConvTranspose1d.forward on [B, Cin, T] with a folded fp32 weight in torch
 * layout; fp32 arithmetic; x and y of `dtype`.  transposed = 1 selects ConvTranspose1d.  The weight is packed into
 * scratch, then the layer runs as kvae_conv1d_win_fwd's engine 0 over all output rows. */
int kvae_conv1d_fwd(const void* x, void* y, const float* w_folded, const float* bias, int transposed, int B,
                    int Cin, int Cout, long long T, int K, int stride, int dilation, int padding, int dtype,
                    void* scratch, size_t scratch_bytes, void* stream);
size_t kvae_conv1d_scratch_bytes(int Cin, int Cout, int K);
/* Whether the tcgen05 engines of kvae_conv1d_win_fwd take this layer (channel counts that are multiples of 64). */
int kvae_conv1d_tc_supported(int Cin, int Cout, int K, int stride, int dilation, int transposed);

/* ---- training step (BASELINE config 5) --------------------------------------------------------------
 * The reference trains the autoencoder with plain autograd through the module tree
 * (AutoencoderTrainingWrapper.training_step, stable_audio_tools/training/autoencoders.py:221-352: encode ->
 * bottleneck -> decode -> losses -> manual_backward -> optimizer step); these entry points are what the
 * autograd nodes of OobleckEncoder / OobleckDecoder, VAEBottleneck and the loss bind to.
 *
 * Parameters and gradients cross the boundary as ONE flat fp32 buffer per plan whose segments follow
 * module.parameters() order: per layer [alpha][beta] of its SnakeBeta (blocks.py:313-329), then the conv's
 * [bias][weight_g][weight_v] (old-style torch weight_norm, dac.nn.layers.WNConv1d/WNConvTranspose1d). */
long long kvae_plan_param_count(const kvae_plan* plan);
/* segment sizes (floats) of the flat buffer, in order; returns the number of segments */
int kvae_plan_param_sizes(const kvae_plan* plan, long long* sizes, int max_segments);
/* Folds weight norm and packs every layer from the flat buffer (replaces kvae_plan_set_conv / _set_snake, one
 * call per optimizer step).  train != 0 also packs the operands of the data-gradient kernels. */
int kvae_plan_load_params(kvae_plan* plan, const float* params, int snake_logscale, int train, void* stream);
/* workspace of a training pass: every layer's pre-activation stream and operand stay live for the backward
 * pass, plus the backward scratch */
size_t kvae_train_workspace_bytes(kvae_plan* plan, int B, long long T);
/* OobleckEncoder.forward / OobleckDecoder.forward under autograd: same result as kvae_encode / kvae_decode,
 * activations saved in `workspace` (must stay untouched until kvae_backward) */
int kvae_forward_train(kvae_plan* plan, const void* x, int x_dtype, void* y, int y_dtype, int B, long long T,
                       void* workspace, size_t workspace_bytes, void* stream);
/* Backward of that pass: gy [B, C_out, T_out] -> grads (flat, overwritten; kvae_plan_param_count floats) and,
 * when gx != NULL, gx [B, C_in, T].  x is the forward input.  params != NULL (the flat buffer the pass ran
 * with) finishes with the weight-norm backward so the weight_g / weight_v segments hold d g / d v; with
 * params == NULL the weight_v segments hold the gradient of the FOLDED weight and weight_g is zero. */
int kvae_backward(kvae_plan* plan, const void* x, int x_dtype, const void* gy, int gy_dtype, void* gx, int gx_dtype,
                  int B, long long T, void* workspace, size_t workspace_bytes, float* grads, const float* params,
                  void* stream);
/* torch.nn.utils.weight_norm backward, dim=0: (dw, v, g) -> (dv, dg); dv may alias dw. */
int kvae_weight_norm_bwd(const float* v, const float* g, const float* dw, float* dv, float* dg, int dim0, int inner,
                         void* stream);
/* SnakeBeta backward on channels-last rows [rows, C] fp32 (blocks.py:301-302 differentiated): gx, d alpha,
 * d beta (overwritten).  scratch: >= 2*C floats. */
int kvae_snake_bwd(const float* x, const float* gy, float* gx, const float* alpha, const float* beta, int logscale,
                   float* d_alpha, float* d_beta, long long rows, int C, void* scratch, void* stream);
/* vae_sample backward (bottleneck.py:51-62): gz (may be NULL) and the scalar gkl (device fp32, may be NULL)
 * -> gmean, gscale. */
int kvae_vae_sample_bwd(const void* mean, const void* scale, const void* noise, const void* gz, const float* gkl,
                        void* gmean, void* gscale, int B, int D, long long T, int dtype, void* stream);
/* sigma-VAE reconstruction term: *loss = sum_i [0.5 ((x_i - xhat_i)/sigma)^2 + log sigma + 0.5 log 2 pi] / B and,
 * when gxhat != NULL, its gradient w.r.t. xhat.  scratch: >= 8*1024 bytes.  (The reference's sigma-vae symlink
 * dangles; SURVEY.md section 8c defines this form.) */
int kvae_gaussian_nll(const void* x, const void* xhat, void* gxhat, float* loss, int B, size_t per_item,
                      float log_sigma, int dtype, void* scratch, void* stream);
/* torch.optim.AdamW step over a flat fp32 buffer; grads are multiplied by grad_scale first (1/world_size
 * after a summing all-reduce).  step counts from 1. */
int kvae_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n, float lr,
                    float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream);

/* ---- Multi-resolution STFT loss of the autoencoder training wrapper (SURVEY section 8f item 4, loss half) ----
 * training/losses/auraloss.py: MultiResolutionSTFTLoss (443-531) / SumAndDifferenceSTFTLoss (534-606) over STFTLoss
 * (220-441: torch.stft with reflect padding and a periodic Hann window, magnitude sqrt(clamp(re^2 + im^2, 1e-8)),
 * w_sc * spectral convergence + w_log_mag * L1 of the log magnitudes) with the optional A-weighting pre-filter
 * (FIRFilter "aw", 70-162), as instantiated at training/autoencoders.py:123-129 and called at :163 as
 * module(input = reals, target = decoded).  input / target [B, C, T] of `dtype`; loss: one device float;
 * grad_input / grad_target: optional device fp32 [B, C, T] (d loss / d argument, overwritten).
 *   fft_sizes / hop_sizes: n_res host ints (fft sizes powers of two in [8, 2048]); windows: device fp32, the n_res
 *   analysis windows back to back, each ALREADY zero-padded to its fft size (torch.stft centres a shorter window);
 *   fir_taps: device fp32 [n_taps] (odd, <= 129) or NULL for no pre-filter; sum_diff = 1: stereo sum / difference
 *   signals weighted w_sum / w_diff and averaged (C must be 2), 0: every channel is a signal (view(-1, T)).
 * Nothing of spectrogram size is stored: the backward pass transforms the frames again. */
size_t kvae_mrstft_scratch_bytes(int B, int C, long long T, int n_res, int sum_diff, int want_grad);
int kvae_mrstft_loss(const void* input, const void* target, int B, int C, long long T, int dtype, int n_res,
                     const int* fft_sizes, const int* hop_sizes, const float* windows, const float* fir_taps, int n_taps,
                     int sum_diff, float w_sum, float w_diff, float w_sc, float w_log_mag, float* loss, float* grad_input,
                     float* grad_target, void* scratch, size_t scratch_bytes, void* stream);

/* ---- BigVGANFlowVAE inference path (backup/flows.py:396-529: the reference's 12.5 Hz VAE) -- leaf kernels ----
 * Activation1d of the AMP blocks (alias_free_torch, un-vendored; flows.py:266, 312, 443): x2 Kaiser-sinc upsampling
 * (replicate padding) -> Snake (beta == NULL: x + sin^2(a x)/a) or SnakeBeta (x + sin^2(a x)/b) -> low-pass and x2
 * decimation, in ONE pass over [B, C, T].  filt_up / filt_down: the module's 12-tap `upsample.filter` /
 * `downsample.lowpass.filter` buffers (device fp32). */
int kvae_aa_act_fwd(const void* x, void* y, const float* alpha, const float* beta, int logscale, const float* filt_up,
                    const float* filt_down, int B, int C, long long T, int dtype, void* stream);
/* Window form of kvae_aa_act_fwd for the streaming decoder (BigVGANStreamingDecoder; every Activation1d of flows.py:266,
   312, 443).  x holds the absolute rows [x0, x0 + nx) of each of the B*C rows at pitch ldx; outputs t in [o0, o1) are
   written to y + row * ldy + (t - o0).  Replicate padding happens only at absolute row 0 and, when t_end >= 0, at the
   stream end t_end; t_end < 0 = the stream continues.  Rows [max(0, o0 - 5), min(o1 + 5, t_end)) must lie in the
   window.  Per-sample arithmetic is the whole-row kernel's: kvae_aa_act_fwd is the case x0 = o0 = 0, o1 = t_end = T.
   Replicate padding at the start only ever touches rows < 0, and outputs o >= 5 read no such row: a window whose
   outputs all lie at o0 >= 5 may therefore be addressed from any origin that keeps o0 >= 5 (the streaming decoder
   passes window-relative rows, x0 = 0, o0 = 5, so that its captured launches repeat from push to push). */
int kvae_aa_act_win_fwd(const void* x, long long ldx, long long x0, long long nx, void* y, long long ldy, long long o0,
                        long long o1, long long t_end, const float* alpha, const float* beta, int logscale,
                        const float* filt_up, const float* filt_down, int B, int C, int dtype, void* stream);
/* Ragged form of kvae_aa_act_fwd for BigVGANFlowVAE batches of clips with different lengths (every Activation1d of
   flows.py:266, 312, 443 under extract_latents / inference_from_latents(valid_len=...)).  valid_len: HOST array of
   B <= 64 ints in [1, T].  Each (b, c) row is its own signal ending at valid_len[b]: replicate padding happens at that
   end, so outputs t < valid_len[b] equal kvae_aa_act_fwd on the row's first valid_len[b] samples bit for bit, and
   outputs t >= valid_len[b] are stored as 0 (a following conv reads them as its zero padding).  Rows of x past a
   clip's end are never read. */
int kvae_aa_act_ragged_fwd(const void* x, void* y, const float* alpha, const float* beta, int logscale,
                           const float* filt_up, const float* filt_down, int B, int C, long long T,
                           const int* valid_len, int dtype, void* stream);
/* y[b, c, t] = 0 for t in [valid_len[b], T): channels-first [B, C] rows of T samples at pitch ldy >= T, valid_len a
   HOST array of B <= 64 ints in [0, T].  Re-creates a clip's end-of-signal zero padding inside a padded BigVGANFlowVAE
   batch where the next op reads past the clip's end (the input, the input of a non-causal ConvTranspose1d
   (flows.py:336-391), the inputs of the encoder's convs (:139-189), the final output). */
int kvae_zero_tail_cf(void* y, int B, int C, long long T, long long ldy, const int* valid_len, int dtype, void* stream);
/* The conv layers of BigVGANFlowVAE (Conv1d / ConvTranspose1d, flows.py:336-391, 566-620; the encoder's strided
   Conv1d).  kvae_conv1d_pack packs a folded fp32 weight ([Cout, Cin, K], transposed: [Cin, Cout, K]) for engine
   0 = CUDA cores fp32, 1 = tcgen05 bf16, 2 = tcgen05 bf16 x 3 split (<= 1e-5), into kvae_conv1d_packed_bytes.
   kvae_conv1d_win_fwd runs the conv (padding `padding`) of the T-row input x ([B, Cin] rows at pitch ldx) with those
   weights and writes only its output rows [o0, o1) to y ([B, Cout] rows at pitch ldy, row o0 first).  The whole layer is the range [0, T_out)
   of a contiguous input; a shorter range [0, T_keep) is the causal Conv1d / ConvTranspose1d of backup/flows.py
   (:607-608 left padding d (K - 1); :388-389 last `stride` samples dropped), the symmetric layer truncated.  The
   streaming decoder runs windows of a stream (o0 > 0).  A strided Conv1d takes o0 = 0 only.  tcgen05 engines need
   kvae_conv1d_tc_supported and o0 and o1 multiples of the stride of a transposed conv; o1 may then reach T_out rounded
   up to a whole stride group (a non-causal ConvTranspose1d with odd K - stride), the rows past T_out being the conv
   continued over zero input rows.  A strided Conv1d takes any input length: its input is staged rounded up to whole
   stride groups, zero rows past T, so the tcgen05 engines need kvae_conv1d_stream_scratch_bytes(B, Cin, T, stride,
   engine) of scratch (kvae_conv1d_win_scratch_bytes(B, Cin, T, engine) for the other layers, the same value). */
size_t kvae_conv1d_packed_bytes(int Cin, int Cout, int K, int engine);
int kvae_conv1d_pack(const float* w, int transposed, int Cin, int Cout, int K, int engine, void* packed,
                     size_t packed_bytes, void* stream);
size_t kvae_conv1d_win_scratch_bytes(int B, int Cin, long long T, int engine);
int kvae_conv1d_win_fwd(const void* x, long long ldx, void* y, long long ldy, const void* packed, const float* bias,
                        int transposed, int B, int Cin, int Cout, long long T, int K, int stride, int dilation,
                        int padding, long long o0, long long o1, int dtype, int engine, void* scratch,
                        size_t scratch_bytes, void* stream);
/* Stream form of the (non-transposed) Conv1d of BigVGANFlowVAE's encoder, strides 1 to 8 (BigVGANStreamingEncoder;
   flows.py:139-189).  x holds the stream rows [x0, x0 + nx) ([B, Cin] rows at pitch ldx); x0 must be a multiple of
   the stride.  The conv runs with the layer's own padding: rows < 0 read as zero and, when t_end >= 0 (the stream
   end), so do rows >= t_end.  Output rows [o0, o1) are written to y ([B, Cout] rows at pitch ldy, row o0 first).
   Every input row a requested output reads must lie in the window, below 0 or at or past t_end; the call checks this
   and refuses otherwise before any device access.  Per output the kernels sum the same taps in the same order as the
   whole-layer call, so the rows equal kvae_conv1d_win_fwd over [0, T_out) of the whole input bit for bit on every
   engine.  The tcgen05 engines copy the window rounded up to whole stride groups, with zero rows past nx, into
   kvae_conv1d_stream_scratch_bytes of scratch.  When no requested output reads a row below the window start, the
   rows may be given window-relative (x0 = 0, o0 and o1 less x0 / stride, t_end less x0): the result is the same,
   and a captured graph replays with the same arguments on every push. */
size_t kvae_conv1d_stream_scratch_bytes(int B, int Cin, long long nx, int stride, int engine);
int kvae_conv1d_stream_fwd(const void* x, long long ldx, long long x0, long long nx, void* y, long long ldy,
                           long long o0, long long o1, long long t_end, const void* packed, const float* bias,
                           int B, int Cin, int Cout, int K, int stride, int dilation, int padding,
                           int dtype, int engine, void* scratch, size_t scratch_bytes, void* stream);
/* op 0: nn.LeakyReLU(param) (flows.py:181-217), op 1: tanh (:527) */
int kvae_unary_fwd(const void* x, void* y, size_t n, int op, float param, int dtype, void* stream);
/* out = alpha*a + beta*b: the residual adds of the AMP blocks (:283) and their average (:519-520) */
int kvae_axpby(const void* a, const void* b, void* out, size_t n, float alpha, float beta, int dtype, void* stream);
/* z = mean + noise * exp(logs) (:500-501) */
int kvae_gauss_sample(const void* mean, const void* logs, const void* noise, void* out, size_t n, int dtype, void* stream);

/* ---- BigVGANFlowVAE decoder backward (BigVGANFlowVAE.decode_with_grad: autograd of inference_from_latents,
 * flows.py:498-529, through AMPBlock1 / AMPBlock2 :243-335) ----
 * Backward of kvae_aa_act_fwd over whole rows (alias_free_torch Activation1d, flows.py:266, 312, 443): from the saved
 * input x and gy ([B, C, T], both of `dtype`) gx (same dtype) and the per-channel fp32 dalpha, dbeta (SnakeBeta; Snake,
 * beta == NULL: dalpha only, both terms of a = b).  The double-rate signal is rebuilt from x tile by tile, as the
 * forward builds it.  dalpha / dbeta are reduced from one partial per (row, 1024-output tile) in a fixed order: two
 * calls give the same bits.  dalpha == NULL (frozen parameters): gx only, no scratch.  scratch:
 * kvae_aa_act_bwd_scratch_bytes. */
size_t kvae_aa_act_bwd_scratch_bytes(int B, int C, long long T);
int kvae_aa_act_bwd(const void* x, const void* gy, void* gx, const float* alpha, const float* beta, int logscale,
                    const float* filt_up, const float* filt_down, float* dalpha, float* dbeta, int B, int C, long long T,
                    int dtype, void* scratch, size_t scratch_bytes, void* stream);
/* Backward of kvae_unary_fwd: op 0 (LeakyReLU, :181-217) takes the forward's input t = x, gx = gy * (x > 0 ? 1 :
 * param); op 1 (tanh, :527) takes the forward's output t = y, gx = gy * (1 - y^2). */
int kvae_unary_bwd(const void* t, const void* gy, void* gx, size_t n, int op, float param, int dtype, void* stream);
/* Backward of the Gaussian sample (:500-501) on the latents x = [B, 2 D, T] (mean | logs): gz and noise [B, D, T];
 * gx[:, :D] = gz, gx[:, D:] = gz * noise * exp(logs).  (The residual adds and the AMP average differentiate through
 * kvae_axpby itself.) */
int kvae_gauss_sample_bwd(const void* x, const void* noise, const void* gz, void* gx, int B, int D, long long T, int dtype,
                          void* stream);
/* Backward of a conv layer of kvae_conv1d_fwd / kvae_conv1d_win_fwd: the stand-alone WNConv1d / WNConvTranspose1d
 * (autograd of F.conv1d / F.conv_transpose1d and weight_norm) and the conv layers of BigVGANFlowVAE (Conv1d :566-620,
 * ConvTranspose1d :336-391, and the encoder's Conv1d_S :139-172, whose downsampling convs have stride 2 .. 8).  The
 * layer geometry is the forward's: padding >= 0 on both sides, a causal layer being the symmetric-padded one truncated;
 * a strided Conv1d and a ConvTranspose1d have dilation 1; the tcgen05 engines take padding <= d (K - 1).  gy: the gradient of
 * the layer's output rows [0, T_gy) ([B, Cout, T_gy] of `dtype`); rows past T_gy (a causal layer's dropped rows) have
 * none.  x: the layer's input [B, Cin, T].  w: the folded fp32 weight.  Each product is optional (NULL = skipped):
 *   gx [B, Cin, T] (`dtype`)  the forward conv kernels under the data-gradient geometry (kvae_conv1d_dgrad_form) on
 *                             `engine`: 0 = CUDA cores fp32, 1 = tcgen05 bf16, 2 = tcgen05 bf16 x 3.  A strided
 *                             Conv1d's is a ConvTranspose1d continued to all T input rows (rows past its natural
 *                             length are rows the forward read); the tcgen05 engines compute it in whole stride groups,
 *                             through scratch when T is not a multiple of the stride;
 *   dv (fp32, torch layout)   with g != NULL the gradients of weight_v and (dg) weight_g of the weight norm (v, g: the
 *                             fp32 parameters), else of the plain weight.  Engine 1: tcgen05 weight gradient from
 *                             channels-last bf16 copies of x (rounded up to whole stride groups
 *                             with zero rows) and gy; engines 0 and 2: fp32 CUDA cores;
 *   dbias [Cout] (fp32).
 * A frozen layer (dv = dbias = NULL) runs no weight-gradient kernel.  tcgen05 engines: kvae_conv1d_tc_supported.
 * scratch: kvae_conv1d_win_bwd_scratch_bytes. */
size_t kvae_conv1d_win_bwd_scratch_bytes(int transposed, int B, int Cin, int Cout, long long T, long long T_gy, int K,
                                         int stride, int engine);
int kvae_conv1d_win_bwd(const void* x, const void* gy, long long T_gy, const float* w, const float* v, const float* g,
                        void* gx, float* dv, float* dg, float* dbias, int transposed, int B, int Cin, int Cout, long long T,
                        int K, int stride, int dilation, int padding, int dtype, int engine, void* scratch,
                        size_t scratch_bytes, void* stream);
/* The data-gradient geometry kvae_conv1d_win_bwd runs: gx = rows [0, T) of the Conv1d (out[0] input channels, out[1]
 * output channels, stride out[2], dilation out[3], left padding out[4], zero rows past the end of gy) of gy with the
 * layer's weight transposed to [Cin, Cout, K] with its taps reversed (out[5] = 1: a Conv1d of stride 1, new left
 * padding d (K - 1) - padding, negative when padding > d (K - 1): gx then reads gy ahead), or as it is (out[5] = 0: a
 * ConvTranspose1d, stride s, padding p). */
int kvae_conv1d_dgrad_geom(int transposed, int Cin, int Cout, int K, int stride, int dilation, int padding, int out[6]);
/* The same for every layer kvae_conv1d_win_bwd accepts, the kind of conv first: gx = rows [0, T) of the Conv1d
 * (out[0] = 0, as kvae_conv1d_dgrad_geom's out[0 .. 5] in out[1 .. 6]) or the ConvTranspose1d (out[0] = 1: a strided
 * Conv1d's; out[1] input channels = the layer's Cout, out[2] output channels = the layer's Cin, stride out[3], dilation
 * out[4] = 1, padding out[5] = the layer's, out[6] = 0: the layer's weight as it is, read as [out[1], out[2], K]) of gy,
 * continued past its natural length to T rows (torch's output_padding T - that length). */
int kvae_conv1d_dgrad_form(int transposed, int Cin, int Cout, int K, int stride, int dilation, int padding, int out[7]);

/* ---- BigVGANFlowVAE flow (backup/flows.py:613-792, the VITS ResidualCouplingBlock with mean_only coupling layers and
 * an unconditioned WN) ----
 * Elementwise steps between the flow's convolutions (which run through kvae_conv1d_win_fwd / kvae_conv1d_win_bwd).
 * Tensors are contiguous [B, C, T] of `dtype` (fp32 or bf16; fp32 arithmetic, one rounding per stored value); x_mask is
 * [B, 1, T] of the same dtype.  Every backward is a pass of its own with no reduction.  A NULL output gradient reads
 * as 0 (an output autograd did not use).
 *
 * torch.split(x, [C/2] * 2, 1)[0] (ResidualCouplingLayer.forward) and torch.flip(x, [1]) (Flip.forward): xs = x, or x
 * with its C channels reversed (flip), and x0 = xs[:, :C/2] as a contiguous [B, C/2, T] copy unless x0 == NULL.  The
 * backward: gx = the reversal (flip) of gxs + (gx0 on the first C/2 channels). */
int kvae_flow_split(const void* x, void* xs, void* x0, int B, int C, long long T, int flip, int dtype, void* stream);
int kvae_flow_split_bwd(const void* gxs, const void* gx0, void* gx, int B, int C, long long T, int flip, int dtype,
                        void* stream);
/* h = pre(x0) * x_mask (ResidualCouplingLayer.forward): y = x * mask over C channels; also its backward (gx = gy * mask). */
int kvae_flow_mask(const void* x, const void* mask, void* y, int B, int C, long long T, int dtype, void* stream);
/* commons.fused_add_tanh_sigmoid_multiply(x_in, 0, H) (WN.forward): acts [B, H, T] = tanh(a[:, :H]) sigmoid(a[:, H:])
 * of a [B, 2H, T].  The backward reads the saved a and writes both halves of ga [B, 2H, T]. */
int kvae_wn_gate_fwd(const void* a, void* acts, int B, int H, long long T, int dtype, void* stream);
int kvae_wn_gate_bwd(const void* a, const void* g, void* ga, int B, int H, long long T, int dtype, void* stream);
/* WN.forward's residual / skip update of one layer from rs = res_skip_layers[i](acts) and the running skip sum (skip ==
 * NULL: 0, the first layer).  last == 0 (rs [B, 2H, T]): x_out = (x + rs[:, :H]) * mask, skip_out = skip + rs[:, H:].
 * last != 0 (rs [B, H, T]): skip_out = (skip + rs) * mask, WN's output (x, x_out unused).  The backward from g_xout and
 * g_skipout: gx = g_xout * mask and grs = (g_xout * mask | g_skipout), or for the last layer grs = g_skipout * mask; the
 * skip input's gradient is g_skipout (g_skipout * mask for the last layer), written to gskip unless it is NULL. */
int kvae_wn_update_fwd(const void* x, const void* rs, const void* skip, const void* mask, void* x_out, void* skip_out,
                       int B, int H, int last, long long T, int dtype, void* stream);
int kvae_wn_update_bwd(const void* g_xout, const void* g_skipout, const void* mask, void* gx, void* grs, void* gskip,
                       int B, int H, int last, long long T, int dtype, void* stream);
/* ResidualCouplingLayer.forward's update (mean_only: logs = 0, the log-determinant 0) followed by Flip: from the layer
 * input x [B, C, T] and m = post(h) [B, C/2, T], mm = m * mask and x1' = mm + x1 * mask (reverse == 0) or (x1 - mm) *
 * mask (reverse != 0); y = cat(x0, x1'), written with its channels reversed when flip, and y0 = y[:, :C/2] as a
 * contiguous copy (the next layer's `pre` input) unless y0 == NULL.  The backward from gy and gy0 (either may be NULL):
 * gx [B, C, T] and gm [B, C/2, T]; it reads neither x nor m. */
int kvae_flow_coupling_fwd(const void* x, const void* m, const void* mask, void* y, void* y0, int B, int C, long long T,
                           int flip, int reverse, int dtype, void* stream);
int kvae_flow_coupling_bwd(const void* gy, const void* gy0, const void* mask, void* gx, void* gm, int B, int C,
                           long long T, int flip, int reverse, int dtype, void* stream);

/* ---- post-decode tail ---- */
/* audio.to(float32).div(max|audio|).clamp(-1,1).mul(32767).to(int16) -- the peak-normalised PCM conversion every
 * caller of the decoder repeats (infer_0828_sigma.py:298, train_offline.py:302,319); bit-exact with torch's
 * separately rounded ops.  scratch: >= 4 bytes. */
int kvae_pcm16(const void* wav, int dtype, int16_t* out, size_t n, void* scratch, void* stream);

/* kvae_decode with phase 1 of that conversion (the global peak) fused into the tail conv's epilogue -- one atomicMax
 * per warp and tile while the waveform is written -- followed by the conversion pass: wav [B, io, T*ratio] as
 * kvae_decode, pcm = int16 of wav / max|wav| * 32767, bit-exact with kvae_decode + kvae_pcm16 (and so with torch)
 * at one pass over the waveform less.  Tensor-core tail only (kvae_plan_fused_pcm_supported).  scratch: >= 4 bytes. */
int kvae_decode_pcm16(kvae_plan* plan, const void* z, int z_dtype, void* wav, int wav_dtype, int16_t* pcm, int B,
                      long long T, void* workspace, size_t workspace_bytes, void* scratch, void* stream);
int kvae_plan_fused_pcm_supported(const kvae_plan* plan);

/* ---- latent sampling ---- */
/* sample(mean,'fix') of model_sigmaVAE.py:153-178 / 187-213: out = mean + std*noise, rounded exactly as
 * torch does (mul, then add).  std_noise != NULL selects 'gaussian': per-item std_b = std_noise[b]*value. */
int kvae_sigma_sample(const void* mean, const void* noise, void* out, size_t n, int dtype, float std,
                      const void* std_noise, float value, size_t per_batch, void* stream);
/* One autoregressive step of the LM <-> VAE glue (model_sigmaVAE.py:123-145, Llasa.infer), ONE launch:
 *   mean = distribution_linear(hidden) = W2 gelu(W1 hidden + b1) + b2      (nn.Sequential(Linear, GELU, Linear), :42-50)
 *   latent = mean + std*noise (sample 'fix', two roundings)   kl_end = KL(N(mean,std) || N(1,e)).sum(-1)/D (:134-139)
 *   embed = audio_linear(latent) = Wa latent + ba                                                           (:143)
 * hidden [B,H] (hidden_dtype), noise / mean / latent [B,D] and embed [B,H] in out_dtype, weights fp32 in torch's
 * nn.Linear layout (W1 [D,H], W2 [D,D], Wa [H,D]), kl_end [B] fp32 or NULL.  H and D multiples of 8. */
int kvae_lm_glue_step(const void* hidden, int hidden_dtype, const float* w1, const float* b1, const float* w2,
                      const float* b2, const float* wa, const float* ba, const void* noise, void* mean, void* latent,
                      void* embed, float* kl_end, int out_dtype, int B, int H, int D, float std, void* stream);
/* vae_sample of bottleneck.py:51-62 (as edited in the reference): out = noise*scale + mean; *kl (device
 * fp32 scalar) = (mean^2 + var - log var - 1).sum(1).mean().  scratch: >= 8*1024 bytes. */
int kvae_vae_sample(const void* mean, const void* scale, const void* noise, void* out, float* kl, int B, int D,
                    long long T, int dtype, void* scratch, void* stream);

/* ---- Oobleck discriminator of the autoencoder's GAN training (SURVEY section 8f item 4, discriminator half) ----
 * stable_audio_tools/models/discriminators.py: SharedDiscriminatorConvNet (62-116), MultiScaleDiscriminator (119-138),
 * MultiPeriodDiscriminator (140-168), MultiDiscriminator (171-238), OobleckDiscriminator.loss (240-297),
 * get_hinge_losses (11-14); wired at training/autoencoders.py:133-134, 288.  Every net is a stack of strided
 * convolutions + SiLU; they run on kvae_disc_conv15_* / kvae_disc_conv1x1_* below (kvae_conv1d_fwd / kvae_conv1d_win_bwd on
 * engine 0 for any other kernel size / stride; the weight gradient may be NULL when only the data gradient is wanted).  The multi-period nets' 15 x 15 Conv2d over [N, C, ceil(T / n), n] becomes a Conv1d over the folded
 * channels (c, w): same products, minus those with padding zeros.  All tensors fp32, contiguous; `backward` = 1 runs the
 * adjoint with the roles of the two tensor arguments exchanged (first = incoming gradient, second = outgoing). */
/* MultiPeriodDiscriminator.fold (:164-168): y[b, c n + w, h] = x[b, c, h n + w] (0 past T); x [N, C, T], y [N, C n, ceil(T / n)] */
int kvae_disc_period_fold(const float* x, float* y, int N, int C, long long T, int n, int backward, void* stream);
/* nn.functional.avg_pool1d(x, 2) between the scales (:137): x [rows, T] -> y [rows, T / 2] */
int kvae_disc_avg_pool2(const float* x, float* y, long long rows, long long T, int backward, void* stream);
/* width of the folded axis after a conv: (W + 2 pad - K) / stride + 1 (0 if the arguments are invalid) */
int kvae_disc_folded_width(int W, int K, int stride, int pad);
/* Conv2d weight w [Cout, Cin, K, K] (weight-norm already folded) + bias [Cout] -> Conv1d weight over the folded channels
 * wf [Cout Wo, Cin W, K], wf[(co, wo), (ci, wi), kh] = w[co, ci, kh, wi - stride wo + pad], bias_f[(co, wo)] = bias[co].
 * backward = 1: wf / bias_f hold gradients, w / bias receive them (overwritten).  bias / bias_f may be NULL together. */
int kvae_disc_fold_weight2d(const float* w, const float* bias, float* wf, float* bias_f, int Cout, int Cin, int K, int stride,
                            int pad, int W, int backward, void* stream);
/* nn.SiLU (:76): a = f sigmoid(f);  backward: gf = ga * silu'(f) + gfeat (gfeat, the gradient arriving at the feature
 * tensor itself, may be NULL; gf may alias ga) */
int kvae_disc_silu_fwd(const float* f, float* a, size_t n, void* stream);
int kvae_disc_silu_bwd(const float* f, const float* ga, const float* gfeat, float* gf, size_t n, void* stream);
/* score[b] (+)= mean(y[b, :]) (:115);  backward: gy[b, i] = gscore[b] / inner + gfeat[b, i] (either may be NULL) */
int kvae_disc_score(const float* y, float* score, int N, long long inner, int accumulate, void* stream);
int kvae_disc_score_bwd(const float* gscore, const float* gfeat, float* gy, int N, long long inner, void* stream);
/* get_hinge_losses (:11-14) on score [2B] = (reals | fakes): losses[0] = relu(1 - s_real).mean() + relu(1 + s_fake).mean(),
 * losses[1] = -s_fake.mean().  With g_losses [2] (device) it writes d / d score into g_score [2B] instead. */
int kvae_disc_hinge(const float* score, int B, float* losses, const float* g_losses, float* g_score, void* stream);
/* feature-matching distance (:285-295) over n_feats tensors in one launch: loss[0] = sum_k mean |real_k - fake_k|, the
 * real half of tensor k being its first half[k] floats and the fake half the next half[k] (feats / half / grads: HOST
 * arrays).  With g_loss (one device float) it writes the gradients into grads[k] (2 half[k] floats each) instead. */
size_t kvae_disc_feature_match_scratch_bytes(const long long* half, int n_feats);
int kvae_disc_feature_match(const float* const* feats, const long long* half, int n_feats, float* loss,
                            const float* g_loss, float* const* grads, void* scratch, size_t scratch_bytes, void* stream);

/* The nets' own conv geometry -- Conv1d(k = 15, stride 4, padding 7) on [N, Cin, T] fp32 with a folded weight in torch
 * layout (discriminators.py:70-71, 85-100) -- on register-tiled kernels written for it; the forward has kvae_conv1d_fwd's
 * contract, the backward writes dw (the gradient of the folded weight, torch layout), dbias and gx, each optional
 * (scratch for both: kvae_conv1d_scratch_bytes(Cin, Cout, 15)). */
int kvae_disc_conv15_supported(int K, int stride, int pad);
int kvae_disc_conv15_fwd(const float* x, float* y, const float* w, const float* bias, int N, int Cin, int Cout, long long T,
                         void* scratch, size_t scratch_bytes, void* stream);
int kvae_disc_conv15_bwd(const float* x, const float* gy, const float* w, float* gx, float* dw, float* dbias, int N, int Cin,
                         int Cout, long long T, void* scratch, size_t scratch_bytes, void* stream);
/* The nets' last layer: Conv1d(k = 1) onto 1..8 channels (discriminators.py:104), x [N, Cin, T] fp32, w [Cout, Cin] */
int kvae_disc_conv1x1_supported(int K, int stride, int pad, int Cout);
int kvae_disc_conv1x1_fwd(const float* x, float* y, const float* w, const float* bias, int N, int Cin, int Cout, long long T,
                          void* stream);
int kvae_disc_conv1x1_bwd(const float* x, const float* gy, const float* w, float* gx, float* dw, float* dbias, int N, int Cin,
                          int Cout, long long T, void* stream);
#ifdef __cplusplus
}
#endif
#endif /* KVAE_H_ */
