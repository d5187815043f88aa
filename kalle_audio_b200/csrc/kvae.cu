// libkvae.so: plan construction, workspace layout, launch sequencing and the C ABI (include/kvae.h).
//
// A plan turns the constructor arguments of OobleckEncoder / OobleckDecoder
// (stable_audio_tools/models/autoencoders.py:116-191 of the reference) into a linear list of
// convolution steps.  SnakeBeta never runs as its own kernel inside a plan: it is folded into the
// epilogue of the producing convolution (which then emits the bf16 tensor-core operand of the next
// convolution) or into the prologue of a CUDA-core convolution.  Residual adds are folded into the
// epilogue of the k=1 convolution of each ResidualUnit (:47-62); the residual stream stays fp32.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/kvae.h"
#include "conv_direct.cuh"
#include "conv_edge.cuh"
#include "conv_umma_host.cuh"
#include "elementwise.cuh"
#include "glue.cuh"
#include "bigvgan.cuh"
#include "flow.cuh"
#include "mrstft.cuh"
#include "disc.cuh"
#include "train.cuh"

using namespace kvae;

namespace {

thread_local std::string g_err;
thread_local long long g_launches = 0;

int fail(const std::string& m) {
  g_err = m;
  return -1;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return -2;
}
#define KV_CUDA(x)                                  \
  do {                                              \
    cudaError_t e_ = (x);                           \
    if (e_ != cudaSuccess) return cuda_fail(e_, #x); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// device that owns a tensor the caller passed in: the stand-alone entry points launch there, whatever the calling
// thread's current device is (torch code routinely holds tensors on cuda:1 while the current device is 0)
int device_of(const void* p) {
  cudaPointerAttributes a;
  if (p && cudaPointerGetAttributes(&a, p) == cudaSuccess && (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged))
    return a.device;
  cudaGetLastError();
  int d = 0;
  cudaGetDevice(&d);
  return d;
}

struct ConvLayer {
  ConvGeom g;
  bool has_bias = true;
  bool umma = false;                  // bf16 mode: tensor-core layer (forward, dgrad, wgrad)
  bool umma32 = false;                // fp32 mode, inference only: tensor-core layer through the bf16x3 split
  __nv_bfloat16* w_umma = nullptr;    // [K][Cout][Cin] bf16: forward tensor-core operand ([K][Cout][2*Cin] hi|lo with umma32)
  float* w_direct = nullptr;          // [K][Cin][Cout] fp32: forward CUDA-core operand
  __nv_bfloat16* w_head = nullptr;    // encoder head on the tensor cores: [Cout][64] bf16, written by wave_in_im2col_kernel
  // training only (allocated by kvae_plan_load_params(train = 1)): the data-gradient kernels see the same
  // weight tensor under the opposite kind (Cin <-> Cout), i.e. the other index order of each precision
  __nv_bfloat16* w_umma_d = nullptr;  // [K][Cin][Cout] bf16
  float* w_direct_d = nullptr;        // [K][Cout][Cin] fp32
  float* bias = nullptr;
  bool set = false;
  // offsets (in floats) into the flat parameter / gradient buffer: [bias][weight_g][weight_v]
  long long off_bias = -1, off_g = -1, off_v = -1;
  long long off_dwp = -1;             // tensor-core convs: offset of the packed [K][Cd][Cs] weight-gradient accumulator
  int dim0() const { return g.kind == kConvT ? g.Cin : g.Cout; }
  size_t numel() const { return static_cast<size_t>(g.Cin) * g.Cout * g.K; }
};

struct SnakeLayer {
  int C = 0;
  float* a = nullptr;
  float* inv_b = nullptr;
  int logscale = 1;
  bool set = false;
  long long off_alpha = -1, off_beta = -1;   // flat parameter / gradient offsets
};

// one convolution of the chain, with its fused prologue / epilogue
struct Step {
  int conv = -1;
  int pre_snake = -1;      // SnakeBeta applied to this conv's input (module order index) or -1
  int residual_from = -1;  // step whose output is added in the epilogue (ResidualUnit skip) or -1
  int len_num = 1, len_den = 1;  // output length = T * len_num / len_den
  // resolved by finalize():
  bool needs_raw = false, needs_act = false;
  int epi_snake = -1;      // SnakeBeta folded into the epilogue for the next (tensor-core) conv
  int fuse = 0;            // 1: k7 conv of a ResidualUnit run by the fused kernel together with the next step (2)
  bool act_f16 = false;    // the activated output is fp16 (the unit in front of the tensor-core decoder tail)
};

struct Tensor {
  size_t bytes = 0;
  int first = 0, last = 0;
  size_t offset = 0;
};

struct Layout {
  // tensors: index 0 = channels-last bf16 copy of the external input (if step 0 is tensor-core),
  //          1 + 2*k = raw (fp32) output of step k, 2 + 2*k = activated bf16 output of step k
  std::vector<Tensor> t;
  size_t total = 0;
};

// The kernel that serves one step of a plan (step_kind); the whole-clip run and the stream both launch these.
enum StepKind {
  kTcConv,      // tensor-core conv (conv_umma2.cuh)
  kDirect,      // CUDA-core conv (conv_direct.cuh)
  kWaveIn,      // encoder head on the CUDA cores (conv_edge.cuh)
  kWaveOut,     // decoder tail on the CUDA cores
  kRuFused,     // fused ResidualUnit (conv_ru2.cuh): this step and the next
  kRuSecond,    // the k = 1 half of a fused unit: computed by the previous step's launch
  kWaveOutTc,   // decoder tail on the tensor cores (TF32, or fp16 with the fp16 stream)
  kWaveInTc,    // encoder head as im2col + a k = 1 tensor-core conv
};

struct DirectLaunch {             // conv_direct_kernel: parameters, tile configuration (direct_cfg_for), grid, smem
  DirectParams d;
  dim3 grid;
  int cfg = 0;
  size_t smem = 0;
};

// what one step needs at launch time; only the members of its kind are filled
struct StepLaunch {
  StepKind kind = kTcConv;
  int k = 0;                      // index of the step
  ConvLaunch2 umma2;              // kTcConv, and the k = 1 conv of kWaveInTc
  RuLaunch ru;                    // kRuFused
  WaveInParams wave_in;           // kWaveIn
  WaveInColParams head_col;       // kWaveInTc: im2col + weight pack in front of the k = 1 conv
  WaveOutParams wave_out;         // kWaveOut
  CUtensorMap wo_tmX;             // kWaveOutTc
  WaveOutTcParams wave_out_tc;
  DirectLaunch direct;            // kDirect
};

struct PreparedRun {
  std::vector<StepLaunch> steps;    // one per step of the plan
  bool stream_f16 = false;
  Layout layout;
  // ---- training runs only: the backward pass over the saved activations
  struct Bwd {
    int dgrad_kind = 0;             // 0 none, 1 tensor-core (conv_umma2 under the dgrad geometry), 2 CUDA-core
    ConvLaunch2 dg_umma;
    DirectLaunch dg_direct;
    int wg_kind = 0;                // 0 CUDA-core (torch-layout atomics), 1 tensor-core (packed accumulator),
                                    // 2 waveform-edge streaming kernel
    EdgeWgradParams wg_edge;
    EdgeDgradParams dg_edge;        // dgrad_kind 3: decoder tail (C -> io) data gradient
    int dg_edge_grid = 0;
    size_t dg_edge_smem = 0;
    int wg_edge_grid = 0;
    size_t wg_edge_smem = 0;
    bool wg_edge_x_is_thin = false;
    WgradLaunch wg_umma;
    WgradParams wg;
    dim3 wg_grid;
    bool wg_x_is_D = false, wg_x_is_S = false;   // step 0: the operand is the caller's input tensor
    bool has_sb = false;
    SnakeBwdParams sb;
    dim3 sb_grid;
    bool sb_fused = false;          // the SnakeBeta backward of this step runs in the epilogue of dg_umma (ConvParams2::bwd)
  };
  std::vector<Bwd> bwd;
  SnakeBwdParams sb_last;           // bf16 copy + bias gradient of the incoming output gradient
  dim3 sb_last_grid;
  size_t off_G[3] = {0, 0, 0}, off_Gb[3] = {0, 0, 0}, off_dA = 0;   // byte offsets in the workspace
  size_t total = 0;                 // forward + backward bytes
};

}  // namespace

struct kvae_plan {
  kvae_arch arch;
  int direction = KVAE_DECODER;
  int precision = KVAE_PREC_BF16;
  int device = 0;
  std::vector<ConvLayer> convs;
  std::vector<SnakeLayer> snakes;
  std::vector<Step> steps;    // inference: fused ResidualUnits, only the tensors the next layer needs
  std::vector<Step> tsteps;   // training: every layer's pre-activation stream is kept for the backward pass
  int ratio = 1;
  long long n_params = 0;     // floats in the flat parameter / gradient buffer
  std::vector<long long> param_sizes;   // segment sizes in module.parameters() order
  bool train_packs = false;
  bool stream_f16 = false;    // inference plans keep the residual stream in fp16 (bf16 mode, all-tensor-core chains)
  bool tail_preact = false;   // the last ResidualUnit writes SnakeBeta(x) in fp16 and the decoder tail reads that (no transform stage)
  bool train_stream_f16 = false;   // ... and so do training plans whose every backward consumer of the stream knows fp16
  float* scale_scratch = nullptr;   // g/||v|| per dim-0 row of the conv being packed
  // batched kvae_plan_load_params (one scale + one pack + one SnakeBeta-constant launch for the whole plan)
  FoldDesc* fold_desc = nullptr;    // device, one per conv
  SnakeDesc* snake_desc = nullptr;  // device, one per SnakeBeta
  float* scale_all = nullptr;       // device, sum of dim-0 rows
  int fold_rows = 0, fold_tiles = 0;
  int fold_train = -1;              // the `train` flag the descriptors were built for (-1: not built)
  WnBwdDesc* wn_desc = nullptr;     // device, one per conv: batched weight-norm backward
  int wn_rows = 0;
  float* dwp = nullptr;             // packed weight-gradient accumulators of the tensor-core convs
  size_t dwp_floats = 0;
  std::map<std::tuple<int, long long, void*>, std::unique_ptr<PreparedRun>> runs;
  std::map<std::tuple<int, long long, void*>, std::unique_ptr<PreparedRun>> truns;
  // optional per-step CUDA-event timing (bench.py's roofline leg)
  bool profile = false;
  std::vector<cudaEvent_t> events;
  int prof_B = 0;
  long long prof_T = 0;
  bool prof_valid = false;
};

namespace {

int ceil_div(int a, int b) { return (a + b - 1) / b; }

bool env_flag(const char* name) {
  const char* e = getenv(name);
  return e && e[0] == '1';
}

void add_conv(kvae_plan* p, int kind, int Cin, int Cout, int K, int stride, int dil, int pad, bool bias) {
  ConvLayer c;
  c.g = ConvGeom{kind, Cin, Cout, K, stride, dil, pad};
  c.has_bias = bias;
  c.umma = (p->precision == KVAE_PREC_BF16) && umma_supported(c.g);
  c.umma32 = (p->precision == KVAE_PREC_F32) && umma_supported(c.g);
  p->convs.push_back(c);
}
int add_snake(kvae_plan* p, int C) {
  SnakeLayer s;
  s.C = C;
  p->snakes.push_back(s);
  return static_cast<int>(p->snakes.size()) - 1;
}

// ResidualUnit (autoencoders.py:39-62): snake -> conv k7 dil d -> snake -> conv k1 -> + x
void add_residual_unit(kvae_plan* p, int C, int d, int num, int den) {
  const int input_step = static_cast<int>(p->steps.size()) - 1;
  const int s0 = add_snake(p, C);
  add_conv(p, kConv, C, C, 7, 1, d, 3 * d, true);
  Step a;
  a.conv = static_cast<int>(p->convs.size()) - 1;
  a.pre_snake = s0;
  a.len_num = num; a.len_den = den;
  p->steps.push_back(a);
  const int s1 = add_snake(p, C);
  add_conv(p, kConv, C, C, 1, 1, 1, 0, true);
  Step b;
  b.conv = static_cast<int>(p->convs.size()) - 1;
  b.pre_snake = s1;
  b.residual_from = input_step;
  b.len_num = num; b.len_den = den;
  p->steps.push_back(b);
}

void build_decoder(kvae_plan* p) {
  const kvae_arch& a = p->arch;
  const int n = a.n_stages;
  std::vector<int> cm(n + 1, 1);
  for (int i = 0; i < n; ++i) cm[i + 1] = a.c_mults[i];
  // layers.0: WNConv1d(latent -> c_mults[-1]*channels, k7, pad 3)                         (:168)
  add_conv(p, kConv, a.latent_dim, cm[n] * a.channels, 7, 1, 1, 3, true);
  Step s;
  s.conv = 0;
  p->steps.push_back(s);
  int num = 1;
  for (int i = n; i >= 1; --i) {            // DecoderBlock (:83-114), strides walked in reverse (:171-180)
    const int cin = cm[i] * a.channels, cout = cm[i - 1] * a.channels, st = a.strides[i - 1];
    const int sn = add_snake(p, cin);
    if (a.use_nearest_upsample) {
      // Upsample(nearest, x st) + Conv1d(k = 2 st, 'same', no bias) (:87-96) == ConvTranspose1d(k = 3 st - 1, stride st,
      // padding st, output_padding 1) with summed taps (include/kvae.h); the host folds the weight
      add_conv(p, kConvT, cin, cout, 3 * st - 1, st, 1, st, false);
      p->convs.back().g.out_pad = 1;
    } else {
      add_conv(p, kConvT, cin, cout, 2 * st + st % 2, st, 1, ceil_div(st, 2), true);
    }
    num *= st;
    Step u;
    u.conv = static_cast<int>(p->convs.size()) - 1;
    u.pre_snake = sn;
    u.len_num = num;
    p->steps.push_back(u);
    for (int d : {1, 3, 9}) add_residual_unit(p, cout, d, num, 1);
  }
  const int sn = add_snake(p, cm[0] * a.channels);
  add_conv(p, kConv, cm[0] * a.channels, a.io_channels, 7, 1, 1, 3, false);   // bias=False (:184)
  Step f;
  f.conv = static_cast<int>(p->convs.size()) - 1;
  f.pre_snake = sn;
  f.len_num = num;
  p->steps.push_back(f);
  p->ratio = num;
}

void build_encoder(kvae_plan* p) {
  const kvae_arch& a = p->arch;
  const int n = a.n_stages;
  std::vector<int> cm(n + 1, 1);
  for (int i = 0; i < n; ++i) cm[i + 1] = a.c_mults[i];
  add_conv(p, kConv, a.io_channels, cm[0] * a.channels, 7, 1, 1, 3, true);      // (:133)
  Step s;
  s.conv = 0;
  p->steps.push_back(s);
  int den = 1;
  for (int i = 0; i < n; ++i) {             // EncoderBlock (:64-81)
    const int cin = cm[i] * a.channels, cout = cm[i + 1] * a.channels, st = a.strides[i];
    for (int d : {1, 3, 9}) add_residual_unit(p, cin, d, 1, den);
    const int sn = add_snake(p, cin);
    add_conv(p, kConv, cin, cout, 2 * st, st, 1, ceil_div(st, 2), true);
    den *= st;
    Step u;
    u.conv = static_cast<int>(p->convs.size()) - 1;
    u.pre_snake = sn;
    u.len_den = den;
    p->steps.push_back(u);
  }
  const int sn = add_snake(p, cm[n] * a.channels);
  add_conv(p, kConv, cm[n] * a.channels, a.latent_dim, 3, 1, 1, 1, true);        // (:141)
  Step f;
  f.conv = static_cast<int>(p->convs.size()) - 1;
  f.pre_snake = sn;
  f.len_den = den;
  p->steps.push_back(f);
  p->ratio = den;
}

bool conv_tc(const ConvLayer& c, bool train) { return c.umma || (!train && c.umma32); }

bool k7same_geom(const ConvGeom& g) {
  return g.kind == kConv && g.K == 7 && g.stride == 1 && g.dilation == 1 && g.pad == 3;
}
// the two waveform-edge convs that have kernels of their own in bf16 mode (conv_edge.cuh)
bool is_wave_out_step(const kvae_plan* p, const std::vector<Step>& steps, int k) {
  const int n = static_cast<int>(steps.size());
  const Step& s = steps[k];
  const ConvLayer& c = p->convs[s.conv];
  return !c.umma && !c.umma32 && k7same_geom(c.g) && k == n - 1 && k > 0 && c.g.Cout <= 2 &&
         !c.has_bias && c.g.Cin == 128 && s.pre_snake >= 0 && s.residual_from < 0;
}
bool is_wave_in_step(const kvae_plan* p, const std::vector<Step>& steps, int k) {
  const int n = static_cast<int>(steps.size());
  const Step& s = steps[k];
  const ConvLayer& c = p->convs[s.conv];
  return !c.umma && !c.umma32 && k7same_geom(c.g) && k == 0 && n > 1 && c.g.Cin <= 2 && c.has_bias &&
         c.g.Cout % 128 == 0 && s.pre_snake < 0 && s.residual_from < 0;
}
// the encoder head runs as im2col + a k = 1 tensor-core conv (conv_edge.cuh, wave_in_im2col_kernel) in inference plans
// with the fp16 stream; KVAE_WAVE_IN_CC=1 keeps the CUDA-core kernel
bool head_on_tc(const kvae_plan* p, const std::vector<Step>& steps, bool train) {
  return !train && p->precision == KVAE_PREC_BF16 && p->stream_f16 && is_wave_in_step(p, steps, 0) &&
         p->convs[steps[0].conv].g.Cin <= 2 && !env_flag("KVAE_WAVE_IN_CC");
}
StepKind step_kind(const kvae_plan* p, const std::vector<Step>& steps, int k, bool train) {
  const Step& s = steps[k];
  if (s.fuse == 2) return kRuSecond;
  if (s.fuse == 1) return kRuFused;
  // fp32 mode keeps the tail's exact fp32 FMAs
  if (is_wave_out_step(p, steps, k)) return p->precision == KVAE_PREC_BF16 ? kWaveOutTc : kWaveOut;
  if (is_wave_in_step(p, steps, k)) return head_on_tc(p, steps, train) ? kWaveInTc : kWaveIn;
  return conv_tc(p->convs[s.conv], train) ? kTcConv : kDirect;
}
void finalize_steps(kvae_plan* p) {
  const int n = static_cast<int>(p->steps.size());
  // fp16 residual stream: only when every step runs on a kernel that knows about it (tensor-core convs and the
  // two waveform-edge kernels), i.e. the graded architectures in bf16 mode; anything else keeps fp32
  p->stream_f16 = p->precision == KVAE_PREC_BF16;
  for (int k = 0; k < n && p->stream_f16; ++k)
    if (!p->convs[p->steps[k].conv].umma && !is_wave_in_step(p, p->steps, k) && !is_wave_out_step(p, p->steps, k))
      p->stream_f16 = false;
  // Training plans: the saved pre-activation stream is fp16 too when every step is a tensor-core conv or one of the
  // two waveform-edge convs (the graded architectures): the forward k=1 convs then move 1024 instead of 1536 bytes per
  // row and use the fragment-mapped epilogue, the SnakeBeta backward reads 2 instead of 4 bytes per element.  The
  // 11 significant bits of fp16 are what the inference path already carries.
  p->train_stream_f16 = p->stream_f16 && n >= 3;
  // a conv is a tensor-core step in bf16 mode (always) or in fp32 mode for inference (bf16x3 split); fp32-mode
  // training stays on the CUDA cores, so the two step lists can differ in who needs which tensor
  auto set_flags = [&](std::vector<Step>& steps, bool train) {
    for (int k = 0; k < n; ++k) {
      Step& s = steps[k];
      const bool last = (k == n - 1);
      const bool next_tc = !last && conv_tc(p->convs[steps[k + 1].conv], train);
      s.needs_act = next_tc;
      s.epi_snake = next_tc ? steps[k + 1].pre_snake : -1;
      s.needs_raw = train || last || (!last && !next_tc);
      for (int j = k + 1; j < n; ++j)
        if (steps[j].residual_from == k) s.needs_raw = true;
    }
  };
  p->tsteps = p->steps;       // training plan: same chain, every pre-activation stream kept, no ResidualUnit fusion
  set_flags(p->steps, false);
  set_flags(p->tsteps, true);
  // flat parameter layout = module.parameters() order: per step [alpha, beta of its SnakeBeta] then the
  // conv's [bias][weight_g][weight_v] (old-style weight_norm keeps bias first)
  long long off = 0;
  p->param_sizes.clear();
  for (const Step& s : p->steps) {
    if (s.pre_snake >= 0) {
      SnakeLayer& sn = p->snakes[s.pre_snake];
      sn.off_alpha = off; off += sn.C; p->param_sizes.push_back(sn.C);
      sn.off_beta = off; off += sn.C; p->param_sizes.push_back(sn.C);
    }
    ConvLayer& c = p->convs[s.conv];
    if (c.has_bias) { c.off_bias = off; off += c.g.Cout; p->param_sizes.push_back(c.g.Cout); }
    c.off_g = off; off += c.dim0(); p->param_sizes.push_back(c.dim0());
    c.off_v = off; off += static_cast<long long>(c.numel()); p->param_sizes.push_back(static_cast<long long>(c.numel()));
  }
  p->n_params = off;
  // ResidualUnits of 128-channel stages run as ONE kernel (conv_ru2.cuh): k7 -> SnakeBeta -> k1 -> + skip.
  // KVAE_NO_RU_FUSION=1 keeps the two-kernel form (the reference of the fused kernel's tests).
  if (env_flag("KVAE_NO_RU_FUSION") || !p->stream_f16) return;   // the fused kernel reads / writes the fp16 stream
  for (int k = 1; k + 1 < n; ++k) {
    Step& a = p->steps[k];
    Step& b = p->steps[k + 1];
    const ConvLayer& c7 = p->convs[a.conv];
    const ConvLayer& c1 = p->convs[b.conv];
    const bool shape = c7.umma && c1.umma && c7.g.kind == kConv && c1.g.kind == kConv && ru_supported(c7.g.Cin) &&
                       c7.g.Cout == c7.g.Cin && c1.g.Cin == c7.g.Cin && c1.g.Cout == c7.g.Cin && c7.g.K == 7 &&
                       c7.g.stride == 1 && c7.g.pad == 3 * c7.g.dilation && c1.g.K == 1 && c1.g.stride == 1 &&
                       c1.g.pad == 0 && c7.has_bias && c1.has_bias;
    const bool flow = b.residual_from == k - 1 && a.residual_from < 0 && !a.needs_raw && a.needs_act &&
                      a.epi_snake >= 0 && p->steps[k - 1].needs_raw && p->steps[k - 1].needs_act && k + 1 < n - 1 + 1 &&
                      (b.needs_raw || b.needs_act);
    if (shape && flow && k + 1 != n - 1) {
      a.fuse = 1;
      b.fuse = 2;
      ++k;
    }
  }
  // Decoder tail (conv_edge.cuh): when the unit in front of it is a fused ResidualUnit, that unit applies the tail's
  // SnakeBeta in its epilogue and writes the result in fp16; the tail's 16 transform warps (0.33 of its 0.49 ms at
  // 16 x 442 368 rows) have nothing left to do.  One rounding fewer than snake(fp16(x)).  KVAE_TAIL_RAW=1: old flow.
  if (n >= 3 && !env_flag("KVAE_TAIL_RAW") && is_wave_out_step(p, p->steps, n - 1) &&
      p->steps[n - 2].fuse == 2 && p->steps[n - 1].pre_snake >= 0) {
    Step& b = p->steps[n - 2];
    b.needs_act = true;
    b.needs_raw = false;
    b.epi_snake = p->steps[n - 1].pre_snake;
    b.act_f16 = true;
    p->tail_preact = true;
  }
}

long long step_len(const Step& s, long long T) { return T * s.len_num / s.len_den; }

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Interval allocation of the intermediate tensors inside one workspace.
bool make_layout(const kvae_plan* p, const std::vector<Step>& steps, bool train, int B, long long T, Layout& L,
                 std::string& err) {
  const int n = static_cast<int>(steps.size());
  L.t.assign(1 + 2 * n, Tensor());
  const ConvLayer& c0 = p->convs[steps[0].conv];
  const int split = (p->precision == KVAE_PREC_F32 && !train) ? 2 : 1;   // operand tensors hold (hi | lo) halves
  if (conv_tc(c0, train)) {
    L.t[0].bytes = static_cast<size_t>(B) * T * c0.g.Cin * 2 * split;
    L.t[0].first = 0;
    L.t[0].last = 0;
  }
  for (int k = 0; k < n; ++k) {
    const Step& s = steps[k];
    const ConvLayer& c = p->convs[s.conv];
    const long long len = step_len(s, T);
    if (len <= 0) { err = "input too short for this architecture"; return false; }
    int last_use = k;
    if (k + 1 < n) last_use = k + 1;
    for (int j = k + 1; j < n; ++j)
      if (steps[j].residual_from == k) last_use = std::max(last_use, j);
    if (train) last_use = 1 << 30;   // saved for the backward pass
    if (s.needs_raw && k != n - 1) {
      Tensor& t = L.t[1 + 2 * k];
      t.bytes = static_cast<size_t>(B) * len * c.g.Cout * ((train ? p->train_stream_f16 : p->stream_f16) ? 2 : 4);
      t.first = k;
      t.last = last_use;
    }
    if (s.needs_act && s.fuse != 1) {   // the fused ResidualUnit keeps its intermediate in shared memory
      Tensor& t = L.t[2 + 2 * k];
      t.bytes = static_cast<size_t>(B) * len * c.g.Cout * 2 * split;
      t.first = k;
      t.last = train ? (1 << 30) : k + 1;
    }
  }
  if (head_on_tc(p, steps, train)) {
    L.t[0].bytes = static_cast<size_t>(B) * T * 64 * 2;     // im2col operand of the head conv
    L.t[0].first = 0;
    L.t[0].last = 0;
  }
  if (train && L.t[0].bytes) L.t[0].last = 1 << 30;
  // first-fit over live intervals, in order of first use
  struct Live { size_t off, size; int last; };
  std::vector<Live> live;
  size_t total = 0;
  auto place = [&](Tensor& t) {
    if (!t.bytes) return;
    const size_t sz = align_up(t.bytes, 1024);
    std::sort(live.begin(), live.end(), [](const Live& a, const Live& b) { return a.off < b.off; });
    size_t off = 0;
    for (const Live& l : live) {
      if (off + sz <= l.off) break;
      off = std::max(off, l.off + l.size);
    }
    t.offset = off;
    live.push_back({off, sz, t.last});
    total = std::max(total, off + sz);
  };
  place(L.t[0]);
  for (int k = 0; k < n; ++k) {
    std::vector<Live> keep;
    for (const Live& l : live)
      if (l.last >= k) keep.push_back(l);
    live.swap(keep);
    if (steps[k].fuse == 2) continue;          // placed together with the fused head (below)
    place(L.t[1 + 2 * k]);
    place(L.t[2 + 2 * k]);
    if (steps[k].fuse == 1) {
      // the fused ResidualUnit kernel runs at step k and writes step k+1's tensors: they must not share
      // memory with anything still live at step k (its own inputs included)
      place(L.t[1 + 2 * (k + 1)]);
      place(L.t[2 + 2 * (k + 1)]);
    }
  }
  L.total = std::max<size_t>(total, 1024);
  return true;
}

// CUDA-core conv tile (time rows x out-channels per 128-thread block) by output width: the 64-wide tile left 50-75 % of
// the threads without a channel on the 32- and 16-channel stages of BigVGANFlowVAE.  The per-output summation order does
// not depend on the tile, so every configuration gives the same bits.
int direct_cfg_for(int Cout) { return Cout <= 4 ? 1 : Cout <= 16 ? 2 : Cout <= 32 ? 3 : 0; }
void direct_tile(int cfg, int& BT, int& BN) {
  BT = cfg == 1 ? 128 : cfg == 2 ? 128 : cfg == 3 ? 64 : 32;
  BN = cfg == 1 ? 4 : cfg == 2 ? 16 : cfg == 3 ? 32 : 64;
}
// conv_direct_kernel for output rows [t_lo, T_out) of the conv of a T_in-row input: taps, geometry, tile, grid and
// shared memory.  Operands, strides and epilogue are zero; the caller fills them.
bool prepare_direct(const ConvGeom& g, int B, long long T_in, long long T_out, long long t_lo, DirectLaunch& L,
                    std::string& err) {
  TapPlan tp;
  if (!build_taps(g, tp, err)) return false;
  DirectParams& d = L.d;
  std::memset(&d, 0, sizeof(d));
  d.B = B; d.P_out = tp.P_out; d.P_in = tp.P_in;
  d.Tq_out = static_cast<int>((T_out + tp.P_out - 1) / tp.P_out); d.T_out = static_cast<int>(T_out);
  d.q_base = static_cast<int>(t_lo / tp.P_out); d.t_lo = static_cast<int>(t_lo);
  d.T_in = static_cast<int>(T_in); d.Cin = g.Cin; d.Cout = g.Cout; d.span = tp.span;
  for (int i = 0; i <= kMaxPhases; ++i) d.tap_begin[i] = tp.tap_begin[i];
  for (size_t i = 0; i < tp.taps.size(); ++i) d.taps[i] = tp.taps[i];
  L.cfg = direct_cfg_for(g.Cout);
  int BT, BN;
  direct_tile(L.cfg, BT, BN);
  L.grid = dim3(ceil_div(d.Tq_out - d.q_base, BT) * tp.P_out, ceil_div(g.Cout, BN), B);
  L.smem = (static_cast<size_t>(BT + tp.span) * (kDirectKC + 1) + kDirectKC * BN) * sizeof(float);
  return true;
}
cudaError_t launch_direct(const DirectLaunch& L, cudaStream_t st) {
  if (L.cfg == 1) conv_direct_kernel<128, 4, 1, 4><<<L.grid, 128, L.smem, st>>>(L.d);
  else if (L.cfg == 2) conv_direct_kernel<128, 16, 4, 4><<<L.grid, 128, L.smem, st>>>(L.d);
  else if (L.cfg == 3) conv_direct_kernel<64, 32, 4, 4><<<L.grid, 128, L.smem, st>>>(L.d);
  else conv_direct_kernel<32, 64, 4, 4><<<L.grid, 128, L.smem, st>>>(L.d);
  return cudaGetLastError();
}

cudaError_t launch_wave_out(WaveOutParams& w, int Cout, int B, cudaStream_t st) {
  const size_t smem = wave_out_smem(w.Cin);
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(conv_wave_out_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_wave_out_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set[dev & 63] = true;
  }
  w.B = B;
  w.tiles_per_clip = (w.T + kWaveOutTile - 1) / kWaveOutTile;
  w.total_tiles = w.tiles_per_clip * B;
  const int grid = std::min(w.total_tiles, sm_count());
  if (Cout == 1) conv_wave_out_kernel<1><<<grid, 288, smem, st>>>(w);
  else conv_wave_out_kernel<2><<<grid, 288, smem, st>>>(w);
  return cudaGetLastError();
}

cudaError_t launch_wave_out_tc(const CUtensorMap& tmX, const WaveOutTcParams& t, bool stream_f16, cudaStream_t st) {
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(conv_wave_out_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_wave_out_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set[dev & 63] = true;
  }
  const int grid = std::min(t.total_tiles, sm_count());
  if (stream_f16) return launch_pdl(conv_wave_out_tc_kernel<true>, dim3(grid), dim3(kWoTcThreads), wave_out_tc_smem<true>(), st, tmX, t);
  return launch_pdl(conv_wave_out_tc_kernel<false>, dim3(grid), dim3(kWoTcThreads), wave_out_tc_smem<false>(), st, tmX, t);
}

cudaError_t launch_wave_in(const WaveInParams& w, int Cin, int B, cudaStream_t st) {
  dim3 grid((w.T + kWaveInTile - 1) / kWaveInTile, w.Cout / 128, B);
  if (Cin == 1) conv_wave_in_kernel<1><<<grid, 128, 0, st>>>(w);
  else conv_wave_in_kernel<2><<<grid, 128, 0, st>>>(w);
  return cudaGetLastError();
}

// Where one step reads and writes.  The whole-clip run points into its workspace (a padded clip: in_row0 = -3, the
// caller's input and output are patched in per call); the stream points into its window buffers (in_row0 = 0, and a
// StreamGeom for the tensor-core kernels, which also carries the output and skip pitches).
struct StepIO {
  const void* in_act = nullptr;       // bf16 operand of the input
  const void* in_raw = nullptr;       // stream tensor of the input (the head: the channels-first samples)
  long long in_rows = 0, in_pitch = 0;
  int in_row0 = 0;                    // edge kernels: input row of output 0's first tap
  long long out_rows = 0, out_pitch = 0;
  void* out_raw = nullptr;            // stream tensor of the output
  __nv_bfloat16* out_act = nullptr;   // operand tensor of the output
  const void* res = nullptr;          // skip connection, row-aligned with the output
  void* ext = nullptr;                // last step: the caller's (or the staging) output, channels-first
  int ext_f32 = 1;
  long long cf_ld = 0;                // its rows per channel (0: out_rows)
  __nv_bfloat16* col = nullptr;       // im2col operand of the head on the tensor cores
  const StreamGeom* sg = nullptr;
};

// Prepares the launch of step k (kRuFused: k and k + 1, whose tensors io describes) for the whole-clip run and the
// stream alike.
bool prepare_step(const kvae_plan* p, const std::vector<Step>& steps, int k, bool train, int B, const StepIO& io,
                  StepLaunch& L, std::string& err) {
  const Step& s = steps[k];
  const ConvLayer& c = p->convs[s.conv];
  const bool last = k == static_cast<int>(steps.size()) - 1;
  const int sf16 = (train ? p->train_stream_f16 : p->stream_f16) ? 1 : 0;
  const int precise = p->precision == KVAE_PREC_F32 ? 1 : 0;
  const int T_in = static_cast<int>(io.in_rows), T_out = static_cast<int>(io.out_rows);
  const float* snake_a = s.epi_snake >= 0 ? p->snakes[s.epi_snake].a : nullptr;
  const float* snake_inv_b = s.epi_snake >= 0 ? p->snakes[s.epi_snake].inv_b : nullptr;
  L.kind = step_kind(p, steps, k, train);
  L.k = k;
  switch (L.kind) {
    case kRuSecond:
      return true;
    case kRuFused: {
      const Step& s1 = steps[k + 1];
      const ConvLayer& c1 = p->convs[s1.conv];
      RuArgs ra;
      ra.a = static_cast<const __nv_bfloat16*>(io.in_act);
      ra.x = io.res;
      ra.stream_f16 = sf16;
      ra.w7 = c.w_umma; ra.w1 = c1.w_umma;
      ra.bias7 = c.bias; ra.bias1 = c1.bias;
      ra.s2_a = snake_a; ra.s2_inv_b = snake_inv_b;
      ra.out_raw = io.out_raw;
      ra.out_act = io.out_act;
      ra.act_f16 = s1.act_f16 ? 1 : 0;
      if (s1.epi_snake >= 0) { ra.sn_a = p->snakes[s1.epi_snake].a; ra.sn_inv_b = p->snakes[s1.epi_snake].inv_b; }
      return prepare_conv_ru(ra, B, T_out, c.g.dilation, L.ru, err, io.sg);
    }
    case kWaveOut:
    case kWaveOutTc: {
      // decoder tail (conv_edge.cuh): reads the stream tensor of the previous step, or its operand tensor when the
      // last unit wrote SnakeBeta(x) in fp16 (finalize_steps, tail_preact)
      const bool preact = p->tail_preact && !train;
      const void* x = preact ? io.in_act : io.in_raw;
      if (!x) { err = "internal: raw input missing"; return false; }
      const int tanh_out = (p->direction == KVAE_DECODER && p->arch.final_tanh) ? 1 : 0;
      const SnakeLayer& sn = p->snakes[s.pre_snake];
      if (L.kind == kWaveOut) {
        WaveOutParams& w = L.wave_out;
        std::memset(&w, 0, sizeof(w));
        w.x = static_cast<const float*>(x);
        w.pro_a = sn.a; w.pro_inv_b = sn.inv_b; w.w = c.w_direct;
        w.y = io.ext; w.y_f32 = io.ext_f32;
        w.T = T_out; w.Cin = c.g.Cin; w.tanh_out = tanh_out; w.precise = precise;
        w.T_in = T_in; w.in_row0 = io.in_row0; w.x_pitch = io.in_pitch;
        return true;
      }
      WaveOutTcParams& t = L.wave_out_tc;
      std::memset(&t, 0, sizeof(t));
      t.pro_a = sn.a; t.pro_inv_b = sn.inv_b; t.w = c.w_direct;
      t.y = io.ext; t.y_f32 = io.ext_f32;
      t.T = T_out; t.B = B; t.COUT = c.g.Cout; t.tanh_out = tanh_out; t.in_row0 = io.in_row0;
      t.preact = preact ? 1 : 0;
      t.tiles_per_clip = (t.T + kWoTcTile - 1) / kWoTcTile;
      t.total_tiles = t.tiles_per_clip * B;
      if (sf16) return make_act_tmap(&L.wo_tmX, x, B, T_in, 128, 1, kWoTcRows, err, io.in_pitch);
      return make_out_tmap(&L.wo_tmX, x, B, T_in, 128, 1, 1, err, kWoTcRows, io.in_pitch);
    }
    case kWaveIn: {
      // encoder head (conv_edge.cuh): reads the channels-first samples
      WaveInParams& w = L.wave_in;
      std::memset(&w, 0, sizeof(w));
      w.x = io.in_raw; w.x_f32 = 1;
      w.w = c.w_direct; w.bias = c.bias;
      w.out_raw = io.out_raw; w.raw_f16 = sf16;
      w.precise = precise;
      w.act_split = (io.out_act && precise && !train) ? 1 : 0;
      w.out_act = io.out_act;
      w.snake_a = snake_a; w.snake_inv_b = snake_inv_b;
      w.T = T_out; w.Cout = c.g.Cout;
      w.T_in = T_in; w.in_row0 = io.in_row0; w.x_pitch = io.in_pitch; w.out_pitch = io.out_pitch;
      return true;
    }
    case kWaveInTc: {
      WaveInColParams& h = L.head_col;
      std::memset(&h, 0, sizeof(h));
      h.x = io.in_raw; h.x_f32 = 1;
      h.col = io.col; h.w = c.w_direct; h.wp = c.w_head;
      h.T = T_out; h.B = B; h.Cout = c.g.Cout; h.CIN = c.g.Cin;
      h.T_in = T_in; h.in_row0 = io.in_row0; h.x_pitch = io.in_pitch;
      h.row_blocks = B * ((T_out + kColRows - 1) / kColRows);
      if (!h.col || !h.wp) { err = "internal: head operand missing"; return false; }
      ConvGeom g1 = c.g;
      g1.Cin = 64; g1.K = 1; g1.pad = 0; g1.dilation = 1; g1.stride = 1;
      ConvEpilogue ep;
      ep.bias = c.bias;
      ep.stream_f16 = 1;
      ep.out_raw = io.out_raw;
      ep.out_act = io.out_act;
      ep.snake_a = snake_a; ep.snake_inv_b = snake_inv_b;
      StreamGeom sg1;   // window form: the k = 1 conv reads all T_out rows of the im2col operand
      if (io.sg) { sg1.in_rows = sg1.out_q = T_out; sg1.in_pitch = T_out; sg1.raw_pitch = io.sg->raw_pitch; sg1.act_pitch = io.sg->act_pitch; }
      return prepare_conv_umma2(g1, h.col, B, T_out, c.w_head, ep, ConvTuning2(), L.umma2, err, io.sg ? &sg1 : nullptr);
    }
    case kTcConv: {
      if (!io.in_act) { err = "internal: tensor-core operand missing"; return false; }
      ConvEpilogue ep;
      ep.bias = c.has_bias ? c.bias : nullptr;
      ep.residual = io.res;
      ep.residual_f32 = sf16 ? 0 : 1;
      ep.stream_f16 = sf16;
      ep.out_raw = last ? io.ext : io.out_raw;
      ep.out_raw_f32 = last ? io.ext_f32 : (sf16 ? 0 : 1);
      ep.out_raw_cf = last ? 1 : 0;
      ep.out_act = io.out_act;
      ep.snake_a = snake_a; ep.snake_inv_b = snake_inv_b;
      if (!c.umma) {               // fp32 mode on the tensor cores: bf16x3 split operands, sinf in the epilogue
        ep.split3 = 1;
        ep.act_split = 1;
        ep.precise = 1;
      }
      if (!prepare_conv_umma2(c.g, static_cast<const __nv_bfloat16*>(io.in_act), B, T_in, c.w_umma, ep, ConvTuning2(),
                              L.umma2, err, io.sg))
        return false;
      if (last) L.umma2.p.cf_ld = io.cf_ld;
      return true;
    }
    case kDirect: {
      // the first step reads the caller's input [B, C, T], the last writes the caller's output; the rest of the chain
      // is channels-last fp32
      if (!prepare_direct(c.g, B, T_in, T_out, 0, L.direct, err)) return false;
      DirectParams& d = L.direct.d;
      d.x = io.in_raw; d.x_f32 = 1;
      if (k == 0) {
        d.x_sB = static_cast<long long>(c.g.Cin) * io.in_pitch; d.x_sT = 1; d.x_sC = io.in_pitch;
      } else {
        if (!d.x) { err = "internal: raw input missing"; return false; }
        d.x_sB = io.in_pitch * c.g.Cin; d.x_sT = c.g.Cin; d.x_sC = 1;
      }
      if (s.pre_snake >= 0) { d.pro_a = p->snakes[s.pre_snake].a; d.pro_inv_b = p->snakes[s.pre_snake].inv_b; }
      d.w = c.w_direct;
      d.bias = c.has_bias ? c.bias : nullptr;
      d.residual = io.res;
      d.residual_f32 = 1;
      if (last) {
        d.out_raw = io.ext; d.out_raw_f32 = io.ext_f32;
        d.o_sB = static_cast<long long>(c.g.Cout) * io.out_pitch; d.o_sT = 1; d.o_sC = io.out_pitch;
        d.tanh_out = (p->direction == KVAE_DECODER && p->arch.final_tanh) ? 1 : 0;
      } else {
        d.out_raw = io.out_raw; d.out_raw_f32 = 1;
        d.o_sB = io.out_pitch * c.g.Cout; d.o_sT = c.g.Cout; d.o_sC = 1;
      }
      d.out_act = io.out_act;
      d.act_split = (io.out_act && precise && !train) ? 1 : 0;
      d.snake_a = snake_a; d.snake_inv_b = snake_inv_b;
      return true;
    }
  }
  err = "internal: unknown step kind";
  return false;
}

// One step's kernels on stream st; g is the step's conv.  Counts every launch in g_launches.
cudaError_t launch_step(StepLaunch& L, const ConvGeom& g, int B, bool stream_f16, cudaStream_t st) {
  cudaError_t e = cudaSuccess;
  switch (L.kind) {
    case kRuSecond: return cudaSuccess;
    case kRuFused: e = launch_conv_ru(L.ru, st); break;
    case kTcConv: e = launch_conv_umma2(L.umma2, st); break;
    case kWaveOutTc: e = launch_wave_out_tc(L.wo_tmX, L.wave_out_tc, stream_f16, st); break;
    case kWaveOut: e = launch_wave_out(L.wave_out, g.Cout, B, st); break;
    case kWaveIn: e = launch_wave_in(L.wave_in, g.Cin, B, st); break;
    case kDirect: e = launch_direct(L.direct, st); break;
    case kWaveInTc: {
      const WaveInColParams& h = L.head_col;
      wave_in_im2col_kernel<<<h.row_blocks + (h.Cout * 64 + 255) / 256, 256, 0, st>>>(h);
      e = cudaGetLastError();
      if (e != cudaSuccess) return e;
      ++g_launches;
      e = launch_conv_umma2(L.umma2, st);
      break;
    }
  }
  if (e == cudaSuccess) ++g_launches;
  return e;
}

bool prepare_run(kvae_plan* p, const std::vector<Step>& steps, bool train, int B, long long T, void* ws,
                 PreparedRun& R, std::string& err) {
  const int n = static_cast<int>(steps.size());
  if (!make_layout(p, steps, train, B, T, R.layout, err)) return false;
  R.steps.assign(n, StepLaunch());
  R.stream_f16 = train ? p->train_stream_f16 : p->stream_f16;
  uint8_t* base = static_cast<uint8_t*>(ws);
  auto tptr = [&](int id) -> void* { return R.layout.t[id].bytes ? base + R.layout.t[id].offset : nullptr; };
  for (int k = 0; k < n; ++k) {
    const Step& s = steps[k];
    const ConvLayer& c = p->convs[s.conv];
    const long long T_in = (k == 0) ? T : step_len(steps[k - 1], T);
    const long long T_out = step_len(s, T);
    if (c.g.out_len(static_cast<int>(T_in)) != T_out) {
      err = "length bookkeeping mismatch at step " + std::to_string(k) + " (input length must be a multiple of the stride product)";
      return false;
    }
    const int ko = (s.fuse == 1) ? k + 1 : k;    // the step whose tensors receive the result
    const Step& so = steps[ko];
    // tensor 0: the channels-last copy of the input for a tensor-core first layer, or the head's im2col operand
    StepIO io;
    io.in_act = tptr(k == 0 ? 0 : 2 + 2 * (k - 1));
    io.in_raw = (k == 0) ? nullptr : tptr(1 + 2 * (k - 1));   // k == 0: the caller's input, patched per call
    io.in_rows = io.in_pitch = T_in;
    io.in_row0 = -3;
    io.out_rows = io.out_pitch = T_out;
    io.out_raw = (so.needs_raw && ko != n - 1) ? tptr(1 + 2 * ko) : nullptr;
    io.out_act = so.needs_act ? static_cast<__nv_bfloat16*>(tptr(2 + 2 * ko)) : nullptr;
    io.res = (so.residual_from >= 0) ? tptr(1 + 2 * so.residual_from) : nullptr;
    if (so.residual_from >= 0 && !io.res) { err = "internal: residual tensor missing"; return false; }
    io.ext = reinterpret_cast<void*>(0x1);      // placeholder: the caller's output, patched per call
    io.col = static_cast<__nv_bfloat16*>(tptr(0));
    if (!prepare_step(p, steps, k, train, B, io, R.steps[k], err)) return false;
  }
  return true;
}

bool prepare_backward(kvae_plan* p, int B, long long T, void* ws, PreparedRun& R, std::string& err);

PreparedRun* get_run(kvae_plan* p, bool train, int B, long long T, void* ws, std::string& err) {
  auto& cache = train ? p->truns : p->runs;
  auto key = std::make_tuple(B, T, ws);
  auto it = cache.find(key);
  if (it == cache.end()) {
    auto R = std::make_unique<PreparedRun>();
    if (!prepare_run(p, train ? p->tsteps : p->steps, train, B, T, ws, *R, err)) return nullptr;
    R->total = R->layout.total;
    if (train && !prepare_backward(p, B, T, ws, *R, err)) return nullptr;
    if (cache.size() > 64) cache.clear();
    it = cache.emplace(key, std::move(R)).first;
  }
  return it->second.get();
}

// Ragged batches: valid rows of clip b after step k, by the reference's own length arithmetic (every conv floors:
// L_out = (L + 2p - d(K-1) - 1) / s + 1, so e.g. the stride-5 stage of the 12.5 Hz models maps 159 rows to 32)
std::vector<std::vector<int>> valid_rows_per_step(const kvae_plan* p, const std::vector<Step>& steps, const int* valid, int B) {
  std::vector<std::vector<int>> v(steps.size(), std::vector<int>(B));
  for (int b = 0; b < B; ++b) {
    int len = valid[b];
    for (size_t k = 0; k < steps.size(); ++k) {
      len = len > 0 ? std::max(0, p->convs[steps[k].conv].g.out_len(len)) : 0;
      v[k][b] = len;
    }
  }
  return v;
}

// zero the rows beyond each clip's valid length in the tensors step k has just written
cudaError_t zero_step_tails(const kvae_plan* p, const std::vector<Step>& steps, const PreparedRun& R, int k, int B,
                            long long T, void* ws, const std::vector<int>& valid_k, bool train, cudaStream_t st) {
  const Step& s = steps[k];
  const ConvLayer& c = p->convs[s.conv];
  const long long rows = step_len(s, T);
  uint8_t* base = static_cast<uint8_t*>(ws);
  const int split = (p->precision == KVAE_PREC_F32 && !train) ? 2 : 1;
  for (int which = 0; which < 2; ++which) {
    const Tensor& t = R.layout.t[1 + which + 2 * k];
    if (!t.bytes) continue;
    const int row_bytes = which == 0 ? c.g.Cout * (R.stream_f16 ? 2 : 4) : c.g.Cout * 2 * split;
    for (int b0 = 0; b0 < B; b0 += kRaggedMaxClips) {
      const int nb = std::min(kRaggedMaxClips, B - b0);
      RaggedLens lens;
      long long max_tail = 0;
      for (int i = 0; i < nb; ++i) {
        lens.v[i] = static_cast<int>(std::min<long long>(rows, valid_k[b0 + i]));
        max_tail = std::max(max_tail, rows - lens.v[i]);
      }
      if (max_tail <= 0) continue;
      const long long vecs = (max_tail * row_bytes + 15) / 16;
      const int blocks = static_cast<int>(std::min<long long>((vecs + 255) / 256, 4 * 148));
      zero_tail_rows_kernel<<<dim3(blocks, nb), 256, 0, st>>>(base + t.offset + static_cast<size_t>(b0) * rows * row_bytes,
                                                             rows * row_bytes, row_bytes, rows, lens);
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return e;
      ++g_launches;
    }
  }
  return cudaSuccess;
}

struct FusedSample { const void* noise = nullptr; void* out = nullptr; int D = 0; float std = 0.f; unsigned int* peak = nullptr; };

int run_plan(kvae_plan* p, bool train, const void* in, int in_dtype, void* out, int out_dtype, int B, long long T,
             void* ws, size_t ws_bytes, cudaStream_t st, const int* valid = nullptr, const FusedSample* fs = nullptr) {
  if (!p) return fail("null plan");
  if (B <= 0 || T <= 0) return fail("empty batch or zero length input");
  if (T > (1ll << 30)) return fail("input too long");
  for (const ConvLayer& c : p->convs)
    if (!c.set) return fail("plan weights not set (kvae_plan_set_conv / kvae_plan_load_params)");
  for (const SnakeLayer& s : p->snakes)
    if (!s.set) return fail("plan SnakeBeta parameters not set (kvae_plan_set_snake / kvae_plan_load_params)");
  if (train && !p->train_packs) return fail("training run needs kvae_plan_load_params(plan, params, train = 1)");
  if (train && p->direction == KVAE_DECODER && p->arch.final_tanh) return fail("final_tanh is not supported in training");
  if (train && p->direction == KVAE_DECODER && p->arch.use_nearest_upsample)
    return fail("use_nearest_upsample is inference-only (its folded taps have no weight-norm parameter layout)");
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail("cannot select device");
  const std::vector<Step>& steps = train ? p->tsteps : p->steps;
  const int n = static_cast<int>(steps.size());
  if (p->direction == KVAE_ENCODER && T % p->ratio) return fail("audio length must be a multiple of the downsampling ratio");
  std::string err;
  PreparedRun* Rp = get_run(p, train, B, T, ws, err);
  if (!Rp) return fail(err);
  PreparedRun& R = *Rp;
  if (ws_bytes < R.total) return fail("workspace too small");
  if (R.total > 1024 && !ws) return fail("null workspace");
  // boundary layout change for a tensor-core first layer
  const ConvLayer& c0 = p->convs[steps[0].conv];
  if (conv_tc(c0, train)) {
    dim3 grid(ceil_div(static_cast<int>(T), 32), ceil_div(c0.g.Cin, 32), B), block(32, 8);
    cf_to_cl_bf16_kernel<<<grid, block, 0, st>>>(in, in_dtype == KVAE_F32,
                                                 reinterpret_cast<__nv_bfloat16*>(static_cast<uint8_t*>(ws) + R.layout.t[0].offset),
                                                 c0.g.Cin, static_cast<int>(T), c0.umma ? 0 : 1);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  std::vector<std::vector<int>> valid_rows;
  if (valid) valid_rows = valid_rows_per_step(p, steps, valid, B);
  const bool prof = p->profile && !train;
  if (prof) {
    while (static_cast<int>(p->events.size()) < n + 1) {
      cudaEvent_t e;
      KV_CUDA(cudaEventCreate(&e));
      p->events.push_back(e);
    }
    KV_CUDA(cudaEventRecord(p->events[0], st));
    p->prof_B = B;
    p->prof_T = T;
    p->prof_valid = true;
  }
  for (int k = 0; k < n; ++k) {
    StepLaunch& S = R.steps[k];
    const bool f32_in = in_dtype == KVAE_F32, f32_out = out_dtype == KVAE_F32;
    switch (S.kind) {   // the caller's tensors
      case kWaveOutTc:
        S.wave_out_tc.y = out;
        S.wave_out_tc.y_f32 = f32_out;
        S.wave_out_tc.peak_bits = fs ? fs->peak : nullptr;
        break;
      case kWaveOut: S.wave_out.y = out; S.wave_out.y_f32 = f32_out; break;
      case kWaveInTc: S.head_col.x = in; S.head_col.x_f32 = f32_in; break;
      case kWaveIn: S.wave_in.x = in; S.wave_in.x_f32 = f32_in; break;
      case kTcConv:
        if (k == n - 1) {
          ConvParams2& cp = S.umma2.p;
          cp.out_cf = out;
          cp.out_cf_f32 = f32_out;
          cp.samp_noise = (fs && fs->out) ? fs->noise : nullptr;
          cp.samp_out = fs ? fs->out : nullptr;
          cp.samp_D = fs ? fs->D : 0;
          cp.samp_std = fs ? fs->std : 0.f;
        }
        break;
      case kDirect:
        if (k == 0) { S.direct.d.x = in; S.direct.d.x_f32 = f32_in; }
        if (k == n - 1) { S.direct.d.out_raw = out; S.direct.d.out_raw_f32 = f32_out; }
        break;
      default: break;
    }
    KV_CUDA(launch_step(S, p->convs[steps[k].conv].g, B, R.stream_f16, st));
    if (valid && k != n - 1) KV_CUDA(zero_step_tails(p, steps, R, k, B, T, ws, valid_rows[k], train, st));
    if (prof) KV_CUDA(cudaEventRecord(p->events[k + 1], st));
  }
  return 0;
}

// ------------------------------------------------------------------ backward pass (training plans)
// Walks tsteps in reverse.  G_k = gradient w.r.t. the raw (pre-activation) output of step k, fp32
// channels-last, plus a bf16 copy when a tensor-core kernel consumes it.  Per step k:
//   wgrad:  dW_k   = G_k (x) a_{k-1}          a_{k-1} = SnakeBeta(raw_{k-1}) as saved by the forward pass
//   dgrad:  dA     = conv^T(G_k, W_k)          the forward kernels under dgrad_geom() with re-packed weights
//   snake:  G_{k-1} = dA * SnakeBeta'(raw_{k-1}) + [G_{k+1} if step k+1 adds raw_{k-1} as its skip connection]
//           and, in the same pass, d alpha / d beta of that SnakeBeta and d bias of conv k-1 (= column sums of G_{k-1})
void set_sb_grid(SnakeBwdParams& sb, dim3& grid) {
  const int width = (sb.C % 4 == 0) ? sb.C / 4 : sb.C;   // float4 columns (vectorised kernel) or scalar columns
  int CW = 1;
  while (CW * 2 <= std::min(width, 256)) CW *= 2;
  sb.CW = CW;
  const int cols = ceil_div(width, CW);
  const int nrl = 256 / CW;
  // enough blocks to fill the machine, each with at least a few passes over its rows
  long long blocks_x = std::max<long long>(1, std::min<long long>((sb.rows + 8 * nrl - 1) / (8 * nrl),
                                                                     (8ll * sm_count() + cols - 1) / cols));
  long long rpb = (sb.rows + blocks_x - 1) / blocks_x;
  rpb = (rpb + nrl - 1) / nrl * nrl;
  blocks_x = (sb.rows + rpb - 1) / rpb;
  sb.rows_per_block = static_cast<int>(rpb);
  grid = dim3(static_cast<unsigned>(blocks_x), cols, 1);
}

cudaError_t launch_snake_bwd(const SnakeBwdParams& sb, dim3 grid, cudaStream_t st) {
  SnakeBwdStreamGeom gm;
  if (snake_bwd_stream_geom(sb, gm)) {
    static bool attr_set[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev & 63]) {
      cudaError_t e = cudaFuncSetAttribute(snake_bwd_stream_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(snake_bwd_stream_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return e;
      attr_set[dev & 63] = true;
    }
    long long ctas = std::min<long long>(gm.row_tiles, std::max(1, sm_count() / gm.ncol)) * gm.ncol;
    if (sb.fast) snake_bwd_stream_kernel<true><<<static_cast<unsigned>(ctas), kSbsThreads, snake_bwd_stream_smem(), st>>>(sb, gm);
    else snake_bwd_stream_kernel<false><<<static_cast<unsigned>(ctas), kSbsThreads, snake_bwd_stream_smem(), st>>>(sb, gm);
    return cudaGetLastError();
  }
  if (sb.C % 4 == 0) {
    if (sb.fast) snake_bwd_vec4_kernel<true><<<grid, 256, 0, st>>>(sb);
    else snake_bwd_vec4_kernel<false><<<grid, 256, 0, st>>>(sb);
  } else {
    snake_bwd_kernel<<<grid, 256, 0, st>>>(sb);
  }
  return cudaGetLastError();
}

// waveform-edge convs (C <-> io_channels, k7): HBM-streaming weight gradient (train.cuh::wgrad_edge_kernel)
bool edge_wgrad_ok(const ConvGeom& g) {
  const int thin = std::min(g.Cin, g.Cout), wide = std::max(g.Cin, g.Cout);
  return g.kind == kConv && g.stride == 1 && g.K <= kEdgeMaxK && thin <= 2 && wide >= 32 && wide <= 256 &&
         (wide & (wide - 1)) == 0;
}

void set_edge_grid(EdgeWgradParams& e, int& grid, size_t& smem) {
  const int per_clip = std::max(1, (8 * sm_count() + e.B - 1) / e.B);
  int rpb = std::max(256, (e.T + per_clip - 1) / per_clip);
  rpb = std::min(rpb, 4096);
  e.rows_per_block = rpb;
  e.blocks_per_clip = (e.T + rpb - 1) / rpb;
  grid = e.blocks_per_clip * e.B;
  const int halo = std::max(e.pad, (e.K - 1) * e.dil - e.pad);
  smem = static_cast<size_t>(rpb + 2 * halo) * 2 * sizeof(float);
}

bool prepare_backward(kvae_plan* p, int B, long long T, void* ws, PreparedRun& R, std::string& err) {
  const std::vector<Step>& steps = p->tsteps;
  const int n = static_cast<int>(steps.size());
  // backward region: three rotating gradient slots (fp32 + bf16) and one dA buffer, each of the largest size
  size_t max_elems = 0;
  for (int k = 0; k < n; ++k) {
    const ConvLayer& c = p->convs[steps[k].conv];
    max_elems = std::max(max_elems, static_cast<size_t>(B) * static_cast<size_t>(step_len(steps[k], T)) * c.g.Cout);
  }
  size_t off = align_up(R.layout.total, 1024);
  for (int i = 0; i < 3; ++i) { R.off_G[i] = off; off += align_up(max_elems * 4, 1024); }
  for (int i = 0; i < 3; ++i) { R.off_Gb[i] = off; off += align_up(max_elems * 2, 1024); }
  R.off_dA = off;
  off += align_up(max_elems * 4, 1024);
  R.total = off;
  uint8_t* base = static_cast<uint8_t*>(ws);
  auto tptr = [&](int id) -> void* { return R.layout.t[id].bytes ? base + R.layout.t[id].offset : nullptr; };
  auto Gf = [&](int k) { return reinterpret_cast<float*>(base + R.off_G[k % 3]); };
  auto Gb = [&](int k) { return reinterpret_cast<__nv_bfloat16*>(base + R.off_Gb[k % 3]); };
  float* dA = reinterpret_cast<float*>(base + R.off_dA);
  R.bwd.assign(n, PreparedRun::Bwd());
  {
    // incoming gradient (already transposed into Gf(n-1) at run time): bf16 copy + last conv's bias gradient
    const ConvLayer& c = p->convs[steps[n - 1].conv];
    SnakeBwdParams& sb = R.sb_last;
    std::memset(&sb, 0, sizeof(sb));
    sb.dA = Gf(n - 1);
    sb.Gb = Gb(n - 1);
    sb.rows = static_cast<long long>(B) * step_len(steps[n - 1], T);
    sb.C = c.g.Cout;
    set_sb_grid(sb, R.sb_last_grid);
  }
  for (int k = n - 1; k >= 0; --k) {
    const Step& s = steps[k];
    const ConvLayer& c = p->convs[s.conv];
    PreparedRun::Bwd& bw = R.bwd[k];
    const long long T_in = (k == 0) ? T : step_len(steps[k - 1], T);
    const long long T_out = step_len(s, T);
    // ---- weight gradient
    WgradParams& w = bw.wg;
    std::memset(&w, 0, sizeof(w));
    const void* a_ptr = nullptr;
    int a_f32 = 0;
    long long a_sB = T_in * c.g.Cin, a_sT = c.g.Cin, a_sC = 1;
    const float* a_sn = nullptr;
    const float* a_ib = nullptr;
    bool a_is_x = false;
    if (k == 0) {
      if (c.umma) {
        a_ptr = tptr(0);
      } else {   // the caller's input tensor, API layout [B, C, T]; pointer / dtype patched per call
        a_is_x = true;
        a_sB = static_cast<long long>(c.g.Cin) * T_in; a_sT = 1; a_sC = T_in;
      }
    } else if (steps[k - 1].needs_act) {
      a_ptr = tptr(2 + 2 * (k - 1));
    } else {
      a_ptr = tptr(1 + 2 * (k - 1));
      a_f32 = 1;
      if (s.pre_snake >= 0) { a_sn = p->snakes[s.pre_snake].a; a_ib = p->snakes[s.pre_snake].inv_b; }
    }
    if (!a_ptr && !a_is_x) { err = "internal: saved operand missing at step " + std::to_string(k); return false; }
    const float* g_ptr = Gf(k);
    const long long g_sB = T_out * c.g.Cout, g_sT = c.g.Cout;
    if (c.g.kind == kConv) {
      w.D = g_ptr; w.D_f32 = 1; w.D_sB = g_sB; w.D_sT = g_sT; w.D_sC = 1;
      w.S = a_ptr; w.S_f32 = a_f32; w.S_sB = a_sB; w.S_sT = a_sT; w.S_sC = a_sC; w.S_a = a_sn; w.S_inv_b = a_ib;
      w.Td = static_cast<int>(T_out); w.Ts = static_cast<int>(T_in); w.Cd = c.g.Cout; w.Cs = c.g.Cin;
      bw.wg_x_is_S = a_is_x;
    } else {
      w.D = a_ptr; w.D_f32 = a_f32; w.D_sB = a_sB; w.D_sT = a_sT; w.D_sC = a_sC; w.D_a = a_sn; w.D_inv_b = a_ib;
      w.S = g_ptr; w.S_f32 = 1; w.S_sB = g_sB; w.S_sT = g_sT; w.S_sC = 1;
      w.Td = static_cast<int>(T_in); w.Ts = static_cast<int>(T_out); w.Cd = c.g.Cin; w.Cs = c.g.Cout;
      bw.wg_x_is_D = a_is_x;
    }
    w.B = B; w.K = c.g.K; w.stride = c.g.stride; w.dil = c.g.dilation; w.pad = c.g.pad;
    if (c.off_dwp >= 0) {
      // tensor-core weight gradient: bf16 operands (saved activation, bf16 copy of the gradient), MN-major
      if (a_f32 || a_is_x) { err = "internal: bf16 operand missing for the tensor-core weight gradient"; return false; }
      bw.wg_kind = 1;
      const __nv_bfloat16* ab = static_cast<const __nv_bfloat16*>(a_ptr);
      const bool conv = c.g.kind == kConv;
      if (!prepare_wgrad_umma(conv ? Gb(k) : ab, w.Td, w.Cd, conv ? ab : Gb(k), w.Ts, w.Cs, B, c.g.K, c.g.stride,
                              c.g.dilation, c.g.pad, p->dwp + c.off_dwp, bw.wg_umma, err))
        return false;
    } else if (edge_wgrad_ok(c.g) && ((c.g.Cout <= 2 && a_f32 && !a_is_x) || (c.g.Cin <= 2 && a_is_x))) {
      bw.wg_kind = 2;
      EdgeWgradParams& e = bw.wg_edge;
      std::memset(&e, 0, sizeof(e));
      e.B = B; e.T = static_cast<int>(T_out); e.K = c.g.K; e.dil = c.g.dilation; e.pad = c.g.pad;
      if (c.g.Cout <= 2) {   // decoder tail: wide = SnakeBeta(stream), thin = output gradient (channels-last)
        e.W = static_cast<const float*>(a_ptr); e.W_a = a_sn; e.W_inv_b = a_ib; e.C = c.g.Cin;
        e.W_f16 = R.stream_f16 ? 1 : 0;
        e.fast_sin = (p->precision == KVAE_PREC_BF16) ? 1 : 0;
        e.N = g_ptr; e.N_f32 = 1; e.N_sB = g_sB; e.N_sT = g_sT; e.N_sC = 1;
        e.sigma = 1; e.out_wide_first = 0;
      } else {               // encoder head: wide = gradient of the stream, thin = the caller's waveform (API layout)
        e.W = g_ptr; e.C = c.g.Cout;
        e.N = nullptr; e.N_sB = a_sB; e.N_sT = a_sT; e.N_sC = a_sC;
        e.sigma = -1; e.out_wide_first = 1;
        bw.wg_edge_x_is_thin = true;
      }
      set_edge_grid(e, bw.wg_edge_grid, bw.wg_edge_smem);
      if (e.W_f16 && !(e.C % 4 == 0 && e.C / 4 >= 8 && e.C / 4 <= 256 && ((e.C / 4) & (e.C / 4 - 1)) == 0)) {
        err = "internal: fp16 training stream with an edge conv the vectorised weight-gradient kernel does not cover";
        return false;
      }
    } else {
      if (R.stream_f16 && a_f32) { err = "internal: fp16 training stream reaches a CUDA-core weight gradient"; return false; }
      const int tiles = ceil_div(w.Cd, 64) * ceil_div(w.Cs, 64);
      const long long rows = static_cast<long long>(B) * w.Td;
      long long nsplit = std::max<long long>(1, (4ll * sm_count()) / (static_cast<long long>(tiles) * w.K));
      nsplit = std::min(nsplit, (rows + 4 * kWgRows - 1) / (4 * kWgRows));
      nsplit = std::max<long long>(1, std::min<long long>(nsplit, 65535));
      long long rps = (rows + nsplit - 1) / nsplit;
      rps = (rps + kWgRows - 1) / kWgRows * kWgRows;
      nsplit = (rows + rps - 1) / rps;
      w.rows_per_split = rps;
      bw.wg_grid = dim3(tiles, w.K, static_cast<unsigned>(nsplit));
    }
    // ---- data gradient (k == 0: only when the caller asks for the input gradient; patched per call)
    const ConvGeom gd = dgrad_geom(c.g, static_cast<int>(T_in));
    if (gd.out_len(static_cast<int>(T_out)) != T_in) { err = "internal: dgrad length bookkeeping"; return false; }
    // bf16 mode: dA crosses HBM as bf16 (written by the data-gradient conv's fragment-mapped epilogue, read by the
    // vectorised SnakeBeta backward)
    const bool da_bf16 = c.umma && k >= 1 && p->precision == KVAE_PREC_BF16 && c.g.Cin % 4 == 0;
    if (c.umma) {
      bw.dgrad_kind = 1;
      ConvEpilogue ep;
      if (da_bf16) {
        ep.out_act = reinterpret_cast<__nv_bfloat16*>(dA);
      } else {
        ep.out_raw = (k == 0) ? reinterpret_cast<void*>(0x1) : static_cast<void*>(dA);
        ep.out_raw_f32 = 1;
        ep.out_raw_cf = (k == 0) ? 1 : 0;
      }
      ConvTuning2 tune;
      if (!prepare_conv_umma2(gd, Gb(k), B, static_cast<int>(T_out), c.w_umma_d, ep, tune, bw.dg_umma, err)) return false;
    } else if (k > 0 && edge_wgrad_ok(c.g) && c.g.Cout <= 2) {
      bw.dgrad_kind = 3;
      EdgeDgradParams& e = bw.dg_edge;
      std::memset(&e, 0, sizeof(e));
      e.gy = Gf(k); e.w = c.w_direct; e.dA = dA;
      e.B = B; e.T = static_cast<int>(T_out); e.C = c.g.Cin; e.K = c.g.K; e.dil = c.g.dilation; e.pad = c.g.pad;
      EdgeWgradParams tmp;
      std::memset(&tmp, 0, sizeof(tmp));
      tmp.B = B; tmp.T = e.T; tmp.K = e.K; tmp.dil = e.dil; tmp.pad = e.pad;
      set_edge_grid(tmp, bw.dg_edge_grid, bw.dg_edge_smem);
      e.rows_per_block = tmp.rows_per_block; e.blocks_per_clip = tmp.blocks_per_clip;
    } else {
      bw.dgrad_kind = 2;
      if (!prepare_direct(gd, B, T_out, T_in, 0, bw.dg_direct, err)) return false;
      DirectParams& d = bw.dg_direct.d;
      d.x = Gf(k); d.x_f32 = 1;
      d.x_sB = T_out * gd.Cin; d.x_sT = gd.Cin; d.x_sC = 1;
      d.w = c.w_direct_d;
      if (k == 0) {   // input gradient in the API layout
        d.out_raw = nullptr;
        d.o_sB = static_cast<long long>(gd.Cout) * T_in; d.o_sT = 1; d.o_sC = T_in;
      } else {
        d.out_raw = dA; d.out_raw_f32 = 1;
        d.o_sB = T_in * gd.Cout; d.o_sT = gd.Cout; d.o_sC = 1;
      }
    }
    // ---- SnakeBeta backward producing G_{k-1}
    if (k >= 1) {
      const ConvLayer& cp = p->convs[steps[k - 1].conv];
      SnakeBwdParams& sb = bw.sb;
      std::memset(&sb, 0, sizeof(sb));
      bw.has_sb = true;
      sb.dA = dA;
      sb.dA_bf16 = da_bf16 ? 1 : 0;
      if (s.pre_snake >= 0) {
        const SnakeLayer& sn = p->snakes[s.pre_snake];
        sb.x = static_cast<const float*>(tptr(1 + 2 * (k - 1)));
        sb.x_f16 = R.stream_f16 ? 1 : 0;
        if (sb.x_f16 && c.g.Cin % 8) { err = "internal: fp16 training stream needs channel counts that are multiples of 8"; return false; }
        if (!sb.x) { err = "internal: saved stream missing at step " + std::to_string(k - 1); return false; }
        sb.a = sn.a; sb.inv_b = sn.inv_b; sb.logscale = sn.logscale;
      }
      for (int j = k + 1; j < n; ++j)
        if (steps[j].residual_from == k - 1) {
          if (j != k + 1) { err = "internal: skip connection spans more than one ResidualUnit"; return false; }
          sb.skip = Gf(j);
          // bf16 mode: read the bf16 copy of that gradient (it exists whenever step j runs on the tensor cores)
          if (p->convs[steps[j].conv].umma && p->precision == KVAE_PREC_BF16 && c.g.Cin % 4 == 0) {
            sb.skip = reinterpret_cast<const float*>(Gb(j));
            sb.skip_bf16 = 1;
          }
        }
      // fp32 copy of G_{k-1}: only where something reads it -- the skip-connection add two steps later (k-1 is the
      // k1 conv of a ResidualUnit), the CUDA-core kernels, or the input-gradient of step 0
      // (the skip-connection reader takes the bf16 copy in bf16 mode, see above)
      bool skip_reader_bf16 = false;
      if (steps[k - 1].residual_from >= 0 && p->precision == KVAE_PREC_BF16) {
        const int rf = steps[k - 1].residual_from;          // G_{k-1} is added into G_{rf} by the pass at step rf + 1
        skip_reader_bf16 = cp.umma && rf + 1 < n && p->convs[steps[rf + 1].conv].g.Cin % 4 == 0;
      }
      const bool tc_only = cp.umma && cp.off_dwp >= 0 && (steps[k - 1].residual_from < 0 || skip_reader_bf16);
      sb.G = tc_only ? nullptr : Gf(k - 1);
      sb.Gb = cp.umma ? Gb(k - 1) : nullptr;
      sb.rows = static_cast<long long>(B) * T_in;
      sb.C = c.g.Cin;
      sb.fast = (p->precision == KVAE_PREC_BF16) ? 1 : 0;
      set_sb_grid(sb, bw.sb_grid);
      // Fuse this pass into the data-gradient conv's epilogue when its only product is the bf16 gradient: tensor-core
      // dgrad with 128-channel tiles, fp16 saved stream, bf16 skip gradient (or none), no fp32 copy of G wanted.
      if (bw.dgrad_kind == 1 && da_bf16 && sb.a && sb.x_f16 && !sb.G && sb.Gb && (!sb.skip || sb.skip_bf16) &&
          gd.Cout % 128 == 0) {
        ConvEpilogue ep;
        ep.out_act = sb.Gb;
        ep.bwd_x = sb.x;
        ep.bwd_skip = sb.skip;
        ep.bwd_a = sb.a;
        ep.bwd_inv_b = sb.inv_b;
        ep.bwd_logscale = sb.logscale;
        ConvTuning2 tune;
        ConvLaunch2 fused;
        std::string ferr;
        if (prepare_conv_umma2(gd, Gb(k), B, static_cast<int>(T_out), c.w_umma_d, ep, tune, fused, ferr)) {
          bw.dg_umma = fused;
          bw.sb_fused = true;
        }
      }
    }
  }
  return true;
}

int run_backward(kvae_plan* p, const void* x, int x_dtype, const void* gy, int gy_dtype, void* gx, int gx_dtype, int B,
                 long long T, void* ws, size_t ws_bytes, float* grads, const float* params, cudaStream_t st) {
  if (!p) return fail("null plan");
  if (!gy || !grads || !x) return fail("null argument");
  if (!p->train_packs) return fail("backward needs kvae_plan_load_params(plan, params, train = 1)");
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail("cannot select device");
  std::string err;
  PreparedRun* Rp = get_run(p, true, B, T, ws, err);
  if (!Rp) return fail(err);
  PreparedRun& R = *Rp;
  if (ws_bytes < R.total) return fail("workspace too small");
  const std::vector<Step>& steps = p->tsteps;
  const int n = static_cast<int>(steps.size());
  uint8_t* base = static_cast<uint8_t*>(ws);
  KV_CUDA(cudaMemsetAsync(grads, 0, static_cast<size_t>(p->n_params) * 4, st));
  if (p->dwp_floats) KV_CUDA(cudaMemsetAsync(p->dwp, 0, p->dwp_floats * 4, st));
  {
    // grad_out [B, C, T_last] -> channels-last fp32, then bf16 copy + bias gradient of the last conv
    const ConvLayer& c = p->convs[steps[n - 1].conv];
    const long long T_last = step_len(steps[n - 1], T);
    float* G = reinterpret_cast<float*>(base + R.off_G[(n - 1) % 3]);
    dim3 grid(static_cast<unsigned>((T_last + 31) / 32), ceil_div(c.g.Cout, 32), B), block(32, 8);
    cf_to_cl_f32_kernel<<<grid, block, 0, st>>>(gy, gy_dtype == KVAE_F32, G, c.g.Cout, T_last);
    KV_CUDA(cudaGetLastError());
    SnakeBwdParams sb = R.sb_last;
    if (!c.umma) sb.Gb = nullptr;
    sb.d_bias = c.has_bias ? grads + c.off_bias : nullptr;
    if (sb.Gb || sb.d_bias) {
      KV_CUDA(launch_snake_bwd(sb, R.sb_last_grid, st));
      ++g_launches;
    }
    ++g_launches;
  }
  for (int k = n - 1; k >= 0; --k) {
    const Step& s = steps[k];
    const ConvLayer& c = p->convs[s.conv];
    PreparedRun::Bwd& bw = R.bwd[k];
    if (bw.wg_kind == 1) {
      KV_CUDA(launch_wgrad_umma(bw.wg_umma, st));
      ++g_launches;
    } else if (bw.wg_kind == 2) {
      EdgeWgradParams e = bw.wg_edge;
      if (bw.wg_edge_x_is_thin) { e.N = x; e.N_f32 = (x_dtype == KVAE_F32); }
      e.dW = grads + c.off_v;
      const int C4 = e.C / 4;
      const bool vec = e.C % 4 == 0 && C4 >= 8 && C4 <= 256 && (C4 & (C4 - 1)) == 0;
      if (vec) {
        // + the lane-reduction scratch: 256 threads x NT x 4 floats behind the thin rows
        const size_t smem = bw.wg_edge_smem + 16 + 256 * 2 * 4 * sizeof(float);
        if (std::min(c.g.Cin, c.g.Cout) == 1) wgrad_edge_vec4_kernel<1><<<bw.wg_edge_grid, 256, smem, st>>>(e);
        else wgrad_edge_vec4_kernel<2><<<bw.wg_edge_grid, 256, smem, st>>>(e);
      } else if (std::min(c.g.Cin, c.g.Cout) == 1) wgrad_edge_kernel<1><<<bw.wg_edge_grid, 256, bw.wg_edge_smem, st>>>(e);
      else wgrad_edge_kernel<2><<<bw.wg_edge_grid, 256, bw.wg_edge_smem, st>>>(e);
      KV_CUDA(cudaGetLastError());
      ++g_launches;
    } else {
      WgradParams w = bw.wg;
      if (bw.wg_x_is_D) { w.D = x; w.D_f32 = (x_dtype == KVAE_F32); }
      if (bw.wg_x_is_S) { w.S = x; w.S_f32 = (x_dtype == KVAE_F32); }
      w.dW = grads + c.off_v;
      wgrad_direct_kernel<<<bw.wg_grid, 256, 0, st>>>(w);
      KV_CUDA(cudaGetLastError());
      ++g_launches;
    }
    if (k == 0 && !gx) break;
    if (bw.dgrad_kind == 3) {
      if (c.g.Cout == 1) dgrad_edge_kernel<1><<<bw.dg_edge_grid, 256, bw.dg_edge_smem, st>>>(bw.dg_edge);
      else dgrad_edge_kernel<2><<<bw.dg_edge_grid, 256, bw.dg_edge_smem, st>>>(bw.dg_edge);
      KV_CUDA(cudaGetLastError());
    } else if (bw.dgrad_kind == 1) {
      ConvLaunch2& L = bw.dg_umma;
      if (k == 0) { L.p.out_cf = gx; L.p.out_cf_f32 = (gx_dtype == KVAE_F32); }
      if (bw.sb_fused) {
        const ConvLayer& cp = p->convs[steps[k - 1].conv];
        L.p.d_alpha = grads + p->snakes[s.pre_snake].off_alpha;
        L.p.d_beta = grads + p->snakes[s.pre_snake].off_beta;
        L.p.d_bias = cp.has_bias ? grads + cp.off_bias : nullptr;
      }
      KV_CUDA(launch_conv_umma2(L, st));
    } else {
      DirectParams& d = bw.dg_direct.d;
      if (k == 0) { d.out_raw = gx; d.out_raw_f32 = (gx_dtype == KVAE_F32); }
      KV_CUDA(launch_direct(bw.dg_direct, st));
    }
    ++g_launches;
    if (bw.has_sb && !bw.sb_fused) {
      SnakeBwdParams sb = bw.sb;
      const ConvLayer& cp = p->convs[steps[k - 1].conv];
      if (s.pre_snake >= 0) {
        sb.d_alpha = grads + p->snakes[s.pre_snake].off_alpha;
        sb.d_beta = grads + p->snakes[s.pre_snake].off_beta;
      }
      sb.d_bias = cp.has_bias ? grads + cp.off_bias : nullptr;
      KV_CUDA(launch_snake_bwd(sb, bw.sb_grid, st));
      ++g_launches;
    }
  }
  // weight-norm backward: dW (folded-weight gradient; in place in the weight_v slot, or packed by the
  // tensor-core kernel) -> (dv, dg); without params the packed gradients are only re-ordered
  if (!p->wn_desc) {
    std::vector<WnBwdDesc> wd(p->convs.size());
    int rows = 0;
    for (size_t i = 0; i < p->convs.size(); ++i) {
      const ConvLayer& c = p->convs[i];
      const int R = c.dim0();
      wd[i].off_v = c.off_v; wd[i].off_g = c.off_g; wd[i].off_dwp = c.off_dwp;
      wd[i].R = R; wd[i].Cc = static_cast<int>(c.numel() / c.g.K / R); wd[i].K = c.g.K; wd[i].row0 = rows;
      rows += R;
    }
    KV_CUDA(cudaMalloc(&p->wn_desc, wd.size() * sizeof(WnBwdDesc)));
    KV_CUDA(cudaMemcpy(p->wn_desc, wd.data(), wd.size() * sizeof(WnBwdDesc), cudaMemcpyHostToDevice));
    p->wn_rows = rows;
  }
  weight_norm_bwd_all_kernel<<<p->wn_rows, 256, 0, st>>>(params, grads, p->dwp, p->wn_desc, static_cast<int>(p->convs.size()));
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

bool check_dtype(int d) { return d == KVAE_F32 || d == KVAE_BF16; }

// fp32 CUDA-core weight gradient of a layer-level Conv1d / ConvTranspose1d straight from the API layout [B, C, T]:
// dw (torch layout, overwritten) from x (T rows) and gy, the gradient of the output rows [0, T_gy) (rows past T_gy,
// a causal layer's dropped rows, have none).
cudaError_t launch_wgrad_direct_cf(const void* x, const void* gy, int f32, float* dw, int transposed, int B, int Cin, int Cout,
                                   long long T, long long T_gy, int K, int stride, int dilation, int padding, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(dw, 0, static_cast<size_t>(Cin) * Cout * K * 4, st);
  if (e != cudaSuccess) return e;
  const long long xsB = static_cast<long long>(Cin) * T, gsB = static_cast<long long>(Cout) * T_gy;
  WgradParams wp;
  std::memset(&wp, 0, sizeof(wp));
  if (!transposed) {
    wp.D = gy; wp.D_sB = gsB; wp.D_sT = 1; wp.D_sC = T_gy; wp.Td = static_cast<int>(T_gy); wp.Cd = Cout;
    wp.S = x; wp.S_sB = xsB; wp.S_sT = 1; wp.S_sC = T; wp.Ts = static_cast<int>(T); wp.Cs = Cin;
  } else {
    wp.D = x; wp.D_sB = xsB; wp.D_sT = 1; wp.D_sC = T; wp.Td = static_cast<int>(T); wp.Cd = Cin;
    wp.S = gy; wp.S_sB = gsB; wp.S_sT = 1; wp.S_sC = T_gy; wp.Ts = static_cast<int>(T_gy); wp.Cs = Cout;
  }
  wp.D_f32 = wp.S_f32 = f32;
  wp.dW = dw; wp.B = B; wp.K = K; wp.stride = stride; wp.dil = dilation; wp.pad = padding;
  const int tiles = ceil_div(wp.Cd, 64) * ceil_div(wp.Cs, 64);
  const long long rows = static_cast<long long>(B) * wp.Td;
  long long nsplit = std::max<long long>(1, (4ll * sm_count()) / (static_cast<long long>(tiles) * K));
  nsplit = std::max<long long>(1, std::min<long long>(std::min(nsplit, (rows + 4 * kWgRows - 1) / (4 * kWgRows)), 65535));
  long long rps = (rows + nsplit - 1) / nsplit;
  rps = (rps + kWgRows - 1) / kWgRows * kWgRows;
  nsplit = (rows + rps - 1) / rps;
  wp.rows_per_split = rps;
  wgrad_direct_kernel<<<dim3(tiles, K, static_cast<unsigned>(nsplit)), 256, 0, st>>>(wp);
  ++g_launches;
  return cudaGetLastError();
}

#include "stream.inc.cuh"

}  // namespace

// =============================================================================== C ABI
extern "C" {

int kvae_version(void) { return 100; }
const char* kvae_last_error(void) { return g_err.c_str(); }

int kvae_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ++ok;
  }
  return ok;
}

long long kvae_launch_count(int reset) {
  const long long v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

int kvae_plan_create(const kvae_arch* arch, int direction, int precision, int device, kvae_plan** out) {
  if (!arch || !out) return fail("null argument");
  if (direction != KVAE_ENCODER && direction != KVAE_DECODER) return fail("bad direction");
  if (precision != KVAE_PREC_BF16 && precision != KVAE_PREC_F32) return fail("bad precision");
  if (arch->n_stages < 1 || arch->n_stages > KVAE_MAX_STAGES) return fail("n_stages out of range");
  if (arch->io_channels < 1 || arch->channels < 1 || arch->latent_dim < 1) return fail("bad channel counts");
  for (int i = 0; i < arch->n_stages; ++i) {
    if (arch->strides[i] < 1 || arch->strides[i] > kMaxPhases) return fail("stride out of range (1..8)");
    if (arch->c_mults[i] < 1) return fail("bad c_mult");
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail("no CUDA device: libkvae has no CPU path");
  }
  if (device < 0 || device >= ndev) return fail("bad device index");
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  if (major != 10) return fail("device is not sm_100 (B200): libkvae is built for sm_100a only");
  auto p = std::make_unique<kvae_plan>();
  p->arch = *arch;
  p->direction = direction;
  p->precision = precision;
  p->device = device;
  if (direction == KVAE_DECODER) build_decoder(p.get());
  else build_encoder(p.get());
  finalize_steps(p.get());
  if (direction == KVAE_DECODER && arch->final_tanh && (p->convs.back().umma || p->convs.back().umma32))
    return fail("final_tanh with a tensor-core output conv is not supported");
  DeviceGuard guard(device);
  if (!guard.ok) return fail("cannot select device");
  for (ConvLayer& c : p->convs) {
    const size_t n = static_cast<size_t>(c.g.Cin) * c.g.Cout * c.g.K;
    if (c.umma) KV_CUDA(cudaMalloc(&c.w_umma, n * 2));
    else KV_CUDA(cudaMalloc(&c.w_direct, n * 4));
    if (c.umma32) KV_CUDA(cudaMalloc(&c.w_umma, n * 2 * 2));      // (hi | lo) halves
    if (!c.umma && !c.umma32 && c.g.K == 7 && c.g.Cin <= 2) KV_CUDA(cudaMalloc(&c.w_head, static_cast<size_t>(c.g.Cout) * 64 * 2));
    if (c.has_bias) KV_CUDA(cudaMalloc(&c.bias, c.g.Cout * 4));
  }
  for (SnakeLayer& s : p->snakes) {
    KV_CUDA(cudaMalloc(&s.a, s.C * 4));
    KV_CUDA(cudaMalloc(&s.inv_b, s.C * 4));
  }
  *out = p.release();
  return 0;
}

void kvae_plan_destroy(kvae_plan* p) {
  if (!p) return;
  DeviceGuard guard(p->device);
  for (cudaEvent_t e : p->events) cudaEventDestroy(e);
  for (ConvLayer& c : p->convs) {
    cudaFree(c.w_umma);
    cudaFree(c.w_direct);
    cudaFree(c.w_head);
    cudaFree(c.w_umma_d);
    cudaFree(c.w_direct_d);
    cudaFree(c.bias);
  }
  for (SnakeLayer& s : p->snakes) {
    cudaFree(s.a);
    cudaFree(s.inv_b);
  }
  cudaFree(p->scale_scratch);
  cudaFree(p->fold_desc);
  cudaFree(p->snake_desc);
  cudaFree(p->scale_all);
  cudaFree(p->wn_desc);
  cudaFree(p->dwp);
  delete p;
}

int kvae_plan_num_convs(const kvae_plan* p) { return p ? static_cast<int>(p->convs.size()) : fail("null plan"); }
int kvae_plan_num_snakes(const kvae_plan* p) { return p ? static_cast<int>(p->snakes.size()) : fail("null plan"); }

int kvae_plan_conv_info(const kvae_plan* p, int idx, int info[8]) {
  if (!p || !info) return fail("null argument");
  if (idx < 0 || idx >= static_cast<int>(p->convs.size())) return fail("conv index out of range");
  const ConvLayer& c = p->convs[idx];
  info[0] = c.g.kind; info[1] = c.g.Cin; info[2] = c.g.Cout; info[3] = c.g.K;
  info[4] = c.g.stride; info[5] = c.g.dilation; info[6] = c.g.pad; info[7] = c.has_bias ? 1 : 0;
  return 0;
}
int kvae_plan_snake_channels(const kvae_plan* p, int idx) {
  if (!p) return fail("null plan");
  if (idx < 0 || idx >= static_cast<int>(p->snakes.size())) return fail("snake index out of range");
  return p->snakes[idx].C;
}

int kvae_plan_set_conv(kvae_plan* p, int idx, const float* w, const float* bias, void* stream) {
  if (!p || !w) return fail("null argument");
  if (idx < 0 || idx >= static_cast<int>(p->convs.size())) return fail("conv index out of range");
  ConvLayer& c = p->convs[idx];
  if (c.has_bias && !bias) return fail("this conv has a bias");
  if (!c.has_bias && bias) return fail("this conv has no bias (bias=False in the reference)");
  DeviceGuard guard(p->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t n = static_cast<size_t>(c.g.Cin) * c.g.Cout * c.g.K;
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 4096));
  pack_weights_kernel<<<blocks, 256, 0, st>>>(w, c.g.kind == kConvT, c.g.Cout, c.g.Cin, c.g.K, c.umma ? c.w_umma : nullptr,
                                              c.w_direct);
  KV_CUDA(cudaGetLastError());
  if (c.umma32) {
    split_pack_kernel<<<blocks, 256, 0, st>>>(c.w_direct, c.g.K, c.g.Cin, c.g.Cout, c.w_umma);
    KV_CUDA(cudaGetLastError());
  }
  if (bias) KV_CUDA(cudaMemcpyAsync(c.bias, bias, c.g.Cout * 4, cudaMemcpyDeviceToDevice, st));
  c.set = true;
  return 0;
}

int kvae_plan_set_snake(kvae_plan* p, int idx, const float* alpha, const float* beta, int logscale, void* stream) {
  if (!p || !alpha || !beta) return fail("null argument");
  if (idx < 0 || idx >= static_cast<int>(p->snakes.size())) return fail("snake index out of range");
  SnakeLayer& s = p->snakes[idx];
  DeviceGuard guard(p->device);
  snake_params_kernel<<<ceil_div(s.C, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(alpha, beta, logscale, s.C,
                                                                                        s.a, s.inv_b);
  KV_CUDA(cudaGetLastError());
  s.logscale = logscale ? 1 : 0;
  s.set = true;
  return 0;
}

size_t kvae_workspace_bytes(kvae_plan* p, int B, long long T) {
  if (!p || B <= 0 || T <= 0) { fail("bad argument"); return 0; }
  Layout L;
  std::string err;
  if (!make_layout(p, p->steps, false, B, T, L, err)) { fail(err); return 0; }
  return L.total;
}

int kvae_decode(kvae_plan* p, const void* z, int z_dtype, void* wav, int wav_dtype, int B, long long T, void* ws,
                size_t ws_bytes, void* stream) {
  if (!p) return fail("null plan");
  if (p->direction != KVAE_DECODER) return fail("plan is not a decoder");
  if (!z || !wav) return fail("null tensor");
  if (!check_dtype(z_dtype) || !check_dtype(wav_dtype)) return fail("bad dtype");
  return run_plan(p, false, z, z_dtype, wav, wav_dtype, B, T, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

int kvae_encode(kvae_plan* p, const void* wav, int wav_dtype, void* lat, int lat_dtype, int B, long long L, void* ws,
                size_t ws_bytes, void* stream) {
  if (!p) return fail("null plan");
  if (p->direction != KVAE_ENCODER) return fail("plan is not an encoder");
  if (!wav || !lat) return fail("null tensor");
  if (!check_dtype(wav_dtype) || !check_dtype(lat_dtype)) return fail("bad dtype");
  return run_plan(p, false, wav, wav_dtype, lat, lat_dtype, B, L, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

static int check_valid(const int* valid, int B, long long T) {
  if (!valid) return fail("null valid_len");
  for (int b = 0; b < B; ++b)
    if (valid[b] < 0 || valid[b] > T) return fail("valid_len out of range (0 .. padded length)");
  return 0;
}

int kvae_decode_ragged(kvae_plan* p, const void* z, int z_dtype, void* wav, int wav_dtype, int B, long long T,
                       const int* valid_len, void* ws, size_t ws_bytes, void* stream) {
  if (!p) return fail("null plan");
  if (p->direction != KVAE_DECODER) return fail("plan is not a decoder");
  if (!z || !wav) return fail("null tensor");
  if (!check_dtype(z_dtype) || !check_dtype(wav_dtype)) return fail("bad dtype");
  if (B > 0 && T > 0 && check_valid(valid_len, B, T)) return -1;
  return run_plan(p, false, z, z_dtype, wav, wav_dtype, B, T, ws, ws_bytes, static_cast<cudaStream_t>(stream), valid_len);
}

int kvae_encode_ragged(kvae_plan* p, const void* wav, int wav_dtype, void* lat, int lat_dtype, int B, long long L,
                       const int* valid_len, void* ws, size_t ws_bytes, void* stream) {
  if (!p) return fail("null plan");
  if (p->direction != KVAE_ENCODER) return fail("plan is not an encoder");
  if (!wav || !lat) return fail("null tensor");
  if (!check_dtype(wav_dtype) || !check_dtype(lat_dtype)) return fail("bad dtype");
  if (B > 0 && L > 0 && check_valid(valid_len, B, L)) return -1;
  return run_plan(p, false, wav, wav_dtype, lat, lat_dtype, B, L, ws, ws_bytes, static_cast<cudaStream_t>(stream), valid_len);
}

long long kvae_plan_out_length(const kvae_plan* p, long long T) {
  if (!p) return fail("null plan");
  long long len = T;
  for (const Step& st : p->steps) {
    if (len <= 0 || len > (1ll << 30)) return 0;
    len = p->convs[st.conv].g.out_len(static_cast<int>(len));
  }
  return len > 0 ? len : 0;
}

int kvae_prep_mono_clips(const float* wav, const long long* offsets, const int* lens, int B, long long L_pad, int channels,
                         float gain, float* out, void* scratch, void* stream) {
  if (!wav || !offsets || !lens || !out || !scratch) return fail("null argument");
  if (B <= 0 || L_pad <= 0 || channels <= 0) return fail("empty input");
  DeviceGuard guard(device_of(out));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  KV_CUDA(cudaMemsetAsync(scratch, 0, static_cast<size_t>(B) * 4, st));
  const int blocks = static_cast<int>(std::min<long long>((L_pad + 255) / 256, 2 * 148));
  clip_peak_kernel<<<dim3(blocks, B), 256, 0, st>>>(wav, offsets, lens, static_cast<unsigned int*>(scratch));
  KV_CUDA(cudaGetLastError());
  clip_normalize_dup_kernel<<<dim3(blocks, B), 256, 0, st>>>(wav, offsets, lens, static_cast<const unsigned int*>(scratch),
                                                            gain, out, L_pad, channels);
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  return 0;
}

int kvae_encode_sample(kvae_plan* p, const void* wav, int wav_dtype, void* lat, void* z, const void* noise, int lat_dtype,
                       int D, float std, int B, long long L, void* ws, size_t ws_bytes, void* stream) {
  if (!p) return fail("null plan");
  if (p->direction != KVAE_ENCODER) return fail("plan is not an encoder");
  if (!wav || !lat || !z || !noise) return fail("null tensor");
  if (!check_dtype(wav_dtype) || !check_dtype(lat_dtype)) return fail("bad dtype");
  if (D <= 0 || D > p->arch.latent_dim) return fail("D must be in 1 .. latent_dim");
  const ConvLayer& cl = p->convs[p->steps.back().conv];
  if (!conv_tc(cl, false))
    return fail("fused sampling needs a tensor-core output conv (use kvae_encode + kvae_sigma_sample)");
  FusedSample fs;
  fs.noise = noise; fs.out = z; fs.D = D; fs.std = std;
  return run_plan(p, false, wav, wav_dtype, lat, lat_dtype, B, L, ws, ws_bytes, static_cast<cudaStream_t>(stream), nullptr, &fs);
}

int kvae_plan_fused_sample_supported(const kvae_plan* p) {
  if (!p) return 0;
  return p->direction == KVAE_ENCODER && conv_tc(p->convs[p->steps.back().conv], false) ? 1 : 0;
}

double kvae_plan_flops(const kvae_plan* p, int B, long long T) {
  if (!p) return 0.0;
  double f = 0.0;
  for (size_t k = 0; k < p->steps.size(); ++k) {
    const Step& s = p->steps[k];
    const ConvGeom& g = p->convs[s.conv].g;
    const double T_in = (k == 0) ? static_cast<double>(T) : static_cast<double>(step_len(p->steps[k - 1], T));
    const double T_out = static_cast<double>(step_len(s, T));
    const double rows = (g.kind == kConv) ? T_out : T_in;
    f += 2.0 * B * rows * g.Cin * g.Cout * g.K;
  }
  return f;
}

static double step_flops(const kvae_plan* p, size_t k, int B, long long T) {
  const Step& s = p->steps[k];
  const ConvGeom& g = p->convs[s.conv].g;
  const double T_in = (k == 0) ? static_cast<double>(T) : static_cast<double>(step_len(p->steps[k - 1], T));
  const double T_out = static_cast<double>(step_len(s, T));
  const double rows = (g.kind == kConv) ? T_out : T_in;
  return 2.0 * B * rows * g.Cin * g.Cout * g.K;
}

int kvae_plan_profile(kvae_plan* p, int enable) {
  if (!p) return fail("null plan");
  p->profile = enable != 0;
  p->prof_valid = false;
  return 0;
}

int kvae_plan_step_profile(kvae_plan* p, float* ms, double* flops, int* tensor_core, int max_steps) {
  if (!p || !ms || !flops || !tensor_core) return fail("null argument");
  if (!p->prof_valid) return fail("no profiled run recorded (kvae_plan_profile(plan, 1), then run)");
  const int n = static_cast<int>(p->steps.size());
  if (max_steps < n) return fail("output arrays too small");
  DeviceGuard guard(p->device);
  KV_CUDA(cudaEventSynchronize(p->events[n]));
  for (int k = 0; k < n; ++k) {
    KV_CUDA(cudaEventElapsedTime(&ms[k], p->events[k], p->events[k + 1]));
    flops[k] = step_flops(p, k, p->prof_B, p->prof_T);
    tensor_core[k] = conv_tc(p->convs[p->steps[k].conv], false) ? 1 : 0;
  }
  return n;
}

// ------------------------------------------------------------------ layer level
int kvae_snake_fwd(const void* x, void* y, const float* alpha, const float* beta, int logscale, int B, int C,
                   long long T, int dtype, void* stream) {
  if (!x || !y || !alpha || !beta) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || C <= 0 || T <= 0) return 0;  // empty tensor: nothing to do
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  if (static_cast<long long>(B) * C > 65535) return fail("B*C too large");
  dim3 grid(static_cast<unsigned>((T + 1023) / 1024), B * C);
  snake_cf_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, alpha, beta, logscale, C, T,
                                                                       dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_weight_norm_fold(const float* v, const float* g, float* w, int dim0, int inner, void* stream) {
  if (!v || !g || !w) return fail("null argument");
  if (dim0 <= 0 || inner <= 0) return 0;
  DeviceGuard guard(device_of(v));
  if (!guard.ok) return fail("cannot select the tensor's device");
  weight_norm_fold_kernel<<<dim0, 256, 0, static_cast<cudaStream_t>(stream)>>>(v, g, w, inner);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

size_t kvae_conv1d_scratch_bytes(int Cin, int Cout, int K) {
  return align_up(static_cast<size_t>(Cin) * Cout * K * 4, 1024);
}

int kvae_conv1d_tc_supported(int Cin, int Cout, int K, int stride, int dilation, int transposed) {
  ConvGeom g{transposed ? kConvT : kConv, Cin, Cout, K, stride, dilation, 0};
  if (!umma_supported(g) || stride < 1 || stride > kMaxPhases || K > kMaxTaps) return 0;
  if (stride > 1 && dilation != 1) return 0;
  return 1;
}

// Layer-level conv with packed weights (kvae_conv1d_pack) on the CUDA cores or the tensor cores: output rows [o0, o1)
// of the conv of a pitched T-row input, written pitched.  Engines: 0 = CUDA cores fp32 (conv_direct_kernel),
// 1 = tcgen05 bf16, 2 = tcgen05 bf16 x 3 split (<= 1e-5).  A whole layer is the range [0, keep) of a contiguous input:
// keep = the natural output length, or less for the causal layers of flows.py (symmetric padding d (K - 1), first T
// outputs; transposed kernel 2 s, last s outputs dropped), which the kernel truncates without a slicing copy.
namespace {
size_t win_pack_main_bytes(int Cin, int Cout, int K, int engine) {
  const size_t n = static_cast<size_t>(Cin) * Cout * K;
  return engine == 0 ? align_up(n * 4, 1024) : align_up(n * 2 * (engine == 2 ? 2 : 1), 1024);
}

// kvae_conv1d_pack's layout for `engine`; w is read as [Cin, Cout, K] (transposed) or [Cout, Cin, K], tap k packed at
// K - 1 - k when flip_taps.  The data gradient of a layer packs the layer's weight under the opposite kind with Cin and
// Cout exchanged (kvae_conv1d_win_bwd).
int pack_conv_weights(const float* w, int transposed, int Cin, int Cout, int K, int engine, int flip_taps, void* packed,
                      cudaStream_t st) {
  const size_t n = static_cast<size_t>(Cin) * Cout * K;
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 4096));
  uint8_t* base = static_cast<uint8_t*>(packed);
  auto pack = flip_taps ? pack_weights_kernel<true> : pack_weights_kernel<false>;
  if (engine == 0) {
    pack<<<blocks, 256, 0, st>>>(w, transposed, Cout, Cin, K, nullptr, reinterpret_cast<float*>(base));
  } else if (engine == 1) {
    pack<<<blocks, 256, 0, st>>>(w, transposed, Cout, Cin, K, reinterpret_cast<__nv_bfloat16*>(base), nullptr);
  } else {
    float* w_direct = reinterpret_cast<float*>(base + win_pack_main_bytes(Cin, Cout, K, 2));
    pack<<<blocks, 256, 0, st>>>(w, transposed, Cout, Cin, K, nullptr, w_direct);
    KV_CUDA(cudaGetLastError());
    split_pack_kernel<<<blocks, 256, 0, st>>>(w_direct, K, Cin, Cout, reinterpret_cast<__nv_bfloat16*>(base));
    ++g_launches;
  }
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}
}  // namespace

size_t kvae_conv1d_packed_bytes(int Cin, int Cout, int K, int engine) {
  if (engine < 0 || engine > 2) return 0;
  const size_t n = static_cast<size_t>(Cin) * Cout * K;
  return win_pack_main_bytes(Cin, Cout, K, engine) + (engine == 2 ? align_up(n * 4, 1024) : 0);
}

int kvae_conv1d_pack(const float* w, int transposed, int Cin, int Cout, int K, int engine, void* packed,
                     size_t packed_bytes, void* stream) {
  if (!w || !packed) return fail("null argument");
  if (engine < 0 || engine > 2) return fail("engine: 0 = CUDA cores, 1 = tcgen05 bf16, 2 = tcgen05 bf16x3");
  if (Cin <= 0 || Cout <= 0 || K <= 0) return fail("empty weight");
  if (packed_bytes < kvae_conv1d_packed_bytes(Cin, Cout, K, engine)) return fail("packed buffer too small");
  DeviceGuard guard(device_of(w));
  if (!guard.ok) return fail("cannot select the tensor's device");
  return pack_conv_weights(w, transposed, Cin, Cout, K, engine, 0, packed, static_cast<cudaStream_t>(stream));
}

size_t kvae_conv1d_win_scratch_bytes(int B, int Cin, long long T, int engine) {
  if (engine == 0) return 0;
  return align_up(static_cast<size_t>(B) * T * Cin * 2 * (engine == 2 ? 2 : 1), 1024);
}

namespace {
// The layer-level conv: output rows [o0, o1) of the conv of a stream whose rows [x0, x0 + nx) the window x holds
// ([B, Cin] rows at pitch ldx), with weights packed for `engine` (kvae_conv1d_pack), written to y ([B, Cout] rows at
// pitch ldy, row o0 first).  Rows < 0 and, when t_end >= 0, rows >= t_end read as zero; a whole layer is the window
// x0 = 0, nx = t_end = T.  The callers check the arguments (every row the outputs read lies in the window or reads as
// zero; x0 a multiple of the stride of a strided conv) and select the device.  A tcgen05 call for the full range of a
// whole layer whose input is whole stride groups runs with no StreamGeom, which keeps the whole-row set-up of the
// strided convs; any other call (a strided conv's input of any length included) copies its window into scratch rounded
// up to whole stride groups, the rows that read as zero written as zeros.  staged (tcgen05, split 1 only): scratch
// already holds that channels-last window (kvae_conv1d_win_bwd shares it with the weight gradient).
int conv1d_rows(const ConvGeom& g, const void* x, long long ldx, long long x0, long long nx, long long t_end, void* y,
                long long ldy, const void* packed, const float* bias, int B, long long o0, long long o1, int dtype,
                int engine, void* scratch, size_t scratch_bytes, cudaStream_t st, bool staged = false) {
  if (engine == 0) {
    DirectLaunch L;
    std::string err;
    const long long x_hi = t_end < 0 ? x0 + nx : std::min(t_end, x0 + nx);
    if (!prepare_direct(g, B, x_hi, o1, o0, L, err)) return fail(err);
    DirectParams& d = L.d;
    // stream row ti is column ti - x0 of the window: the kernel reads x moved back by x0 rows.  It reads rows
    // [0, x_hi) only; rows below the window are never read, because the lowest row of each tile's slab is a tap of
    // its first output, and the callers check that every row a requested output reads is in the window or < 0.
    d.x = static_cast<const char*>(x) - x0 * (dtype == KVAE_F32 ? 4 : 2); d.x_f32 = (dtype == KVAE_F32);
    d.x_sB = static_cast<long long>(g.Cin) * ldx; d.x_sT = 1; d.x_sC = ldx;
    d.w = static_cast<const float*>(packed); d.bias = bias;
    d.out_raw = y; d.out_raw_f32 = (dtype == KVAE_F32);
    d.o_sB = static_cast<long long>(g.Cout) * ldy; d.o_sT = 1; d.o_sC = ldy;
    KV_CUDA(launch_direct(L, st));
    ++g_launches;
    return 0;
  }
  const int transposed = g.kind == kConvT;
  if (!kvae_conv1d_tc_supported(g.Cin, g.Cout, g.K, g.stride, g.dilation, transposed))
    return fail("tcgen05 engine: the layer needs channel counts that are multiples of 64");
  const int P_out = transposed ? g.stride : 1, P_in = transposed ? 1 : g.stride;
  if (o0 % P_out || o1 % P_out) return fail("tcgen05 engine: o0 and o1 must be multiples of the stride (transposed)");
  const bool full = x0 == 0 && t_end == nx && nx % P_in == 0 && o0 == 0 && o1 == g.out_len(static_cast<int>(nx));
  const long long W = full ? nx : (nx + P_in - 1) / P_in * P_in;
  StreamGeom sg;                 // rows q of the window's output from o0 / P_out on: taps shifted by that many rows
  sg.in_rows = static_cast<int>(W);
  sg.out_q = static_cast<int>((o1 - o0) / P_out);
  sg.row_bias = static_cast<int>(o0 / P_out - x0 / P_in);
  if (sg.row_bias < -16384 || sg.row_bias > 16384) return fail("tcgen05 engine: outputs too far from the window origin");
  if (scratch_bytes < kvae_conv1d_win_scratch_bytes(B, g.Cin, W, engine) || !scratch) return fail("scratch too small");
  const int split = engine == 2 ? 2 : 1;
  __nv_bfloat16* xcl = static_cast<__nv_bfloat16*>(scratch);
  if (!staged) {
    const long long lo = std::max(0LL, -x0), hi = t_end < 0 ? nx : std::min(nx, t_end - x0);
    dim3 grid(ceil_div(static_cast<int>(W), 32), ceil_div(g.Cin, 32), B), block(32, 8);
    cf_to_cl_bf16_kernel<<<grid, block, 0, st>>>(x, dtype == KVAE_F32, xcl, g.Cin, static_cast<int>(W),
                                                 split == 2 ? 1 : 0, 0, ldx, static_cast<int>(lo),
                                                 static_cast<int>(std::max(lo, hi)));
    KV_CUDA(cudaGetLastError());
  }
  ConvEpilogue ep;
  ep.bias = bias;
  ep.out_raw = y;
  ep.out_raw_cf = 1;
  ep.out_raw_f32 = (dtype == KVAE_F32);
  if (split == 2) { ep.split3 = 1; ep.precise = 1; }
  ConvTuning2 tune;
  ConvLaunch2 L;
  std::string err;
  if (!prepare_conv_umma2(g, xcl, B, static_cast<int>(W), static_cast<const __nv_bfloat16*>(packed), ep, tune, L, err,
                          full ? nullptr : &sg))
    return fail(err);
  L.p.cf_ld = ldy;
  KV_CUDA(launch_conv_umma2(L, st));
  g_launches += 2;
  return 0;
}
}  // namespace

int kvae_conv1d_win_fwd(const void* x, long long ldx, void* y, long long ldy, const void* packed, const float* bias,
                        int transposed, int B, int Cin, int Cout, long long T, int K, int stride, int dilation,
                        int padding, long long o0, long long o1, int dtype, int engine, void* scratch,
                        size_t scratch_bytes, void* stream) {
  if (!x || !y || !packed) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (engine < 0 || engine > 2) return fail("engine: 0 = CUDA cores, 1 = tcgen05 bf16, 2 = tcgen05 bf16x3");
  if (B <= 0 || Cin <= 0 || Cout <= 0 || K <= 0 || T <= 0) return fail("empty input");
  if (stride < 1 || stride > kMaxPhases) return fail("stride out of range (1..8)");
  if (!transposed && stride != 1 && o0 != 0) return fail("a strided conv (not transposed) starts at o0 = 0");
  if (ldx < T) return fail("ldx < T");
  ConvGeom g{transposed ? kConvT : kConv, Cin, Cout, K, stride, dilation, padding};
  const long long T_nat = g.out_len(static_cast<int>(T));
  // the tcgen05 engines write whole stride groups of a transposed conv: its last group may run past T_nat (odd K - s
  // without causal truncation), those rows being the conv's own continuation over zero input rows
  const long long o_max = transposed && engine ? (T_nat + stride - 1) / stride * stride : T_nat;
  if (o0 < 0 || o1 <= o0 || o1 > o_max)
    return fail("output rows must satisfy 0 <= o0 < o1 <= the conv's output length (rounded up to whole stride groups "
                "for a transposed conv on the tcgen05 engines)");
  if (ldy < o1 - o0) return fail("ldy < o1 - o0");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  return conv1d_rows(g, x, ldx, 0, T, T, y, ldy, packed, bias, B, o0, o1, dtype, engine, scratch, scratch_bytes,
                     static_cast<cudaStream_t>(stream));
}

size_t kvae_conv1d_stream_scratch_bytes(int B, int Cin, long long nx, int stride, int engine) {
  if (stride < 1 || nx < 0) return 0;
  return kvae_conv1d_win_scratch_bytes(B, Cin, (nx + stride - 1) / stride * stride, engine);
}

int kvae_conv1d_stream_fwd(const void* x, long long ldx, long long x0, long long nx, void* y, long long ldy,
                           long long o0, long long o1, long long t_end, const void* packed, const float* bias,
                           int B, int Cin, int Cout, int K, int stride, int dilation, int padding,
                           int dtype, int engine, void* scratch, size_t scratch_bytes, void* stream) {
  if (!x || !y || !packed) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (engine < 0 || engine > 2) return fail("engine: 0 = CUDA cores, 1 = tcgen05 bf16, 2 = tcgen05 bf16x3");
  if (B <= 0 || Cin <= 0 || Cout <= 0 || K <= 0 || nx <= 0) return fail("empty input");
  if (stride < 1 || stride > kMaxPhases) return fail("stride out of range (1..8)");
  if (dilation < 1 || padding < 0) return fail("dilation >= 1 and padding >= 0");
  if (x0 % stride) return fail("the window origin x0 must be a multiple of the stride");
  if (ldx < nx) return fail("ldx < nx");
  if (o0 < 0 || o1 <= o0) return fail("output rows must satisfy 0 <= o0 < o1");
  if (ldy < o1 - o0) return fail("ldy < o1 - o0");
  const long long lim = 1LL << 30;   // the kernels address rows in 32 bits
  if (x0 <= -lim || x0 + nx >= lim || o1 * stride >= lim || t_end >= lim) return fail("rows beyond 2^30");
  ConvGeom g{kConv, Cin, Cout, K, stride, dilation, padding};
  if (t_end >= 0 && o1 > g.out_len(static_cast<int>(t_end))) return fail("output rows past the stream's output length");
  // every input row a requested output reads, [o0 s - p, (o1 - 1) s - p + d (K - 1)], that does not read as zero
  // must lie in the window
  const long long lo = std::max(0LL, o0 * stride - padding);
  long long hi = (o1 - 1) * stride - padding + static_cast<long long>(dilation) * (K - 1);
  if (t_end >= 0) hi = std::min(hi, t_end - 1);
  if (lo <= hi && (lo < x0 || hi >= x0 + nx))
    return fail("the window does not hold every input row the requested outputs read");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  return conv1d_rows(g, x, ldx, x0, nx, t_end, y, ldy, packed, bias, B, o0, o1, dtype, engine, scratch, scratch_bytes,
                     static_cast<cudaStream_t>(stream));
}

int kvae_conv1d_fwd(const void* x, void* y, const float* w, const float* bias, int transposed, int B, int Cin,
                    int Cout, long long T, int K, int stride, int dilation, int padding, int dtype, void* scratch,
                    size_t scratch_bytes, void* stream) {
  if (!x || !y || !w || !scratch) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || Cin <= 0 || Cout <= 0 || K <= 0 || T <= 0) return fail("empty input");
  if (stride < 1 || stride > kMaxPhases) return fail("stride out of range (1..8)");
  if (scratch_bytes < kvae_conv1d_scratch_bytes(Cin, Cout, K)) return fail("scratch too small");
  ConvGeom g{transposed ? kConvT : kConv, Cin, Cout, K, stride, dilation, padding};
  const long long T_out = g.out_len(static_cast<int>(T));
  if (T_out <= 0) return fail("input shorter than the kernel");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t n = static_cast<size_t>(Cin) * Cout * K;
  pack_weights_kernel<<<static_cast<int>(std::min<size_t>((n + 255) / 256, 4096)), 256, 0, st>>>(
      w, transposed, Cout, Cin, K, nullptr, static_cast<float*>(scratch));
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return conv1d_rows(g, x, T, 0, T, T, y, T_out, scratch, bias, B, 0, T_out, dtype, 0, nullptr, 0, st);
}

// ------------------------------------------------------------------ layer-level conv backward
namespace {
// The data gradient of a layer as a conv over the layer's output gradient gy (run by conv1d_rows, rows of gy past its
// end reading as zero):
//   Conv1d, stride 1, padding pl: gx = the conv of gy with the weight transposed ([Cin, Cout, K]) and its taps
//     reversed, same dilation, left padding d (K - 1) - pl (negative when pl > d (K - 1): gx reads gy ahead);
//   Conv1d, stride s > 1, dilation 1, padding p: gx = the ConvTranspose1d of gy with the same weight (read as the
//     transposed conv's [Cin', Cout', K] = [Cout, Cin, K]), stride s, padding p, continued past its natural length over
//     zero gy rows to the layer's T input rows (torch's output_padding): those rows are input rows the forward read;
//   ConvTranspose1d, stride s, padding p: gx = the strided Conv1d of gy with the same weight, stride s, padding p.
// conv_direct_kernel takes any tap offset; the tcgen05 engines take padding <= d (K - 1) only (kvae_conv1d_win_bwd).
struct DgradGeom {
  ConvGeom g;      // Cin = the layer's Cout, Cout = the layer's Cin; kConvT for a strided Conv1d, else kConv
  int flip;        // the weight's taps reversed (Conv1d of stride 1)
};
bool dgrad_conv_geom(int transposed, int Cin, int Cout, int K, int stride, int dilation, int padding, DgradGeom& d,
                     std::string& err) {
  if (Cin <= 0 || Cout <= 0 || K <= 0 || dilation < 1) { err = "conv backward: empty layer"; return false; }
  if (stride < 1 || stride > kMaxPhases) { err = "stride out of range (1..8)"; return false; }
  if (padding < 0) { err = "conv backward: negative padding"; return false; }
  if (!transposed && stride > 1) {
    if (dilation != 1) { err = "conv backward: a strided Conv1d of dilation 1 only"; return false; }
    d.g = ConvGeom{kConvT, Cout, Cin, K, stride, 1, padding};
    d.flip = 0;
  } else if (!transposed) {
    d.g = ConvGeom{kConv, Cout, Cin, K, 1, dilation, dilation * (K - 1) - padding};
    d.flip = 1;
  } else {
    if (dilation != 1) { err = "conv backward: ConvTranspose1d of dilation 1 only"; return false; }
    d.g = ConvGeom{kConv, Cout, Cin, K, stride, 1, padding};
    d.flip = 0;
  }
  return true;
}

long long round_up_ll(long long v, long long m) { return (v + m - 1) / m * m; }

// gx [B, Cin, T] of `dtype` of a layer (`transposed`, its data-gradient geometry d) from gy [B, Cout, T_gy] on
// `engine`: the layer's weight w packed under the opposite kind into wpk (kvae_conv1d_packed_bytes(Cout, Cin, K,
// engine)), then rows [0, T) of the conv d.g of gy.  gcl / gcl_bytes: conv1d_rows' scratch; engine 1 expects gy already
// staged there channels-last.  The tcgen05 engines emit whole stride groups of a transposed conv: a strided Conv1d's gx
// of T rows not whole groups is computed into gx_groups and its rows [0, T) are copied out.
int conv1d_dgrad(int transposed, const DgradGeom& d, const void* gy, long long T_gy, const float* w, void* gx, int B,
                 long long T, int dtype, int engine, void* wpk, void* gcl, size_t gcl_bytes, void* gx_groups,
                 cudaStream_t st) {
  if (pack_conv_weights(w, !transposed, d.g.Cin, d.g.Cout, d.g.K, engine, d.flip, wpk, st)) return -1;
  const long long To = engine && d.g.kind == kConvT ? round_up_ll(T, d.g.stride) : T;
  if (conv1d_rows(d.g, gy, T_gy, 0, T_gy, T_gy, To != T ? gx_groups : gx, To, wpk, nullptr, B, 0, To, dtype, engine, gcl,
                  gcl_bytes, st, engine == 1))
    return -1;
  if (To != T) {
    const size_t es = dtype == KVAE_F32 ? 4 : 2;
    KV_CUDA(cudaMemcpy2DAsync(gx, T * es, gx_groups, To * es, T * es, static_cast<size_t>(B) * d.g.Cout,
                              cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}
}  // namespace

int kvae_conv1d_dgrad_geom(int transposed, int Cin, int Cout, int K, int stride, int dilation, int padding, int out[6]) {
  if (!out) return fail("null argument");
  if (!transposed && stride != 1)
    return fail("conv backward: a strided Conv1d's data gradient is a ConvTranspose1d (kvae_conv1d_dgrad_form)");
  int f[7];
  if (kvae_conv1d_dgrad_form(transposed, Cin, Cout, K, stride, dilation, padding, f)) return -1;
  std::memcpy(out, f + 1, 6 * sizeof(int));
  return 0;
}

int kvae_conv1d_dgrad_form(int transposed, int Cin, int Cout, int K, int stride, int dilation, int padding, int out[7]) {
  if (!out) return fail("null argument");
  DgradGeom d;
  std::string err;
  if (!dgrad_conv_geom(transposed, Cin, Cout, K, stride, dilation, padding, d, err)) return fail(err);
  const int v[7] = {d.g.kind == kConvT, d.g.Cin, d.g.Cout, d.g.stride, d.g.dilation, d.g.pad, d.flip};
  std::memcpy(out, v, sizeof(v));
  return 0;
}

size_t kvae_conv1d_win_bwd_scratch_bytes(int transposed, int B, int Cin, int Cout, long long T, long long T_gy, int K,
                                         int stride, int engine) {
  if (engine < 0 || engine > 2 || B <= 0 || Cin <= 0 || Cout <= 0 || K <= 0 || T <= 0 || T_gy <= 0 || stride < 1) return 0;
  const long long Tg = round_up_ll(T_gy, transposed ? stride : 1), Tx = round_up_ll(T, transposed ? 1 : stride);
  size_t bytes = kvae_conv1d_packed_bytes(Cout, Cin, K, engine) + kvae_conv1d_win_scratch_bytes(B, Cout, Tg, engine) +
                 align_up(static_cast<size_t>(Cin) * Cout * K * 4, 1024);
  if (engine == 1) bytes += align_up(static_cast<size_t>(B) * Tx * Cin * 2, 1024);
  if (engine && Tx != T) bytes += align_up(static_cast<size_t>(B) * Cin * Tx * 4, 1024);   // gx in whole stride groups
  return bytes;
}

int kvae_conv1d_win_bwd(const void* x, const void* gy, long long T_gy, const float* w, const float* v, const float* g,
                        void* gx, float* dv, float* dg, float* dbias, int transposed, int B, int Cin, int Cout, long long T,
                        int K, int stride, int dilation, int padding, int dtype, int engine, void* scratch,
                        size_t scratch_bytes, void* stream) {
  if (!gy) return fail("null argument");
  if (!gx && !dv && !dbias) return fail("nothing to compute (gx, dv and dbias are all null)");
  if ((gx && !w) || (dv && !x) || (g && (!v || !dg))) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (engine < 0 || engine > 2) return fail("engine: 0 = CUDA cores, 1 = tcgen05 bf16, 2 = tcgen05 bf16x3");
  if (B <= 0 || Cin <= 0 || Cout <= 0 || K <= 0 || T <= 0) return fail("empty input");
  DgradGeom dgg;
  std::string err;
  if (!dgrad_conv_geom(transposed, Cin, Cout, K, stride, dilation, padding, dgg, err)) return fail(err);
  if (engine && padding > dilation * (K - 1)) return fail("tcgen05 engines: conv backward padding outside 0 .. d (K - 1)");
  const ConvGeom lg{transposed ? kConvT : kConv, Cin, Cout, K, stride, dilation, padding};
  if (T >= (1LL << 30) || lg.out_len(static_cast<int>(T)) >= (1LL << 30)) return fail("rows beyond 2^30");
  if (T_gy < 1 || T_gy > lg.out_len(static_cast<int>(T))) return fail("T_gy outside 1 .. the layer's output length");
  if (engine && !kvae_conv1d_tc_supported(Cin, Cout, K, stride, dilation, transposed))
    return fail("tcgen05 engine: the layer needs channel counts that are multiples of 64");
  if (!scratch || scratch_bytes < kvae_conv1d_win_bwd_scratch_bytes(transposed, B, Cin, Cout, T, T_gy, K, stride, engine))
    return fail("scratch too small");
  DeviceGuard guard(device_of(gy));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int f32 = dtype == KVAE_F32;
  // gy staged in whole stride groups of the data-gradient conv (a strided Conv1d; a transposed one reads single rows),
  // x (the weight gradient's strided operand) in whole stride groups of the layer
  const long long Tg = round_up_ll(T_gy, dgg.g.kind == kConv ? dgg.g.stride : 1);
  const long long Tx = round_up_ll(T, transposed ? 1 : stride);
  uint8_t* base = static_cast<uint8_t*>(scratch);
  void* wpk = base;
  base += kvae_conv1d_packed_bytes(Cout, Cin, K, engine);
  __nv_bfloat16* gcl = reinterpret_cast<__nv_bfloat16*>(base);
  const size_t gcl_bytes = kvae_conv1d_win_scratch_bytes(B, Cout, Tg, engine);
  base += gcl_bytes;
  float* dW = reinterpret_cast<float*>(base);
  base += align_up(static_cast<size_t>(Cin) * Cout * K * 4, 1024);
  __nv_bfloat16* xcl = reinterpret_cast<__nv_bfloat16*>(base);
  if (engine == 1) base += align_up(static_cast<size_t>(B) * Tx * Cin * 2, 1024);
  void* gx_groups = base;     // tcgen05 data gradient of a strided Conv1d whose T is not whole stride groups
  if (dbias) {
    bias_grad_cf_kernel<<<Cout, 256, 0, st>>>(gy, f32, dbias, B, Cout, T_gy);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  // engine 1: gy channels-last bf16 once, the data-gradient conv's input and a weight-gradient operand
  if (engine == 1 && (gx || dv)) {
    dim3 grid(ceil_div(static_cast<int>(Tg), 32), ceil_div(Cout, 32), B), block(32, 8);
    cf_to_cl_bf16_kernel<<<grid, block, 0, st>>>(gy, f32, gcl, Cout, static_cast<int>(Tg), 0, 0, T_gy, 0,
                                                 static_cast<int>(T_gy));
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  if (dv) {
    const int R = transposed ? Cin : Cout, Cc = transposed ? Cout : Cin;   // dim 0 of the torch weight and the rest
    if (engine == 1) {
      // tensor-core weight gradient into the packed [K][R][Cc] layout, then the weight-norm backward from it
      // rows [T, Tx) (a strided layer's last stride group) written as zeros
      dim3 grid(ceil_div(static_cast<int>(Tx), 32), ceil_div(Cin, 32), B), block(32, 8);
      cf_to_cl_bf16_kernel<<<grid, block, 0, st>>>(x, f32, xcl, Cin, static_cast<int>(Tx), 0, 0, T, 0, static_cast<int>(T));
      KV_CUDA(cudaGetLastError());
      ++g_launches;
      KV_CUDA(cudaMemsetAsync(dW, 0, static_cast<size_t>(Cin) * Cout * K * 4, st));
      WgradLaunch L;
      const bool ok = transposed
          ? prepare_wgrad_umma(xcl, static_cast<int>(T), Cin, gcl, static_cast<int>(Tg), Cout, B, K, stride, dilation, padding, dW, L, err)
          : prepare_wgrad_umma(gcl, static_cast<int>(T_gy), Cout, xcl, static_cast<int>(Tx), Cin, B, K, stride, dilation, padding, dW, L, err);
      if (!ok) return fail(err);
      KV_CUDA(launch_wgrad_umma(L, st));
      ++g_launches;
      weight_norm_bwd_packed_kernel<<<R, 256, 0, st>>>(v, g, dW, dv, g ? dg : nullptr, R, Cc, K);
      KV_CUDA(cudaGetLastError());
      ++g_launches;
    } else {
      // fp32 CUDA cores (engine 0, and engine 2, whose bf16x3 split would take three tensor-core passes)
      KV_CUDA(launch_wgrad_direct_cf(x, gy, f32, g ? dW : dv, transposed, B, Cin, Cout, T, T_gy, K, stride, dilation,
                                     padding, st));
      if (g) {
        weight_norm_bwd_kernel<<<R, 256, 0, st>>>(v, g, dW, dv, dg, Cc * K);
        KV_CUDA(cudaGetLastError());
        ++g_launches;
      }
    }
  }
  if (!gx) return 0;
  return conv1d_dgrad(transposed, dgg, gy, T_gy, w, gx, B, T, dtype, engine, wpk, gcl, gcl_bytes, gx_groups, st);
}

// ------------------------------------------------------------------ multi-resolution STFT loss (mrstft.cuh)
namespace {
int mrstft_signals(int B, int C, int sum_diff) { return sum_diff ? 2 * B : B * C; }
}
size_t kvae_mrstft_scratch_bytes(int B, int C, long long T, int n_res, int sum_diff, int want_grad) {
  if (B <= 0 || C <= 0 || T <= 0 || n_res <= 0) return 0;
  const size_t M = static_cast<size_t>(mrstft_signals(B, C, sum_diff));
  const size_t sig = align_up(M * static_cast<size_t>(T) * 4, 1024);
  return (want_grad ? 4 : 2) * sig + align_up(static_cast<size_t>(n_res) * M * 3 * 8, 1024);
}

int kvae_mrstft_loss(const void* input, const void* target, int B, int C, long long T, int dtype, int n_res,
                     const int* fft_sizes, const int* hop_sizes, const float* windows, const float* fir_taps, int n_taps,
                     int sum_diff, float w_sum, float w_diff, float w_sc, float w_log_mag, float* loss, float* grad_input,
                     float* grad_target, void* scratch, size_t scratch_bytes, void* stream) {
  if (!input || !target || !fft_sizes || !hop_sizes || !windows || !loss || !scratch) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || C <= 0 || T <= 0) return fail("empty input");
  if (n_res <= 0 || n_res > kStftMaxRes) return fail("mrstft: 1..16 resolutions");
  if (sum_diff && C != 2) return fail("mrstft: the sum-and-difference form needs stereo input");
  if (n_taps < 0 || n_taps > kFirMaxTaps || (n_taps && !(n_taps & 1)) || (n_taps && !fir_taps)) return fail("mrstft: the pre-filter needs an odd number of taps <= 129");
  const bool want_grad = grad_input || grad_target;
  if (scratch_bytes < kvae_mrstft_scratch_bytes(B, C, T, n_res, sum_diff, want_grad)) return fail("scratch too small");
  const int M = mrstft_signals(B, C, sum_diff);
  if (M > 65535) return fail("mrstft: too many signals");
  StftRes res[kStftMaxRes];
  for (int r = 0; r < n_res; ++r) {
    const int n = fft_sizes[r];
    int l2 = 0;
    while ((1 << l2) < n) ++l2;
    if (n < 8 || n > kStftMaxN || (1 << l2) != n) return fail("mrstft: fft sizes must be powers of two in [8, 2048]");
    if (hop_sizes[r] <= 0) return fail("mrstft: bad hop size");
    if (T <= n / 2) return fail("mrstft: signal shorter than half an fft frame (reflect padding)");
    res[r] = StftRes{n, l2, hop_sizes[r], static_cast<int>(1 + T / hop_sizes[r])};
  }
  DeviceGuard guard(device_of(input));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t sig = align_up(static_cast<size_t>(M) * T * 4, 1024);
  uint8_t* sp = static_cast<uint8_t*>(scratch);
  float* Xf = reinterpret_cast<float*>(sp);
  float* Yf = reinterpret_cast<float*>(sp + sig);
  float* gX = want_grad ? reinterpret_cast<float*>(sp + 2 * sig) : nullptr;
  float* gY = want_grad ? reinterpret_cast<float*>(sp + 3 * sig) : nullptr;
  double* sums = reinterpret_cast<double*>(sp + (want_grad ? 4 : 2) * sig);
  KV_CUDA(cudaMemsetAsync(sums, 0, static_cast<size_t>(n_res) * M * 3 * 8, st));
  KV_CUDA(cudaMemsetAsync(loss, 0, 4, st));
  if (want_grad) KV_CUDA(cudaMemsetAsync(gX, 0, 2 * sig, st));
  const dim3 pgrid(static_cast<unsigned>((T + kFirTile - 1) / kFirTile), M);
  const int f32 = dtype == KVAE_F32;
  mrstft_prep_kernel<<<pgrid, 256, 0, st>>>(input, f32, sum_diff, B, T, fir_taps, n_taps, Xf);
  mrstft_prep_kernel<<<pgrid, 256, 0, st>>>(target, f32, sum_diff, B, T, fir_taps, n_taps, Yf);
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  const int Mg = sum_diff ? B : M, n_groups = sum_diff ? 2 : 1;
  const float wg0 = sum_diff ? 0.5f * w_sum : 1.f, wg1 = sum_diff ? 0.5f * w_diff : 1.f;
  const float* win = windows;
  for (int r = 0; r < n_res; ++r) {
    const int fpb = kStftMaxN / res[r].n;
    const dim3 grid((res[r].frames + fpb - 1) / fpb, M);
    mrstft_fwd_kernel<<<grid, 256, 0, st>>>(Xf, Yf, win, res[r], T, sums + static_cast<size_t>(r) * M * 3);
    mrstft_finish_kernel<<<1, 256, 0, st>>>(sums + static_cast<size_t>(r) * M * 3, M, Mg, w_sc, w_log_mag, wg0, wg1, n_groups,
                                            1.0 / n_res, static_cast<double>(res[r].n / 2 + 1) * res[r].frames, loss);
    win += res[r].n;
    g_launches += 2;
  }
  KV_CUDA(cudaGetLastError());
  if (!want_grad) return 0;
  win = windows;
  for (int r = 0; r < n_res; ++r) {
    const int fpb = kStftMaxN / res[r].n;
    const dim3 grid((res[r].frames + fpb - 1) / fpb, M);
    mrstft_bwd_kernel<<<grid, 256, 0, st>>>(Xf, Yf, win, res[r], T, sums + static_cast<size_t>(r) * M * 3, Mg, w_sc, w_log_mag,
                                            wg0, wg1, n_groups, 1.f / n_res, grad_input ? gX : nullptr, grad_target ? gY : nullptr);
    win += res[r].n;
    ++g_launches;
  }
  KV_CUDA(cudaGetLastError());
  const dim3 tgrid(static_cast<unsigned>((T + kFirTile - 1) / kFirTile), sum_diff ? B : M);
  if (grad_input) { mrstft_prep_T_kernel<<<tgrid, 256, 0, st>>>(gX, sum_diff, B, C, T, fir_taps, n_taps, 1.f, grad_input); ++g_launches; }
  if (grad_target) { mrstft_prep_T_kernel<<<tgrid, 256, 0, st>>>(gY, sum_diff, B, C, T, fir_taps, n_taps, 1.f, grad_target); ++g_launches; }
  KV_CUDA(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ training step
long long kvae_plan_param_count(const kvae_plan* p) { return p ? p->n_params : fail("null plan"); }

int kvae_plan_param_sizes(const kvae_plan* p, long long* sizes, int max_segments) {
  if (!p || !sizes) return fail("null argument");
  const int n = static_cast<int>(p->param_sizes.size());
  if (max_segments < n) return fail("output array too small");
  for (int i = 0; i < n; ++i) sizes[i] = p->param_sizes[i];
  return n;
}

int kvae_plan_load_params(kvae_plan* p, const float* params, int logscale, int train, void* stream) {
  if (!p || !params) return fail("null argument");
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail("cannot select device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!p->scale_scratch) {
    int m = 1;
    for (const ConvLayer& c : p->convs) m = std::max(m, c.dim0());
    KV_CUDA(cudaMalloc(&p->scale_scratch, static_cast<size_t>(m) * 4));
  }
  bool batched = true;               // one scale + one pack + one SnakeBeta-constant launch for the whole plan
  for (const ConvLayer& c : p->convs) {
    if (c.g.K > kPackMaxK) return fail("kernel size > 16 unsupported by kvae_plan_load_params");
    if (c.umma32) batched = false;   // fp32-mode inference operands need the extra split pass per layer
  }
  if (batched) {
    for (ConvLayer& c : p->convs)
      if (train) {   // the backward pass needs the other index order of each precision
        const size_t n = c.numel();
        if (c.umma && !c.w_umma_d) KV_CUDA(cudaMalloc(&c.w_umma_d, n * 2));
        if (!c.umma && !c.w_direct_d) KV_CUDA(cudaMalloc(&c.w_direct_d, n * 4));
      }
    if (p->fold_train != (train ? 1 : 0)) {
      std::vector<FoldDesc> fd(p->convs.size());
      int rows = 0, tiles = 0;
      for (size_t i = 0; i < p->convs.size(); ++i) {
        const ConvLayer& c = p->convs[i];
        FoldDesc& d = fd[i];
        const int R = c.dim0(), Cc = static_cast<int>(c.numel() / c.g.K / R);
        d.off_v = c.off_v; d.off_g = c.off_g; d.off_bias = c.has_bias ? c.off_bias : -1;
        d.R = R; d.Cc = Cc; d.K = c.g.K; d.Cout = c.g.Cout;
        d.row0 = rows; d.tile0 = tiles; d.tiles_x = ceil_div(R, kPackTR);
        rows += R;
        tiles += d.tiles_x * ceil_div(Cc, kPackTC);
        // index order A = [K][Cout][Cin]: forward tensor-core operand / CUDA-core dgrad operand;
        // index order B = [K][Cin][Cout]: forward CUDA-core operand / tensor-core dgrad operand
        if (c.g.kind == kConv) {   // R = Cout, Cc = Cin: out1 = A, out2 = B
          d.o1b = c.umma ? c.w_umma : nullptr; d.o1f = train ? c.w_direct_d : nullptr;
          d.o2b = train ? c.w_umma_d : nullptr; d.o2f = c.w_direct;
        } else {                   // R = Cin, Cc = Cout: out1 = B, out2 = A
          d.o1b = train ? c.w_umma_d : nullptr; d.o1f = c.w_direct;
          d.o2b = c.umma ? c.w_umma : nullptr; d.o2f = train ? c.w_direct_d : nullptr;
        }
        d.bias = c.bias;
      }
      std::vector<SnakeDesc> sd(p->snakes.size());
      for (size_t i = 0; i < p->snakes.size(); ++i) {
        const SnakeLayer& sl = p->snakes[i];
        sd[i].off_alpha = sl.off_alpha; sd[i].off_beta = sl.off_beta; sd[i].C = sl.C; sd[i].a = sl.a; sd[i].inv_b = sl.inv_b;
      }
      if (!p->fold_desc) KV_CUDA(cudaMalloc(&p->fold_desc, fd.size() * sizeof(FoldDesc)));
      if (!p->snake_desc && !sd.empty()) KV_CUDA(cudaMalloc(&p->snake_desc, sd.size() * sizeof(SnakeDesc)));
      if (!p->scale_all) KV_CUDA(cudaMalloc(&p->scale_all, static_cast<size_t>(rows) * 4));
      // synchronous copies of pageable host vectors: once per plan and mode, not per step.  A (non-blocking) caller
      // stream may still be running kernels that read the previous descriptors: drain it before rewriting them
      KV_CUDA(cudaStreamSynchronize(st));
      KV_CUDA(cudaMemcpy(p->fold_desc, fd.data(), fd.size() * sizeof(FoldDesc), cudaMemcpyHostToDevice));
      if (!sd.empty()) KV_CUDA(cudaMemcpy(p->snake_desc, sd.data(), sd.size() * sizeof(SnakeDesc), cudaMemcpyHostToDevice));
      p->fold_rows = rows; p->fold_tiles = tiles;
      p->fold_train = train ? 1 : 0;
    }
    const int nl = static_cast<int>(p->convs.size());
    weight_norm_scale_all_kernel<<<p->fold_rows, 256, 0, st>>>(params, p->fold_desc, nl, p->scale_all);
    KV_CUDA(cudaGetLastError());
    fold_pack_all_kernel<<<p->fold_tiles, 256, 0, st>>>(params, p->fold_desc, nl, p->scale_all);
    KV_CUDA(cudaGetLastError());
    g_launches += 2;
    if (!p->snakes.empty()) {
      snake_params_all_kernel<<<static_cast<int>(p->snakes.size()), 256, 0, st>>>(params, p->snake_desc, logscale ? 1 : 0);
      KV_CUDA(cudaGetLastError());
      ++g_launches;
    }
    for (ConvLayer& c : p->convs) c.set = true;
    for (SnakeLayer& sl : p->snakes) { sl.logscale = logscale ? 1 : 0; sl.set = true; }
  } else {
  for (ConvLayer& c : p->convs) {
    if (c.g.K > kPackMaxK) return fail("kernel size > 16 unsupported by kvae_plan_load_params");
    const size_t n = c.numel();
    if (train) {   // the backward pass needs the other index order of each precision
      if (c.umma && !c.w_umma_d) KV_CUDA(cudaMalloc(&c.w_umma_d, n * 2));
      if (!c.umma && !c.w_direct_d) KV_CUDA(cudaMalloc(&c.w_direct_d, n * 4));
    }
    const int R = c.dim0(), Cc = static_cast<int>(n / c.g.K / R);
    weight_norm_scale_kernel<<<R, 256, 0, st>>>(params + c.off_v, params + c.off_g, p->scale_scratch, Cc * c.g.K);
    KV_CUDA(cudaGetLastError());
    dim3 grid(ceil_div(R, kPackTR), ceil_div(Cc, kPackTC));
    // index order A = [K][Cout][Cin]: forward tensor-core operand / CUDA-core dgrad operand;
    // index order B = [K][Cin][Cout]: forward CUDA-core operand / tensor-core dgrad operand
    if (c.g.kind == kConv)   // R = Cout, Cc = Cin: out1 = A, out2 = B
      fold_pack_kernel<<<grid, 256, 0, st>>>(params + c.off_v, p->scale_scratch, R, Cc, c.g.K, c.umma ? c.w_umma : nullptr,
                                             train ? c.w_direct_d : nullptr, train ? c.w_umma_d : nullptr, c.w_direct);
    else                     // R = Cin, Cc = Cout: out1 = B, out2 = A
      fold_pack_kernel<<<grid, 256, 0, st>>>(params + c.off_v, p->scale_scratch, R, Cc, c.g.K,
                                             train ? c.w_umma_d : nullptr, c.w_direct, c.umma ? c.w_umma : nullptr,
                                             train ? c.w_direct_d : nullptr);
    KV_CUDA(cudaGetLastError());
    if (c.umma32) {          // fp32-mode inference operand: (hi | lo) halves from the fp32 packing just written
      const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 4096));
      split_pack_kernel<<<blocks, 256, 0, st>>>(c.w_direct, c.g.K, c.g.Cin, c.g.Cout, c.w_umma);
      KV_CUDA(cudaGetLastError());
    }
    if (c.has_bias) KV_CUDA(cudaMemcpyAsync(c.bias, params + c.off_bias, c.g.Cout * 4, cudaMemcpyDeviceToDevice, st));
    c.set = true;
    g_launches += 2;
  }
  for (SnakeLayer& s : p->snakes) {
    snake_params_kernel<<<ceil_div(s.C, 128), 128, 0, st>>>(params + s.off_alpha, params + s.off_beta, logscale, s.C,
                                                           s.a, s.inv_b);
    KV_CUDA(cudaGetLastError());
    s.logscale = logscale ? 1 : 0;
    s.set = true;
    ++g_launches;
  }
  }
  if (train && !p->dwp) {
    size_t off = 0;
    for (ConvLayer& c : p->convs)
      if (c.umma) { c.off_dwp = static_cast<long long>(off); off += c.numel(); }
    p->dwp_floats = off;
    if (off) KV_CUDA(cudaMalloc(&p->dwp, off * 4));
  }
  if (train) p->train_packs = true;
  return 0;
}

size_t kvae_train_workspace_bytes(kvae_plan* p, int B, long long T) {
  if (!p || B <= 0 || T <= 0) { fail("bad argument"); return 0; }
  Layout L;
  std::string err;
  if (!make_layout(p, p->tsteps, true, B, T, L, err)) { fail(err); return 0; }
  size_t max_elems = 0;
  for (const Step& s : p->tsteps)
    max_elems = std::max(max_elems, static_cast<size_t>(B) * static_cast<size_t>(step_len(s, T)) * p->convs[s.conv].g.Cout);
  return align_up(L.total, 1024) + 4 * align_up(max_elems * 4, 1024) + 3 * align_up(max_elems * 2, 1024);
}

int kvae_forward_train(kvae_plan* p, const void* x, int x_dtype, void* y, int y_dtype, int B, long long T, void* ws,
                       size_t ws_bytes, void* stream) {
  if (!p) return fail("null plan");
  if (!x || !y) return fail("null tensor");
  if (!check_dtype(x_dtype) || !check_dtype(y_dtype)) return fail("bad dtype");
  return run_plan(p, true, x, x_dtype, y, y_dtype, B, T, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

int kvae_backward(kvae_plan* p, const void* x, int x_dtype, const void* gy, int gy_dtype, void* gx, int gx_dtype,
                  int B, long long T, void* ws, size_t ws_bytes, float* grads, const float* params, void* stream) {
  if (!check_dtype(x_dtype) || !check_dtype(gy_dtype) || (gx && !check_dtype(gx_dtype))) return fail("bad dtype");
  return run_backward(p, x, x_dtype, gy, gy_dtype, gx, gx_dtype, B, T, ws, ws_bytes, grads, params,
                      static_cast<cudaStream_t>(stream));
}

int kvae_weight_norm_bwd(const float* v, const float* g, const float* dw, float* dv, float* dg, int dim0, int inner,
                         void* stream) {
  if (!v || !g || !dw || !dv || !dg) return fail("null argument");
  if (dim0 <= 0 || inner <= 0) return 0;
  DeviceGuard guard(device_of(v));
  if (!guard.ok) return fail("cannot select the tensor's device");
  weight_norm_bwd_kernel<<<dim0, 256, 0, static_cast<cudaStream_t>(stream)>>>(v, g, dw, dv, dg, inner);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_snake_bwd(const float* x, const float* gy, float* gx, const float* alpha, const float* beta, int logscale,
                   float* d_alpha, float* d_beta, long long rows, int C, void* scratch, void* stream) {
  if (!x || !gy || !gx || !alpha || !beta || !d_alpha || !d_beta || !scratch) return fail("null argument");
  if (rows <= 0 || C <= 0) return 0;
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* a = static_cast<float*>(scratch);
  float* ib = a + C;
  snake_params_kernel<<<ceil_div(C, 128), 128, 0, st>>>(alpha, beta, logscale, C, a, ib);
  KV_CUDA(cudaGetLastError());
  KV_CUDA(cudaMemsetAsync(d_alpha, 0, C * 4, st));
  KV_CUDA(cudaMemsetAsync(d_beta, 0, C * 4, st));
  SnakeBwdParams sb;
  std::memset(&sb, 0, sizeof(sb));
  sb.dA = gy; sb.x = x; sb.a = a; sb.inv_b = ib; sb.logscale = logscale ? 1 : 0;
  sb.G = gx; sb.d_alpha = d_alpha; sb.d_beta = d_beta; sb.rows = rows; sb.C = C;
  dim3 grid;
  set_sb_grid(sb, grid);
  KV_CUDA(launch_snake_bwd(sb, grid, st));
  g_launches += 2;
  return 0;
}

int kvae_vae_sample_bwd(const void* mean, const void* scale, const void* noise, const void* gz, const float* gkl,
                        void* gmean, void* gscale, int B, int D, long long T, int dtype, void* stream) {
  if (!mean || !scale || !noise || !gmean || !gscale) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  const size_t n = static_cast<size_t>(B) * D * T;
  if (n == 0) return 0;
  DeviceGuard guard(device_of(mean));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  vae_sample_bwd_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      mean, scale, noise, gz, gkl, static_cast<float>(1.0 / (static_cast<double>(B) * static_cast<double>(T))), gmean,
      gscale, n, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_gaussian_nll(const void* x, const void* xhat, void* gxhat, float* loss, int B, size_t per_item, float log_sigma,
                      int dtype, void* scratch, void* stream) {
  if (!x || !xhat || !loss || !scratch) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  const size_t n = static_cast<size_t>(B) * per_item;
  if (n == 0) return fail("empty input");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 1024));
  const double inv_var = std::exp(-2.0 * static_cast<double>(log_sigma));
  gaussian_nll_kernel<<<blocks, 256, 0, st>>>(x, xhat, n, dtype == KVAE_F32, static_cast<float>(inv_var),
                                              1.0f / static_cast<float>(B), gxhat, static_cast<double*>(scratch));
  KV_CUDA(cudaGetLastError());
  gaussian_nll_finish_kernel<<<1, 256, 0, st>>>(static_cast<const double*>(scratch), blocks, static_cast<double>(n),
                                                inv_var, static_cast<double>(log_sigma), 1.0 / B, loss);
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  return 0;
}

int kvae_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1,
                    float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq) return fail("null argument");
  if (step < 1) return fail("step counts from 1");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(params));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const float bc1 = 1.f - std::pow(beta1, static_cast<float>(step));
  const float bc2 = 1.f - std::pow(beta2, static_cast<float>(step));
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  adamw_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1,
                                                                       beta2, eps, weight_decay, bc1, std::sqrt(bc2),
                                                                       grad_scale);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

// ------------------------------------------------------------------ PCM tail
int kvae_decode_pcm16(kvae_plan* p, const void* z, int z_dtype, void* wav, int wav_dtype, int16_t* pcm, int B, long long T,
                      void* ws, size_t ws_bytes, void* scratch, void* stream) {
  if (!p) return fail("null plan");
  if (p->direction != KVAE_DECODER) return fail("plan is not a decoder");
  if (!z || !wav || !pcm || !scratch) return fail("null tensor");
  if (!check_dtype(z_dtype) || !check_dtype(wav_dtype)) return fail("bad dtype");
  if (B <= 0 || T <= 0) return fail("empty batch or zero length input");
  if (!(p->precision == KVAE_PREC_BF16 && p->stream_f16 && is_wave_out_step(p, p->steps, static_cast<int>(p->steps.size()) - 1)))
    return fail("fused PCM tail needs the tensor-core tail conv (use kvae_decode + kvae_pcm16)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail("cannot select device");
  KV_CUDA(cudaMemsetAsync(scratch, 0, 4, st));
  FusedSample fs;
  fs.peak = static_cast<unsigned int*>(scratch);
  const int rc = run_plan(p, false, z, z_dtype, wav, wav_dtype, B, T, ws, ws_bytes, st, nullptr, &fs);
  if (rc) return rc;
  const size_t n = static_cast<size_t>(B) * p->arch.io_channels * static_cast<size_t>(T) * p->ratio;
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  pcm16_kernel<<<blocks, 256, 0, st>>>(wav, n, wav_dtype == KVAE_F32, static_cast<const unsigned int*>(scratch), pcm);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_plan_fused_pcm_supported(const kvae_plan* p) {
  if (!p || p->direction != KVAE_DECODER) return 0;
  return (p->precision == KVAE_PREC_BF16 && p->stream_f16 && is_wave_out_step(p, p->steps, static_cast<int>(p->steps.size()) - 1)) ? 1 : 0;
}

int kvae_pcm16(const void* wav, int dtype, int16_t* out, size_t n, void* scratch, void* stream) {
  if (!wav || !out || !scratch) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(wav));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  KV_CUDA(cudaMemsetAsync(scratch, 0, 4, st));
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  absmax_kernel<<<blocks, 256, 0, st>>>(wav, n, dtype == KVAE_F32, static_cast<unsigned int*>(scratch));
  KV_CUDA(cudaGetLastError());
  pcm16_kernel<<<blocks, 256, 0, st>>>(wav, n, dtype == KVAE_F32, static_cast<const unsigned int*>(scratch), out);
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  return 0;
}

// ------------------------------------------------------------------ latent sampling
int kvae_sigma_sample(const void* mean, const void* noise, void* out, size_t n, int dtype, float std,
                      const void* std_noise, float value, size_t per_batch, void* stream) {
  if (!mean || !noise || !out) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (n == 0) return 0;
  if (std_noise && per_batch == 0) return fail("per_batch must be > 0");
  DeviceGuard guard(device_of(mean));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  sigma_sample_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(mean, noise, out, n, dtype == KVAE_F32,
                                                                             std, std_noise, value, per_batch);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

// ------------------------------------------------------------------ BigVGANFlowVAE leaf kernels (bigvgan.cuh)
int kvae_aa_act_fwd(const void* x, void* y, const float* alpha, const float* beta, int logscale, const float* filt_up,
                    const float* filt_down, int B, int C, long long T, int dtype, void* stream) {
  return kvae_aa_act_win_fwd(x, T, 0, T, y, T, 0, T, T, alpha, beta, logscale, filt_up, filt_down, B, C, dtype, stream);
}

// ragged: per-clip ends from lens; otherwise the stream end t_end, kAaNoEnd for none
static int launch_aa_act(bool ragged, const void* x, long long ldx, long long x0, long long nx, void* y, long long ldy, long long o0,
                         long long o1, long long t_end, const float* alpha, const float* beta, int logscale,
                         const float* filt_up, const float* filt_down, int B, int C, int dtype, const RaggedLens& lens,
                         void* stream) {
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  dim3 grid(static_cast<unsigned>((o1 - o0 + kAaTile - 1) / kAaTile), B * C);
  (ragged ? aa_act_kernel<true> : aa_act_kernel<false>)<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, ldx, x0, nx, y, ldy, o0, o1, t_end, alpha, beta, logscale, filt_up, filt_down, C, dtype == KVAE_F32, lens);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_aa_act_win_fwd(const void* x, long long ldx, long long x0, long long nx, void* y, long long ldy, long long o0,
                        long long o1, long long t_end, const float* alpha, const float* beta, int logscale,
                        const float* filt_up, const float* filt_down, int B, int C, int dtype, void* stream) {
  if (!x || !y || !alpha || !filt_up || !filt_down) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || C <= 0 || o1 <= o0) return 0;
  if (static_cast<long long>(B) * C > 65535) return fail("B*C too large");
  const long long te = t_end < 0 ? kAaNoEnd : t_end;
  if (x0 < 0 || nx <= 0 || o0 < 0 || o1 > te || ldx < nx || ldy < o1 - o0)
    return fail("aa_act window: need 0 <= x0, 0 <= o0 < o1 <= t_end, nx <= ldx, o1 - o0 <= ldy");
  if (std::max(0ll, o0 - kAaHalo) < x0 || std::min(o1 + kAaHalo, te) > x0 + nx)
    return fail("aa_act window: the input rows [o0 - 5, o1 + 5) (clipped to the stream) must be inside [x0, x0 + nx)");
  return launch_aa_act(false, x, ldx, x0, nx, y, ldy, o0, o1, te, alpha, beta, logscale, filt_up, filt_down, B, C, dtype,
                       RaggedLens{}, stream);
}

// host valid_len -> RaggedLens, each value in [lo, T]
static int ragged_lens(const int* valid_len, int B, long long T, int lo, RaggedLens* lens) {
  if (!valid_len) return fail("null valid_len");
  if (B > kRaggedMaxClips) return fail("ragged batch: at most 64 clips (kRaggedMaxClips) per call");
  for (int b = 0; b < B; ++b) {
    if (valid_len[b] < lo || valid_len[b] > T) return fail(lo ? "valid_len out of range (1 .. padded length)"
                                                              : "valid_len out of range (0 .. padded length)");
    lens->v[b] = valid_len[b];
  }
  return 0;
}

int kvae_aa_act_ragged_fwd(const void* x, void* y, const float* alpha, const float* beta, int logscale,
                           const float* filt_up, const float* filt_down, int B, int C, long long T,
                           const int* valid_len, int dtype, void* stream) {
  if (!x || !y || !alpha || !filt_up || !filt_down) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || C <= 0 || T <= 0) return 0;
  if (static_cast<long long>(B) * C > 65535) return fail("B*C too large");
  RaggedLens lens;
  if (ragged_lens(valid_len, B, T, 1, &lens)) return -1;
  return launch_aa_act(true, x, T, 0, T, y, T, 0, T, T, alpha, beta, logscale, filt_up, filt_down, B, C, dtype, lens, stream);
}

int kvae_zero_tail_cf(void* y, int B, int C, long long T, long long ldy, const int* valid_len, int dtype, void* stream) {
  if (!y) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || C <= 0 || T <= 0) return 0;
  if (C > 65535) return fail("C too large");
  if (ldy < T) return fail("zero_tail_cf: need T <= ldy");
  RaggedLens lens;
  if (ragged_lens(valid_len, B, T, 0, &lens)) return -1;
  long long tail = 0;
  for (int b = 0; b < B; ++b) tail = std::max(tail, T - lens.v[b]);
  if (tail == 0) return 0;
  DeviceGuard guard(device_of(y));
  if (!guard.ok) return fail("cannot select the tensor's device");
  dim3 grid(static_cast<unsigned>(std::min<long long>((tail + 255) / 256, 64)), C, B);
  zero_tail_cf_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(y, C, T, ldy, lens, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_unary_fwd(const void* x, void* y, size_t n, int op, float param, int dtype, void* stream) {
  if (!x || !y) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (op != 0 && op != 1) return fail("unary op: 0 = leaky_relu, 1 = tanh");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  unary_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, n, op, param, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_axpby(const void* a, const void* b, void* out, size_t n, float alpha, float beta, int dtype, void* stream) {
  if (!a || !b || !out) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(a));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  axpby_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a, b, out, n, alpha, beta, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_gauss_sample(const void* mean, const void* logs, const void* noise, void* out, size_t n, int dtype, void* stream) {
  if (!mean || !logs || !noise || !out) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(mean));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  gauss_sample_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(mean, logs, noise, out, n, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

// ------------------------------------------------------------------ BigVGANFlowVAE leaf backward (bigvgan.cuh)
size_t kvae_aa_act_bwd_scratch_bytes(int B, int C, long long T) {
  if (B <= 0 || C <= 0 || T <= 0) return 0;
  return align_up(static_cast<size_t>(B) * C * ((T + kAaTile - 1) / kAaTile) * 2 * sizeof(double), 1024);
}

int kvae_aa_act_bwd(const void* x, const void* gy, void* gx, const float* alpha, const float* beta, int logscale,
                    const float* filt_up, const float* filt_down, float* dalpha, float* dbeta, int B, int C, long long T,
                    int dtype, void* scratch, size_t scratch_bytes, void* stream) {
  if (!x || !gy || !gx || !alpha || !filt_up || !filt_down || (dalpha && beta && !dbeta)) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || C <= 0 || T <= 0) return fail("empty input");
  if (static_cast<long long>(B) * C > 65535) return fail("B*C too large");
  if (T >= (1LL << 40)) return fail("rows beyond 2^40");
  if (dalpha && (!scratch || scratch_bytes < kvae_aa_act_bwd_scratch_bytes(B, C, T))) return fail("scratch too small");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int tiles = static_cast<int>((T + kAaTile - 1) / kAaTile);
  double* part = dalpha ? static_cast<double*>(scratch) : nullptr;
  aa_act_bwd_kernel<<<dim3(tiles, B * C), 256, 0, st>>>(x, gy, gx, part, T, alpha, beta, logscale, filt_up, filt_down, C,
                                                        dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  if (!dalpha) return 0;
  aa_act_bwd_params_kernel<<<C, 256, 0, st>>>(part, alpha, beta, logscale, dalpha, dbeta, B, C, tiles);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_unary_bwd(const void* t, const void* gy, void* gx, size_t n, int op, float param, int dtype, void* stream) {
  if (!t || !gy || !gx) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (op != 0 && op != 1) return fail("unary op: 0 = leaky_relu, 1 = tanh");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(t));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  unary_bwd_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(t, gy, gx, n, op, param, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_gauss_sample_bwd(const void* x, const void* noise, const void* gz, void* gx, int B, int D, long long T, int dtype,
                          void* stream) {
  if (!x || !noise || !gz || !gx) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || D <= 0 || T <= 0) return 0;
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const size_t n = static_cast<size_t>(B) * D * T;
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 148 * 16));
  gauss_sample_bwd_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, noise, gz, gx, static_cast<long long>(D) * T,
                                                                                 n, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

// ------------------------------------------------------------------ BigVGANFlowVAE flow (flow.cuh)
namespace {
// shared argument checks of the flow kernels: rows = the grid's (b, channel) rows, each of T frames
int flow_launch_check(int B, int rows_per_clip, long long T, int dtype, dim3* grid) {
  if (!check_dtype(dtype)) return fail("bad dtype");
  if (B <= 0 || rows_per_clip <= 0 || T <= 0) return fail("empty input");
  if (static_cast<long long>(B) * rows_per_clip > 65535) return fail("B * channels too large");
  if (T >= (1LL << 40)) return fail("rows beyond 2^40");
  *grid = dim3(static_cast<unsigned>((T + kFlowThreads - 1) / kFlowThreads), static_cast<unsigned>(B * rows_per_clip));
  return 0;
}
}  // namespace

int kvae_flow_split(const void* x, void* xs, void* x0, int B, int C, long long T, int flip, int dtype, void* stream) {
  if (!x || !xs) return fail("null argument");
  if (C % 2) return fail("flow: odd channel count");
  dim3 grid;
  if (flow_launch_check(B, C, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  flow_split_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, xs, x0, C, T, flip, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_flow_split_bwd(const void* gxs, const void* gx0, void* gx, int B, int C, long long T, int flip, int dtype,
                        void* stream) {
  if (!gx) return fail("null argument");
  if (C % 2) return fail("flow: odd channel count");
  dim3 grid;
  if (flow_launch_check(B, C, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(gx));
  if (!guard.ok) return fail("cannot select the tensor's device");
  flow_split_bwd_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(gxs, gx0, gx, C, T, flip,
                                                                                      dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_flow_mask(const void* x, const void* mask, void* y, int B, int C, long long T, int dtype, void* stream) {
  if (!x || !mask || !y) return fail("null argument");
  dim3 grid;
  if (flow_launch_check(B, C, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  flow_mask_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, mask, y, C, T, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_wn_gate_fwd(const void* a, void* acts, int B, int H, long long T, int dtype, void* stream) {
  if (!a || !acts) return fail("null argument");
  dim3 grid;
  if (flow_launch_check(B, H, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(a));
  if (!guard.ok) return fail("cannot select the tensor's device");
  wn_gate_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(a, acts, H, T, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_wn_gate_bwd(const void* a, const void* g, void* ga, int B, int H, long long T, int dtype, void* stream) {
  if (!a || !g || !ga) return fail("null argument");
  dim3 grid;
  if (flow_launch_check(B, H, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(a));
  if (!guard.ok) return fail("cannot select the tensor's device");
  wn_gate_bwd_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(a, g, ga, H, T, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_wn_update_fwd(const void* x, const void* rs, const void* skip, const void* mask, void* x_out, void* skip_out,
                       int B, int H, int last, long long T, int dtype, void* stream) {
  if (!rs || !mask || !skip_out || (!last && (!x || !x_out))) return fail("null argument");
  dim3 grid;
  if (flow_launch_check(B, H, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(rs));
  if (!guard.ok) return fail("cannot select the tensor's device");
  wn_update_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, rs, skip, mask, x_out, skip_out, H,
                                                                                 last ? 1 : 0, T, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_wn_update_bwd(const void* g_xout, const void* g_skipout, const void* mask, void* gx, void* grs, void* gskip,
                       int B, int H, int last, long long T, int dtype, void* stream) {
  if (!mask || !grs || (!last && !gx)) return fail("null argument");
  dim3 grid;
  if (flow_launch_check(B, H, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(grs));
  if (!guard.ok) return fail("cannot select the tensor's device");
  wn_update_bwd_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(g_xout, g_skipout, mask, gx, grs,
                                                                                     gskip, H, last ? 1 : 0, T,
                                                                                     dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_flow_coupling_fwd(const void* x, const void* m, const void* mask, void* y, void* y0, int B, int C, long long T,
                           int flip, int reverse, int dtype, void* stream) {
  if (!x || !m || !mask || !y) return fail("null argument");
  if (C % 2) return fail("flow: odd channel count");
  dim3 grid;
  if (flow_launch_check(B, C / 2, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  flow_coupling_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, m, mask, y, y0, C / 2, T, flip,
                                                                                     reverse, dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_flow_coupling_bwd(const void* gy, const void* gy0, const void* mask, void* gx, void* gm, int B, int C,
                           long long T, int flip, int reverse, int dtype, void* stream) {
  if (!mask || !gx || !gm) return fail("null argument");
  if (C % 2) return fail("flow: odd channel count");
  dim3 grid;
  if (flow_launch_check(B, C / 2, T, dtype, &grid)) return -1;
  DeviceGuard guard(device_of(gx));
  if (!guard.ok) return fail("cannot select the tensor's device");
  flow_coupling_bwd_kernel<<<grid, kFlowThreads, 0, static_cast<cudaStream_t>(stream)>>>(gy, gy0, mask, gx, gm, C / 2, T,
                                                                                         flip, reverse,
                                                                                         dtype == KVAE_F32);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

// ------------------------------------------------------------------ stateful streaming decode
int kvae_decode_stream_begin(kvae_plan* plan, int B, int max_frames, int use_graphs, kvae_stream** out) {
  if (plan && plan->direction != KVAE_DECODER) return fail("streaming: plan is not a decoder");
  return stream_create(plan, B, max_frames, use_graphs, out);
}

void kvae_decode_stream_destroy(kvae_stream* s) {
  if (!s) return;
  DeviceGuard guard(s->plan->device);
  s->cache.clear();
  if (s->cap_stream) cudaStreamDestroy(s->cap_stream);
  cudaFree(s->ws);
  cudaFree(s->z_stage);
  cudaFree(s->wav_stage);
  cudaFree(s->scratch);
  delete s;
}

long long kvae_decode_stream_samples(kvae_stream* s, int n_frames, int end) {
  if (!s) return fail("null stream");
  if (n_frames < 0 || n_frames > s->max_frames) return fail("streaming: n_frames out of range (0 .. max_frames)");
  DeviceGuard guard(s->plan->device);
  PreparedPush* P = stream_get(s, end ? 0 : n_frames, end != 0, KVAE_F32, KVAE_F32);
  return P ? P->n_out : -1;
}

long long kvae_decode_stream_lookahead(const kvae_stream* s) {
  if (!s) return fail("null stream");
  // samples by which the emitted waveform trails the pushed latents in steady state
  long long lag = 0;                       // in rows of the current rate, accumulated front to back
  for (size_t k = 0; k < s->ss.size(); ++k) {
    if (s->ss[k].kind == kRuSecond) continue;
    lag = (lag + s->ss[k].dmax) * s->ss[k].P_out;
  }
  return lag;
}

int kvae_decode_stream_push(kvae_stream* s, const void* z, int z_dtype, int n_frames, void* wav, int wav_dtype,
                            long long wav_capacity, long long* n_samples, void* stream) {
  if (!s) return fail("null stream");
  if (n_frames > 0 && !z) return fail("null latents");
  if (!check_dtype(z_dtype) || !check_dtype(wav_dtype)) return fail("bad dtype");
  if (!wav && wav_capacity > 0) return fail("null wav");
  return stream_run(s, z, z_dtype, n_frames, false, wav, wav_dtype, wav_capacity, n_samples, static_cast<cudaStream_t>(stream));
}

int kvae_decode_stream_end(kvae_stream* s, void* wav, int wav_dtype, long long wav_capacity, long long* n_samples,
                           void* stream) {
  if (!s) return fail("null stream");
  if (!check_dtype(wav_dtype)) return fail("bad dtype");
  return stream_run(s, nullptr, KVAE_F32, 0, true, wav, wav_dtype, wav_capacity, n_samples, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------ stateful streaming encode
int kvae_encode_stream_begin(kvae_plan* plan, int B, long long max_samples, int use_graphs, kvae_stream** out) {
  if (plan && plan->direction != KVAE_ENCODER) return fail("streaming: plan is not an encoder");
  return stream_create(plan, B, max_samples, use_graphs, out);
}

void kvae_encode_stream_destroy(kvae_stream* s) { kvae_decode_stream_destroy(s); }

long long kvae_encode_stream_frames(kvae_stream* s, long long n_samples, int end) {
  if (!s || !s->enc) return fail("null or non-encoder stream");
  if (n_samples < 0 || n_samples > s->max_in) return fail("streaming: n_samples out of range (0 .. max_samples)");
  DeviceGuard guard(s->plan->device);
  PreparedPush* P = stream_get(s, end ? 0 : static_cast<int>(n_samples), end != 0, KVAE_F32, KVAE_F32);
  return P ? P->n_out : -1;
}

long long kvae_encode_stream_lookahead(const kvae_stream* s) {
  if (!s || !s->enc) return fail("null or non-encoder stream");
  // last sample frame t reads is t * ratio + reach, accumulated back to front; the lookahead is what lies beyond
  // the frame's own last sample
  long long reach = 0;
  for (int k = static_cast<int>(s->ss.size()) - 1; k >= 0; --k) {
    if (s->ss[k].kind == kRuSecond) continue;            // the k = 1 half of a fused unit reads its own row
    reach = reach * s->ss[k].P_in + s->ss[k].dmax;
  }
  return reach - (s->ratio - 1);
}

int kvae_encode_stream_push(kvae_stream* s, const void* wav, int wav_dtype, long long n_samples, void* lat, int lat_dtype,
                            long long lat_capacity, long long* n_frames, void* stream) {
  if (!s || !s->enc) return fail("null or non-encoder stream");
  if (n_samples > 0 && !wav) return fail("null wav");
  if (!check_dtype(wav_dtype) || !check_dtype(lat_dtype)) return fail("bad dtype");
  if (!lat && lat_capacity > 0) return fail("null latents");
  if (n_samples < 0 || n_samples > s->max_in) return fail("streaming: n_samples out of range (0 .. max_samples)");
  return stream_run(s, wav, wav_dtype, static_cast<int>(n_samples), false, lat, lat_dtype, lat_capacity, n_frames,
                    static_cast<cudaStream_t>(stream));
}

int kvae_encode_stream_end(kvae_stream* s, void* lat, int lat_dtype, long long lat_capacity, long long* n_frames,
                           void* stream) {
  if (!s || !s->enc) return fail("null or non-encoder stream");
  if (!check_dtype(lat_dtype)) return fail("bad dtype");
  return stream_run(s, nullptr, KVAE_F32, 0, true, lat, lat_dtype, lat_capacity, n_frames, static_cast<cudaStream_t>(stream));
}

int kvae_lm_glue_step(const void* hidden, int hidden_dtype, const float* w1, const float* b1, const float* w2,
                      const float* b2, const float* wa, const float* ba, const void* noise, void* mean, void* latent,
                      void* embed, float* kl_end, int out_dtype, int B, int H, int D, float std, void* stream) {
  if (!hidden || !w1 || !b1 || !w2 || !b2 || !wa || !ba || !noise || !mean || !latent || !embed)
    return fail("null argument");
  if (!check_dtype(hidden_dtype) || !check_dtype(out_dtype)) return fail("bad dtype");
  if (B <= 0) return 0;
  if (H <= 0 || D <= 0 || H % kGlueCluster || D % kGlueCluster) return fail("H and D must be positive multiples of 8");
  if (glue_smem_bytes(H, D) > 200 * 1024) return fail("H / D too large for the glue kernel's shared memory");
  DeviceGuard guard(device_of(hidden));
  if (!guard.ok) return fail("cannot select the tensor's device");
  GlueParams p;
  p.hidden = hidden; p.hidden_f32 = (hidden_dtype == KVAE_F32);
  p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.wa = wa; p.ba = ba;
  p.noise = noise; p.mean = mean; p.latent = latent; p.embed = embed; p.kl_end = kl_end;
  p.out_f32 = (out_dtype == KVAE_F32); p.H = H; p.D = D; p.std = std;
  KV_CUDA(launch_lm_glue_step(p, B, static_cast<cudaStream_t>(stream)));
  ++g_launches;
  return 0;
}

int kvae_vae_sample(const void* mean, const void* scale, const void* noise, void* out, float* kl, int B, int D,
                    long long T, int dtype, void* scratch, void* stream) {
  if (!mean || !scale || !noise || !out || !kl || !scratch) return fail("null argument");
  if (!check_dtype(dtype)) return fail("bad dtype");
  const size_t n = static_cast<size_t>(B) * D * T;
  if (n == 0) return fail("empty input");
  DeviceGuard guard(device_of(mean));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const int blocks = static_cast<int>(std::min<size_t>((n + 255) / 256, 1024));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  vae_sample_kernel<<<blocks, 256, 0, st>>>(mean, scale, noise, out, n, dtype == KVAE_F32,
                                            static_cast<double*>(scratch));
  KV_CUDA(cudaGetLastError());
  kl_finish_kernel<<<1, 256, 0, st>>>(static_cast<const double*>(scratch), blocks,
                                      static_cast<double>(B) * static_cast<double>(T), kl);
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  return 0;
}

// ------------------------------------------------------------------ Oobleck discriminator (disc.cuh)
namespace {
inline int disc_grid(size_t total) {
  return static_cast<int>(std::max<size_t>(1, std::min<size_t>((total + kDiscThreads - 1) / kDiscThreads,
                                                               static_cast<size_t>(sm_count()) * 16)));
}
}  // namespace

int kvae_disc_period_fold(const float* x, float* y, int N, int C, long long T, int n, int backward, void* stream) {
  if (!x || !y) return fail("null argument");
  if (N <= 0 || C <= 0 || T <= 0) return fail("empty input");
  if (n < 1) return fail("disc: the period must be >= 1");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long H = (T + n - 1) / n;
  if (!backward) {
    const size_t total = static_cast<size_t>(N) * C * n * H;
    disc_period_fold_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(x, y, C, T, n, H, total);
  } else {   // x: gradient of the folded tensor [N, C n, H] -> y: gradient of the waveform [N, C, T]
    const size_t total = static_cast<size_t>(N) * C * T;
    disc_period_unfold_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(x, y, T, n, H, total);
  }
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_avg_pool2(const float* x, float* y, long long rows, long long T, int backward, void* stream) {
  if (!x || !y) return fail("null argument");
  if (rows <= 0 || T < 2) return fail("disc: avg_pool1d(2) needs at least two samples");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long To = T / 2;
  if (!backward) {
    const size_t total = static_cast<size_t>(rows) * To;
    if (T % 2 == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0)
      disc_avg_pool2_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(x, y, T, To, total);
    else
      disc_avg_pool2_odd_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(x, y, T, To, total);
  } else {   // x: gradient of the pooled tensor [rows, T / 2] -> y: gradient of the input [rows, T]
    const size_t total = static_cast<size_t>(rows) * T;
    disc_avg_pool2_bwd_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(x, y, T, To, total);
  }
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_folded_width(int W, int K, int stride, int pad) {
  if (W <= 0 || K <= 0 || stride <= 0 || pad < 0 || W + 2 * pad < K) return 0;
  return (W + 2 * pad - K) / stride + 1;
}

int kvae_disc_fold_weight2d(const float* w, const float* bias, float* wf, float* bias_f, int Cout, int Cin, int K, int stride,
                            int pad, int W, int backward, void* stream) {
  if (!w || !wf) return fail("null argument");
  if (Cout <= 0 || Cin <= 0 || K <= 0) return fail("empty weight");
  const int Wo = kvae_disc_folded_width(W, K, stride, pad);
  if (Wo <= 0) return fail("disc: folded width smaller than the kernel");
  DeviceGuard guard(device_of(w));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!backward) {
    const size_t total = static_cast<size_t>(Cout) * Wo * Cin * W * K;
    disc_fold_weight2d_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(w, bias, wf, bias_f, Cout, Cin, K, stride, pad, W, Wo);
  } else {   // wf / bias_f: gradients of the folded tensors (in) -> w / bias: gradients in torch layout (out; const cast)
    const size_t total = static_cast<size_t>(Cout) * Cin * K * K;
    disc_unfold_weight2d_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(wf, bias_f, const_cast<float*>(w),
                                                                         const_cast<float*>(bias), Cout, Cin, K, stride,
                                                                         pad, W, Wo);
  }
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_silu_fwd(const float* f, float* a, size_t n, void* stream) {
  if (!f || !a) return fail("null argument");
  if (n == 0) return 0;
  if ((reinterpret_cast<uintptr_t>(f) | reinterpret_cast<uintptr_t>(a)) & 15) return fail("disc: 16-byte aligned buffers");
  DeviceGuard guard(device_of(f));
  if (!guard.ok) return fail("cannot select the tensor's device");
  disc_silu_kernel<<<disc_grid((n + 3) / 4), kDiscThreads, 0, static_cast<cudaStream_t>(stream)>>>(f, a, n);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_silu_bwd(const float* f, const float* ga, const float* gfeat, float* gf, size_t n, void* stream) {
  if (!f || !ga || !gf) return fail("null argument");
  if (n == 0) return 0;
  DeviceGuard guard(device_of(f));
  if (!guard.ok) return fail("cannot select the tensor's device");
  disc_silu_bwd_kernel<<<disc_grid(n), kDiscThreads, 0, static_cast<cudaStream_t>(stream)>>>(f, ga, gfeat, gf, n);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_score(const float* y, float* score, int N, long long inner, int accumulate, void* stream) {
  if (!y || !score) return fail("null argument");
  if (N <= 0 || inner <= 0) return fail("empty input");
  DeviceGuard guard(device_of(y));
  if (!guard.ok) return fail("cannot select the tensor's device");
  disc_score_kernel<<<N, kDiscThreads, 0, static_cast<cudaStream_t>(stream)>>>(y, score, inner, accumulate);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_score_bwd(const float* gscore, const float* gfeat, float* gy, int N, long long inner, void* stream) {
  if (!gy) return fail("null argument");
  if (N <= 0 || inner <= 0) return fail("empty input");
  DeviceGuard guard(device_of(gy));
  if (!guard.ok) return fail("cannot select the tensor's device");
  const size_t total = static_cast<size_t>(N) * inner;
  disc_score_bwd_kernel<<<disc_grid(total), kDiscThreads, 0, static_cast<cudaStream_t>(stream)>>>(gscore, gfeat, gy, inner, total);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_hinge(const float* score, int B, float* losses, const float* g_losses, float* g_score, void* stream) {
  if (!score) return fail("null argument");
  if (B <= 0) return fail("empty input");
  if (g_losses ? !g_score : !losses) return fail("null argument");
  DeviceGuard guard(device_of(score));
  if (!guard.ok) return fail("cannot select the tensor's device");
  disc_hinge_kernel<<<1, kDiscThreads, 0, static_cast<cudaStream_t>(stream)>>>(score, B, losses, g_losses, g_score);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

size_t kvae_disc_feature_match_scratch_bytes(const long long* half, int n_feats) {
  size_t blocks = 0;
  for (int i = 0; half && i < n_feats; ++i)
    if (half[i] > 0) blocks += static_cast<size_t>((half[i] + kFmChunk - 1) / kFmChunk);
  return align_up(std::max<size_t>(blocks, 1) * 4, 1024);
}

int kvae_disc_feature_match(const float* const* feats, const long long* half, int n_feats, float* loss,
                            const float* g_loss, float* const* grads, void* scratch, size_t scratch_bytes, void* stream) {
  if (!feats || !half || !loss) return fail("null argument");
  if (n_feats <= 0) return fail("disc: no feature tensors");
  const bool backward = g_loss != nullptr;
  if (backward && !grads) return fail("null argument");
  if (!backward && (!scratch || scratch_bytes < kvae_disc_feature_match_scratch_bytes(half, n_feats)))
    return fail("scratch too small");
  for (int i = 0; i < n_feats; ++i) {
    if (!feats[i] || half[i] <= 0) return fail("disc: empty feature tensor");
    if (backward && !grads[i]) return fail("null argument");
  }
  DeviceGuard guard(device_of(feats[0]));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(scratch);
  for (int first = 0; first < n_feats; first += kFmMax) {
    FmTable t;
    std::memset(&t, 0, sizeof(t));
    t.n = std::min(kFmMax, n_feats - first);
    long long blocks = 0;
    for (int k = 0; k < t.n; ++k) {
      t.feat[k] = feats[first + k];
      t.grad[k] = backward ? grads[first + k] : nullptr;
      t.half[k] = half[first + k];
      t.blk_begin[k] = static_cast<int>(blocks);
      blocks += (half[first + k] + kFmChunk - 1) / kFmChunk;
      if (blocks > 0x7fffffffll) return fail("disc: feature tensors too large");
    }
    t.blk_begin[t.n] = static_cast<int>(blocks);
    if (backward) {
      disc_fm_bwd_kernel<<<static_cast<unsigned>(blocks), kDiscThreads, 0, st>>>(t, g_loss);
      KV_CUDA(cudaGetLastError());
      ++g_launches;
    } else {
      disc_fm_partial_kernel<<<static_cast<unsigned>(blocks), kDiscThreads, 0, st>>>(t, partial);
      KV_CUDA(cudaGetLastError());
      disc_fm_finish_kernel<<<1, kDiscThreads, 0, st>>>(partial, static_cast<int>(blocks), loss, first > 0);
      KV_CUDA(cudaGetLastError());
      g_launches += 2;
    }
  }
  return 0;
}

// ---- the discriminator's own conv geometry (k = 15, stride 4, padding 7) on the register-tiled kernels of disc.cuh
int kvae_disc_conv15_supported(int K, int stride, int pad) { return K == kDK && stride == kDS && pad == kDP; }

int kvae_disc_conv15_fwd(const float* x, float* y, const float* w, const float* bias, int N, int Cin, int Cout, long long T,
                         void* scratch, size_t scratch_bytes, void* stream) {
  if (!x || !y || !w || !scratch) return fail("null argument");
  if (N <= 0 || Cin <= 0 || Cout <= 0 || T <= 0) return fail("empty input");
  if (N > 65535 || T > 0x7fffffffll - 64) return fail("disc conv: batch or length too large");
  if (scratch_bytes < kvae_conv1d_scratch_bytes(Cin, Cout, kDK)) return fail("scratch too small");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int To = static_cast<int>((T - 1) / kDS + 1);
  float* wp = static_cast<float*>(scratch);
  const size_t n = static_cast<size_t>(Cin) * Cout * kDK;
  pack_weights_kernel<<<static_cast<int>(std::min<size_t>((n + 255) / 256, 4096)), 256, 0, st>>>(w, 0, Cout, Cin, kDK, nullptr, wp);
  KV_CUDA(cudaGetLastError());
  const long long long_blocks = static_cast<long long>(ceil_div(To, CfGeom<8>::BT)) * ceil_div(Cout, kCfCo) * N;
  if (2 * long_blocks >= sm_count()) {      // (measured: the short tiles only pay when the long ones fill < half the SMs)
    dim3 grid(ceil_div(To, CfGeom<8>::BT), ceil_div(Cout, kCfCo), N);
    KV_CUDA(cudaFuncSetAttribute(disc_conv15_fwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(CfGeom<8>::SMEM)));
    disc_conv15_fwd_kernel<8><<<grid, 256, CfGeom<8>::SMEM, st>>>(x, wp, bias, y, Cin, Cout, static_cast<int>(T), To);
  } else {      // short layer: 32 outputs per block instead of 128, four times the blocks
    dim3 grid(ceil_div(To, CfGeom<2>::BT), ceil_div(Cout, kCfCo), N);
    KV_CUDA(cudaFuncSetAttribute(disc_conv15_fwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(CfGeom<2>::SMEM)));
    disc_conv15_fwd_kernel<2><<<grid, 256, CfGeom<2>::SMEM, st>>>(x, wp, bias, y, Cin, Cout, static_cast<int>(T), To);
  }
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  return 0;
}

int kvae_disc_conv15_bwd(const float* x, const float* gy, const float* w, float* gx, float* dw, float* dbias, int N, int Cin,
                         int Cout, long long T, void* scratch, size_t scratch_bytes, void* stream) {
  if (!x || !gy || !w || !scratch) return fail("null argument");
  if (!dw && !gx && !dbias) return fail("nothing to compute (dw, dbias and gx are all null)");
  if (N <= 0 || Cin <= 0 || Cout <= 0 || T <= 0) return fail("empty input");
  if (N > 65535 || T > 0x7fffffffll - 64) return fail("disc conv: batch or length too large");
  if (scratch_bytes < kvae_conv1d_scratch_bytes(Cin, Cout, kDK)) return fail("scratch too small");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int To = static_cast<int>((T - 1) / kDS + 1);
  const size_t n = static_cast<size_t>(Cin) * Cout * kDK;
  if (dw) {
    KV_CUDA(cudaMemsetAsync(dw, 0, n * 4, st));
    const int tiles = ceil_div(Cout, kWgCo) * ceil_div(Cin, kWgCi);
    const long long items = static_cast<long long>(N) * ceil_div(To, kWgTc);
    const int nsplit = static_cast<int>(std::max<long long>(1, std::min<long long>(std::min<long long>(items, 65535),
                                                                                   (6ll * sm_count() + tiles - 1) / tiles)));
    KV_CUDA(cudaFuncSetAttribute(disc_conv15_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kWgSmem)));
    disc_conv15_wgrad_kernel<<<dim3(tiles, nsplit), 256, kWgSmem, st>>>(x, gy, dw, Cin, Cout, static_cast<int>(T), To,
                                                                        static_cast<int>(items));
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  if (dbias) {
    KV_CUDA(cudaMemsetAsync(dbias, 0, static_cast<size_t>(Cout) * 4, st));
    const int splits = static_cast<int>(std::max<long long>(1, std::min<long long>((2ll * sm_count() + Cout - 1) / Cout,
                                                                                 (static_cast<long long>(N) * To + 4095) / 4096)));
    disc_bias_grad_kernel<<<dim3(Cout, splits), kDiscThreads, 0, st>>>(gy, dbias, N, Cout, To);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  if (!gx) return 0;
  if (Cin < 32 && Cout <= kDsMaxCo) {      // the io-side layer (2 .. 22 folded channels): no channel tile to fill
    dim3 grid(ceil_div(static_cast<int>(T), kDiscThreads), ceil_div(Cin, 4), N);
    disc_conv15_dgrad_small_kernel<<<grid, kDiscThreads, 0, st>>>(gy, w, gx, Cin, Cout, static_cast<int>(T), To);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
    return 0;
  }
  if (Cin < 32) {        // the layer-level data gradient on the CUDA cores: a ConvTranspose1d of stride 4
    DgradGeom d;
    std::string err;
    if (!dgrad_conv_geom(0, Cin, Cout, kDK, kDS, 1, kDP, d, err)) return fail(err);
    return conv1d_dgrad(0, d, gy, To, w, gx, N, T, KVAE_F32, 0, scratch, nullptr, 0, nullptr, st);
  }
  float* wT = static_cast<float*>(scratch);
  pack_weights_kernel<<<static_cast<int>(std::min<size_t>((n + 255) / 256, 4096)), 256, 0, st>>>(w, 1, Cin, Cout, kDK, nullptr, wT);
  KV_CUDA(cudaGetLastError());
  {
    const int Ti = static_cast<int>(T);
    const bool narrow = ceil_div(Cin, 32) * 32 < ceil_div(Cin, 64) * 64;      // a 32-channel tile wastes less (32, 96, ...)
    const int ci_tiles = narrow ? ceil_div(Cin, 32) : ceil_div(Cin, 64);
    const bool shortl = 2ll * ceil_div(Ti + kDP, 256) * ci_tiles * N < sm_count();
#define KVAE_DG_LAUNCH(VQ, CPT)                                                                                           \
    do {                                                                                                                  \
      using G = DgGeom<VQ, CPT>;                                                                                          \
      dim3 grid(ceil_div(Ti + kDP, G::BV), ceil_div(Cin, G::CI), N);                                                      \
      KV_CUDA(cudaFuncSetAttribute(disc_conv15_dgrad_kernel<VQ, CPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                   static_cast<int>(G::SMEM)));                                                           \
      disc_conv15_dgrad_kernel<VQ, CPT><<<grid, 256, G::SMEM, st>>>(gy, wT, gx, Cin, Cout, Ti, To);                        \
    } while (0)
    if (!shortl && !narrow) KVAE_DG_LAUNCH(4, 4);
    else if (!shortl) KVAE_DG_LAUNCH(4, 2);
    else if (!narrow) KVAE_DG_LAUNCH(1, 4);
    else KVAE_DG_LAUNCH(1, 2);
#undef KVAE_DG_LAUNCH
  }
  KV_CUDA(cudaGetLastError());
  g_launches += 2;
  return 0;
}

// ---- the nets' last layer (1 x 1 conv onto <= 8 channels): streaming kernels of disc.cuh
int kvae_disc_conv1x1_supported(int K, int stride, int pad, int Cout) {
  return K == 1 && stride == 1 && pad == 0 && Cout >= 1 && Cout <= kC1MaxCo;
}

int kvae_disc_conv1x1_fwd(const float* x, float* y, const float* w, const float* bias, int N, int Cin, int Cout, long long T,
                          void* stream) {
  if (!x || !y || !w) return fail("null argument");
  if (N <= 0 || Cin <= 0 || T <= 0) return fail("empty input");
  if (Cout < 1 || Cout > kC1MaxCo || N > 65535) return fail("disc 1x1 conv: 1..8 output channels, batch <= 65535");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  dim3 grid(static_cast<unsigned>((T + 31) / 32), N);
  disc_conv1x1_fwd_kernel<<<grid, kDiscThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, w, bias, y, Cin, Cout, T);
  KV_CUDA(cudaGetLastError());
  ++g_launches;
  return 0;
}

int kvae_disc_conv1x1_bwd(const float* x, const float* gy, const float* w, float* gx, float* dw, float* dbias, int N, int Cin,
                          int Cout, long long T, void* stream) {
  if (!x || !gy || !w) return fail("null argument");
  if (!dw && !gx && !dbias) return fail("nothing to compute (dw, dbias and gx are all null)");
  if (N <= 0 || Cin <= 0 || T <= 0) return fail("empty input");
  if (Cout < 1 || Cout > kC1MaxCo || N > 65535 || Cin > 65535) return fail("disc 1x1 conv: 1..8 output channels, batch and channels <= 65535");
  DeviceGuard guard(device_of(x));
  if (!guard.ok) return fail("cannot select the tensor's device");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dw) {
    disc_conv1x1_wgrad_kernel<<<dim3(Cin, Cout), kDiscThreads, 0, st>>>(x, gy, dw, N, Cin, Cout, T);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  if (dbias) {
    bias_grad_cf_kernel<<<Cout, 256, 0, st>>>(gy, 1, dbias, N, Cout, T);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  if (gx) {
    const size_t total = static_cast<size_t>(N) * Cin * T;
    disc_conv1x1_dgrad_kernel<<<disc_grid(total), kDiscThreads, 0, st>>>(gy, w, gx, Cin, Cout, T, total);
    KV_CUDA(cudaGetLastError());
    ++g_launches;
  }
  return 0;
}

}  // extern "C"
