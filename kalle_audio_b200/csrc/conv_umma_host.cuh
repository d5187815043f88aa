// Host side of the tcgen05 convolution: tap tables (how Conv1d / strided Conv1d /
// ConvTranspose1d decompose into (input phase, row shift, weight slab) contributions),
// TMA tensor maps over the channels-last activations and the packed weights, launch.
#pragma once
#include <utility>
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "conv_common.cuh"
#include "conv_umma2.cuh"
#include "conv_ru2.cuh"
#include "wgrad_umma.cuh"

namespace kvae {

enum ConvKind { kConv = 0, kConvT = 1 };

// Geometry of one weight-normalised convolution layer of the Oobleck stack.
struct ConvGeom {
  int kind;      // kConv: nn.Conv1d ; kConvT: nn.ConvTranspose1d
  int Cin, Cout, K, stride, dilation, pad;
  int out_pad = 0;   // ConvTranspose1d output_padding (only the data-gradient geometries use it)
  int out_len(int T_in) const {
    if (kind == kConv) {   // floor division, as torch computes it (the numerator is negative for inputs shorter than the kernel)
      const int num = T_in + 2 * pad - dilation * (K - 1) - 1;
      return (num >= 0 ? num / stride : -((-num + stride - 1) / stride)) + 1;
    }
    return (T_in - 1) * stride - 2 * pad + dilation * (K - 1) + 1 + out_pad;
  }
};

// Geometry of the data gradient of `g` for an input of length T_in: the gradient of a Conv1d w.r.t. its
// input is the ConvTranspose1d with the same weight tensor (and vice versa), so the backward pass reuses
// the forward kernels with the weight re-packed under the opposite kind.
inline ConvGeom dgrad_geom(const ConvGeom& g, int T_in) {
  ConvGeom d = g;
  d.kind = (g.kind == kConv) ? kConvT : kConv;
  d.Cin = g.Cout;
  d.Cout = g.Cin;
  d.out_pad = 0;
  if (d.kind == kConvT) d.out_pad = T_in - d.out_len(g.out_len(T_in));
  return d;
}

inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
inline int posmod(int a, int b) { int r = a % b; return r < 0 ? r + b : r; }

struct TapPlan {
  int P_in = 1;    // input phases (strided Conv1d views x as [T/s, s, C])
  int P_out = 1;   // output phases (ConvTranspose1d stride)
  int span = 0;    // max over slabs of (max shift - min shift)
  int tap_begin[kMaxPhases + 1] = {0};
  std::vector<Tap> taps;
};

inline bool build_taps(const ConvGeom& g, TapPlan& tp, std::string& err) {
  tp = TapPlan();
  struct Raw { int a_phase, delta, w; };
  std::vector<std::vector<Raw>> by_out_phase;
  if (g.kind == kConv) {
    tp.P_in = g.stride;
    tp.P_out = 1;
    if (g.stride > 1 && g.dilation != 1) { err = "strided conv with dilation unsupported"; return false; }
    std::vector<Raw> v;
    for (int k = 0; k < g.K; ++k) {
      const int off = k * g.dilation - g.pad;          // input row = t*stride + off
      v.push_back({posmod(off, g.stride), floordiv(off, g.stride), k});
    }
    by_out_phase.push_back(v);
  } else {
    if (g.dilation != 1 && g.stride != 1) { err = "dilated strided transposed conv unsupported"; return false; }
    tp.P_in = 1;
    tp.P_out = g.stride;
    for (int phi = 0; phi < g.stride; ++phi) {
      std::vector<Raw> v;
      for (int k = 0; k < g.K; ++k)
        if (posmod(phi + g.pad - k * g.dilation, g.stride) == 0)     // t_out = q*s+phi = t_in*s - pad + k*dil
          v.push_back({0, floordiv(phi + g.pad - k * g.dilation, g.stride), k});
      by_out_phase.push_back(v);
    }
  }
  if (tp.P_out > kMaxPhases) { err = "too many output phases"; return false; }
  for (int phi = 0; phi < tp.P_out; ++phi) {
    tp.tap_begin[phi] = static_cast<int>(tp.taps.size());
    auto& v = by_out_phase[phi];
    // group by input phase; a group shares one staged slab
    std::stable_sort(v.begin(), v.end(), [](const Raw& a, const Raw& b) { return a.a_phase < b.a_phase; });
    size_t i = 0;
    while (i < v.size()) {
      size_t j = i;
      int dmin = v[i].delta, dmax = v[i].delta;
      while (j < v.size() && v[j].a_phase == v[i].a_phase) {
        dmin = std::min(dmin, v[j].delta);
        dmax = std::max(dmax, v[j].delta);
        ++j;
      }
      tp.span = std::max(tp.span, dmax - dmin);
      for (size_t t = i; t < j; ++t) {
        Tap tap;
        tap.a_phase = static_cast<int16_t>(v[t].a_phase);
        tap.w_slab = static_cast<int16_t>(v[t].w);
        tap.a_row = static_cast<int16_t>(dmin);
        tap.shift = static_cast<int16_t>(v[t].delta - dmin);
        tap.first = (t == i) ? 1 : 0;
        tap.last = (t + 1 == j) ? 1 : 0;
        tp.taps.push_back(tap);
      }
      i = j;
    }
  }
  tp.tap_begin[tp.P_out] = static_cast<int>(tp.taps.size());
  for (int phi = tp.P_out + 1; phi <= kMaxPhases; ++phi) tp.tap_begin[phi] = tp.tap_begin[tp.P_out];
  if (static_cast<int>(tp.taps.size()) > kMaxTaps) { err = "too many taps"; return false; }
  return true;
}

// ------------------------------------------------------------------ tensor maps
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                        const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_tmapEncodeTiled tmap_encoder() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}

// Activations x: [B, T, C] bf16 viewed as [B, T/P, P, C]; box = {64 ch, 1 phase, RB rows, 1}.
// pitch_rows (0 = T): rows between consecutive clips in memory -- streaming buffers hold more rows than are valid
inline bool make_act_tmap(CUtensorMap* m, const void* x, int B, int T, int C, int P, int RB,
                          std::string& err, long long pitch_rows = 0) {
  auto enc = tmap_encoder();
  if (!enc) { err = "cuTensorMapEncodeTiled unavailable"; return false; }
  if (T % P) { err = "input length not divisible by stride"; return false; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)P, (cuuint64_t)(T / P), (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)P * C * 2, (cuuint64_t)(pitch_rows ? pitch_rows : T) * C * 2};
  cuuint32_t box[4] = {64, 1, (cuuint32_t)RB, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { err = "cuTensorMapEncodeTiled(act) failed: " + std::to_string((int)r); return false; }
  return true;
}

// Packed weights: [nslab, Cout, Cin] bf16; box = {64 ch, NT out-channels, 1 slab}.
inline bool make_w_tmap(CUtensorMap* m, const void* w, int nslab, int Cout, int Cin, int NT,
                        std::string& err) {
  auto enc = tmap_encoder();
  if (!enc) { err = "cuTensorMapEncodeTiled unavailable"; return false; }
  cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)Cout, (cuuint64_t)nslab};
  cuuint64_t strides[2] = {(cuuint64_t)Cin * 2, (cuuint64_t)Cout * Cin * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)NT, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(w), dims, strides, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { err = "cuTensorMapEncodeTiled(w) failed: " + std::to_string((int)r); return false; }
  return true;
}

// Output tensor [B, T, C] viewed as [B, T/P, P, C] for TMA transfers of 32-row x 32-channel blocks:
// fp32 blocks are 128 B wide (SWIZZLE_128B), bf16 blocks 64 B (SWIZZLE_64B).
// dtype: 1 fp32, 0 bf16, 2 fp16 (2-byte types differ only in the tensor map's element type)
inline bool make_out_tmap(CUtensorMap* m, const void* y, int B, int T, int C, int P, int dtype, std::string& err,
                          int box_rows = 32, long long pitch_rows = 0) {
  const bool f32 = (dtype == 1);
  auto enc = tmap_encoder();
  if (!enc) { err = "cuTensorMapEncodeTiled unavailable"; return false; }
  if (T % P) { err = "output length not divisible by stride"; return false; }
  const cuuint64_t es = f32 ? 4 : 2;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)P, (cuuint64_t)(T / P), (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * es, (cuuint64_t)P * C * es, (cuuint64_t)(pitch_rows ? pitch_rows : T) * C * es};
  cuuint32_t box[4] = {32, 1, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                          : (dtype == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16), 4,
                   const_cast<void*>(y), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { err = "cuTensorMapEncodeTiled(out) failed: " + std::to_string((int)r); return false; }
  return true;
}

// ------------------------------------------------------------------ launch
struct ConvEpilogue {
  const float* bias = nullptr;
  const void* residual = nullptr;
  int residual_f32 = 0;
  void* out_raw = nullptr;
  int out_raw_f32 = 0;
  int out_raw_cf = 0;
  __nv_bfloat16* out_act = nullptr;
  const float* snake_a = nullptr;
  const float* snake_inv_b = nullptr;
  int stream_f16 = 0;     // residual and channels-last out_raw are fp16 instead of fp32
  // fp32-mode arithmetic on the tensor cores (see ConvParams2::split3)
  int split3 = 0;         // x is [B, T, 2*Cin] (hi | lo), wpacked is [K][Cout][2*Cin]
  int act_split = 0;      // out_act is [B, T, 2*Cout] (hi | lo)
  int precise = 0;        // sinf instead of MUFU sin in the fused SnakeBeta
  // training backward (ConvParams2::bwd): SnakeBeta derivative of the previous layer + skip-gradient add in the epilogue
  const void* bwd_x = nullptr;        // that layer's saved stream, fp16 channels-last, same shape as this conv's output
  const void* bwd_skip = nullptr;     // bf16 gradient arriving through the skip connection, or nullptr
  const float* bwd_a = nullptr;
  const float* bwd_inv_b = nullptr;
  int bwd_logscale = 1;
};

inline bool umma_supported(const ConvGeom& g) {
  return g.Cin % 64 == 0 && g.Cout % 64 == 0 && g.Cout >= 64;
}

inline int pick_nt(int Cout) {
  if (Cout % 256 == 0) return 256;
  if (Cout % 128 == 0) return 128;
  return 64;
}

// ------------------------------------------------------------------ persistent kernel (conv_umma2.cuh)
struct ConvLaunch2 {
  CUtensorMap tmA, tmW, tmR, tmO, tmX;
  ConvParams2 p;
  int grid = 0;
  size_t smem = 0;
  int T_out = 0;
};

struct ConvTuning2 {
  int MT = 0, NT = 0, acc_stages = 0;   // 0 = auto
  int swap = -1;                        // -1 = auto (swap whenever the tile is 128 out-channels wide)
  int max_ctas = 0;                     // 0 = one per SM
};

inline int sm_count() {
  static int n[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  int& v = n[dev & 63];
  if (!v && (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0)) v = 148;
  return v;
}

// Incremental ("valid") form of a layer for the stateful streaming decoder: the input is a window buffer
// [carry rows | new rows] of in_rows rows, every tap reads at a non-negative offset (row_bias = -min tap offset is
// added to all of them), and exactly out_q output rows per phase are produced -- those whose receptive field lies
// inside the window (or, at the end of the stream, beyond its last row, where TMA's out-of-bounds zero fill is the
// conv's zero padding).  Output / skip pointers are passed already offset to their first row; *_pitch = rows between
// clips in those buffers.  A strided conv (the encoder's downsampling, input viewed as [T/s, s, C]) keeps its phase
// assignment: window row 0 is an absolute input row = 0 (mod s), in_rows and in_pitch are multiples of s and row_bias
// counts groups of s rows.
struct StreamGeom {
  int in_rows = 0, out_q = 0, row_bias = 0;
  long long in_pitch = 0, raw_pitch = 0, act_pitch = 0, res_pitch = 0;
};

// ep.out_raw: fp32 channels-last via TMA unless ep.out_raw_cf (then channels-first direct, any dtype).
// ep.residual must be fp32 channels-last.
inline bool prepare_conv_umma2(const ConvGeom& g, const __nv_bfloat16* x, int B, int T_in,
                               const __nv_bfloat16* wpacked, const ConvEpilogue& ep, const ConvTuning2& tune,
                               ConvLaunch2& L, std::string& err, const StreamGeom* sg = nullptr) {
  if (!umma_supported(g)) { err = "channel counts not multiples of 64"; return false; }
  if (ep.residual && !ep.residual_f32 && !ep.stream_f16) { err = "residual must be fp32 (or the fp16 stream)"; return false; }
  if (ep.out_raw && !ep.out_raw_cf && !ep.out_raw_f32 && !ep.stream_f16) { err = "channels-last raw output must be fp32 (or the fp16 stream)"; return false; }
  TapPlan tp;
  if (!build_taps(g, tp, err)) return false;
  if (sg) {
    if (sg->in_rows % tp.P_in || sg->in_pitch % tp.P_in) { err = "streaming form of a strided conv needs whole phase groups"; return false; }
    T_in = sg->in_rows;
    for (Tap& t : tp.taps) t.a_row = static_cast<int16_t>(t.a_row + sg->row_bias);
  }
  const int T_out = sg ? sg->out_q * tp.P_out : g.out_len(T_in);
  if (T_out <= 0 || T_out % tp.P_out) { err = "bad output length"; return false; }
  ConvParams2& p = L.p;
  std::memset(&p, 0, sizeof(p));
  p.B = B;
  p.P_out = tp.P_out;
  p.Tq_out = T_out / tp.P_out;
  p.Cout = g.Cout;
  p.n_chunks = g.Cin / 64;
  p.raw_mode = ep.out_raw ? (ep.out_raw_cf ? 2 : 1) : 0;
  p.act_mode = ep.out_act ? 1 : 0;
  p.raw_f16 = ep.stream_f16 ? 1 : 0;
  p.split3 = ep.split3 ? 1 : 0;
  p.act_split = (ep.act_split && ep.out_act) ? 1 : 0;
  p.precise = ep.precise ? 1 : 0;
  p.Cin = g.Cin;
  const int sdt = ep.stream_f16 ? 2 : 1;     // element type of the stream tensor maps
  if (ep.bwd_x) {
    if (!ep.out_act || ep.out_raw || ep.residual || ep.split3 || !ep.bwd_a || !ep.bwd_inv_b || g.Cout % 128) {
      err = "fused SnakeBeta backward needs a bf16-only output and 128-channel tiles";
      return false;
    }
    p.bwd = 1;
    p.bwd_skip = ep.bwd_skip ? 1 : 0;
    p.bwd_logscale = ep.bwd_logscale;
    p.bwd_a = ep.bwd_a;
    p.bwd_inv_b = ep.bwd_inv_b;
  }
  // (the 8-warp and 16-warp epilogues stage the same number of bytes per CTA: 16-row instead of 32-row blocks; the fused
  // SnakeBeta backward only runs on the 16-warp one)
  const size_t stage = (p.bwd ? 16 : 8) * static_cast<size_t>(conv_umma2_stage_bytes_per_warp(p.raw_mode, p.act_mode, ep.residual != nullptr,
                                                                                               p.raw_f16, p.act_split, p.bwd));
  const size_t budget = 227 * 1024 - 2048 - stage;
  // candidate tilings, best first: double-buffered accumulators when they fit the 512 TMEM columns
  struct Cand { int MT, NT, acc; };
  std::vector<Cand> cands;
  if (tune.MT || tune.NT || tune.acc_stages) {
    const int NT = tune.NT ? tune.NT : pick_nt(g.Cout);
    const int MT = tune.MT ? tune.MT : 2;
    cands.push_back({MT, NT, tune.acc_stages ? tune.acc_stages : (2 * MT * NT <= 512 ? 2 : 1)});
  } else {
    const int mt = p.Tq_out > 128 ? 2 : 1;
    // tiles the big tiling would give; short sequences (first decoder / last encoder stages, small batches)
    // would leave most of the 148 SMs idle, so they get smaller tiles (more CTAs) instead
    const long long big_tiles = static_cast<long long>(B) * tp.P_out * ((p.Tq_out + 128 * mt - 1) / (128 * mt)) *
                                (g.Cout % 256 == 0 && g.Cout >= 512 ? g.Cout / 256 : (g.Cout + 127) / 128);
    const bool starved = big_tiles * 10 < static_cast<long long>(sm_count()) * 6;
    if (starved && g.Cout % 128 == 0) cands.push_back({1, 128, 2});
    // Cout >= 512: 128-channel swap tiles (N = 256 time rows) with double-buffered accumulators, like the narrower
    // layers.  256 x 256 tiles (the first choice until the end of round 1) fill all 512 TMEM columns
    // with ONE accumulator set, so their epilogue cannot overlap the next tile's MMAs: 63 % tensor-pipe activity at
    // C = 512 (profiles/r01_ncu_summary.txt); the swap tiles read the activation slab twice as often from L2 but
    // measured k7 C=512 0.295 -> 0.254 ms, k1 C=512 0.164 -> 0.121 ms, ConvTranspose 1024->512 0.249 -> 0.197 ms at
    // B = 8 (profiles/r01_tile_shapes_B8.log).  (A 256-wide candidate after the 128-wide one could never be taken: it
    // needs more shared memory for the same slab.)
    if (g.Cout % 128 == 0) cands.push_back({mt, 128, 2});
    if (g.Cout % 128 == 0) cands.push_back({1, 128, 2});
    cands.push_back({mt, 64, 2});
    cands.push_back({1, 64, 2});
  }
  bool ok = false;
  for (const Cand& c : cands) {
    if (g.Cout % c.NT || c.NT % 32 || c.NT > 256 || c.acc * c.MT * c.NT > 512) continue;
    const int rows = 128 * c.MT + tp.span;
    const int nbox = (rows + 255) / 256;
    const int RB = (((rows + nbox - 1) / nbox) + 7) & ~7;
    if (RB > 256) continue;
    const size_t a_bytes = static_cast<size_t>(nbox) * RB * 128, b_bytes = static_cast<size_t>(c.NT) * 128;
    if (2 * a_bytes + 2 * b_bytes > budget) continue;
    p.MT = c.MT; p.NT = c.NT; p.acc_stages = c.acc; p.nbox = nbox; p.RB = RB;
    p.swap = (tune.swap >= 0) ? tune.swap : (c.NT == 128 ? 1 : 0);
    if (p.swap && c.NT != 128) { err = "swap mode needs 128-channel tiles"; return false; }
    p.SA = 2;
    p.SB = static_cast<int>(std::min<size_t>(8, (budget - 2 * a_bytes) / b_bytes));
    while (p.SA < 4 && (p.SA + 1) * a_bytes + p.SB * b_bytes <= budget) ++p.SA;
    {
      // Light-GEMM layers (k = 1, strided and transposed convs: at most two weight stages per activation slab) consume
      // an activation stage every 4-8 MMAs, so with two stages the slab ring covers less than one L2 round trip while
      // the weight ring sits on 4-5 stages it cannot use: give the third slab stage priority over weight stages
      // (k1 C512 0.233 -> 0.190 ms, strided 256 -> 512 0.469 -> 0.394 ms, ConvTranspose 512 -> 256 0.502 -> 0.446 ms
      // at 16 clips; the k = 7 layers keep two slab stages, each serves seven weight stages).
      int n_slabs = 0;
      for (int t = tp.tap_begin[0]; t < tp.tap_begin[1]; ++t) n_slabs += tp.taps[t].first ? 1 : 0;
      const int n_taps = tp.tap_begin[1] - tp.tap_begin[0];
      if (p.SA < 3 && n_taps <= 2 * std::max(1, n_slabs) && 3 * a_bytes + 2 * b_bytes <= budget) {
        p.SA = 3;
        p.SB = static_cast<int>(std::min<size_t>(8, (budget - 3 * a_bytes) / b_bytes));
      }
    }
    ok = true;
    break;
  }
  if (!ok) { err = "no tiling fits shared memory"; return false; }
  // conv_umma2_kernel<1>: forward launches in the swap orientation whose stream / operand blocks are 2-byte
  // (KVAE_FAST_EPI=0 sends them to the generic epilogue of <0>); <2>: every fused SnakeBeta backward
  static const bool fast_on = [] { const char* e = getenv("KVAE_FAST_EPI"); return !(e && e[0] == '0'); }();
  p.fast = (fast_on && p.swap && !p.bwd && !p.act_split && !p.precise && p.raw_mode != 2 &&
            (p.raw_f16 || (p.raw_mode == 0 && !ep.residual))) ? 1 : 0;
  if (p.bwd) p.fast = 2;
  const int box_rows = p.fast ? 16 : 32;
  int cols = 32;
  while (cols < p.acc_stages * p.MT * p.NT) cols <<= 1;
  p.tmem_cols = cols;
  for (int i = 0; i <= kMaxPhases; ++i) p.tap_begin[i] = tp.tap_begin[i];
  for (size_t i = 0; i < tp.taps.size(); ++i) {
    const Tap& t = tp.taps[i];
    if (t.shift * 8 > 0xffff || t.a_phase > 255 || t.w_slab > 255) { err = "tap does not fit the packed table"; return false; }
    p.tap_mma[i] = static_cast<uint32_t>(t.shift * 8) | (t.first ? 0x10000u : 0u) | (t.last ? 0x20000u : 0u);
    p.tap_ld[i] = static_cast<uint32_t>(t.a_phase) | (static_cast<uint32_t>(t.w_slab) << 8) |
                  (static_cast<uint32_t>(static_cast<uint16_t>(t.a_row)) << 16);
  }
  p.q_tiles = (p.Tq_out + 128 * p.MT - 1) / (128 * p.MT);
  p.n_tiles = g.Cout / p.NT;
  p.total_tiles = p.q_tiles * p.n_tiles * tp.P_out * B;
  p.bias = ep.bias;
  p.residual = static_cast<const float*>(ep.residual);
  p.out_cf = (p.raw_mode == 2) ? ep.out_raw : nullptr;
  p.out_cf_f32 = ep.out_raw_f32;
  p.snake_a = ep.snake_a;
  p.snake_inv_b = ep.snake_inv_b;
  const int kmul = p.split3 ? 2 : 1;
  if (!make_act_tmap(&L.tmA, x, B, T_in, g.Cin * kmul, tp.P_in, p.RB, err, sg ? sg->in_pitch : 0)) return false;
  if (!make_w_tmap(&L.tmW, wpacked, g.K, g.Cout, g.Cin * kmul, p.NT, err)) return false;
  if (p.raw_mode == 1) { if (!make_out_tmap(&L.tmR, ep.out_raw, B, T_out, g.Cout, tp.P_out, sdt, err, box_rows, sg ? sg->raw_pitch : 0)) return false; }
  else L.tmR = L.tmA;
  if (p.act_mode == 1) {
    if (!make_out_tmap(&L.tmO, ep.out_act, B, T_out, g.Cout * (p.act_split ? 2 : 1), tp.P_out, false, err, box_rows, sg ? sg->act_pitch : 0)) return false;
  }
  else L.tmO = L.tmA;
  if (ep.residual) { if (!make_out_tmap(&L.tmX, ep.residual, B, T_out, g.Cout, tp.P_out, sdt, err, box_rows, sg ? sg->res_pitch : 0)) return false; }
  else L.tmX = L.tmA;
  if (p.bwd) {
    if (!p.swap) { err = "fused SnakeBeta backward needs the swap orientation"; return false; }
    if (!make_out_tmap(&L.tmX, ep.bwd_x, B, T_out, g.Cout, tp.P_out, 2, err, box_rows)) return false;
    if (ep.bwd_skip && !make_out_tmap(&L.tmR, ep.bwd_skip, B, T_out, g.Cout, tp.P_out, 0, err, box_rows)) return false;
  }
  const int ctas = tune.max_ctas ? tune.max_ctas : sm_count();
  L.grid = std::min(p.total_tiles, ctas);
  L.smem = conv_umma2_smem_bytes(p);
  L.T_out = T_out;
  return true;
}

// Launch with programmatic stream serialization (ptx.cuh, pdl_*): the kernel may begin while its predecessor drains.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

inline cudaError_t launch_conv_umma2(const ConvLaunch2& L, cudaStream_t stream) {
  static bool attr_set[64] = {false};   // per device (the attribute is per device context)
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(conv_umma2_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_umma2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_umma2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set[dev & 63] = true;
  }
  if (L.p.fast == 2)
    return launch_pdl(conv_umma2_kernel<2>, dim3(L.grid), dim3(640), L.smem, stream, L.tmA, L.tmW, L.tmR, L.tmO, L.tmX, L.p);
  if (L.p.fast)
    return launch_pdl(conv_umma2_kernel<1>, dim3(L.grid), dim3(640), L.smem, stream, L.tmA, L.tmW, L.tmR, L.tmO, L.tmX, L.p);
  return launch_pdl(conv_umma2_kernel<0>, dim3(L.grid), dim3(384), L.smem, stream, L.tmA, L.tmW, L.tmR, L.tmO, L.tmX, L.p);
}

// ------------------------------------------------------------------ fused ResidualUnit (conv_ru2.cuh)
struct RuLaunch {
  CUtensorMap tmA, tmW7, tmW1, tmR, tmO, tmX;
  RuParams p;
  int grid = 0;
  size_t smem = 0;
};

struct RuArgs {
  const __nv_bfloat16* a = nullptr;       // SnakeBeta1(x), bf16 [B, T, 128]
  const void* x = nullptr;                // residual stream, fp32 (or fp16: stream_f16) [B, T, 128]
  const __nv_bfloat16* w7 = nullptr;      // packed [7][128][128]
  const __nv_bfloat16* w1 = nullptr;      // packed [1][128][128]
  const float* bias7 = nullptr;
  const float* s2_a = nullptr;
  const float* s2_inv_b = nullptr;
  const float* bias1 = nullptr;
  void* out_raw = nullptr;                // stream out, same type as x, [B, T, 128] or nullptr
  __nv_bfloat16* out_act = nullptr;       // bf16 [B, T, 128] or nullptr
  const float* sn_a = nullptr;
  const float* sn_inv_b = nullptr;
  int stream_f16 = 0;                     // x and out_raw are fp16 instead of fp32
  int act_f16 = 0;                        // out_act is fp16 (SnakeBeta applied) for the decoder tail's kind::f16 GEMM
};

inline bool ru_supported(int C) { return C == kRuC; }

// sg (streaming form): T = sg->out_q output rows from a window of sg->in_rows rows; a.x is the skip pointer already
// offset by the unit's lag (3 * dilation rows into the window), out pointers offset to their first row
inline bool prepare_conv_ru(const RuArgs& a, int B, int T, int dilation, RuLaunch& L, std::string& err,
                            const StreamGeom* sg = nullptr) {
  if (!a.a || !a.x || !a.w7 || !a.w1 || !a.bias7 || !a.bias1 || !a.s2_a || !a.s2_inv_b) { err = "fused RU: null argument"; return false; }
  if (!a.out_raw && !a.out_act) { err = "fused RU: no output"; return false; }
  RuParams& p = L.p;
  std::memset(&p, 0, sizeof(p));
  if (sg) T = sg->out_q;
  p.B = B;
  p.T = T;
  const int rows = 256 + 6 * dilation;
  p.nbox = (rows + 255) / 256;
  p.RB = (((rows + p.nbox - 1) / p.nbox) + 7) & ~7;
  if (p.RB > 256) { err = "fused RU: dilation too large"; return false; }
  p.slab_row0 = sg ? -3 * dilation + sg->row_bias : -3 * dilation;
  for (int t = 0; t < 7; ++t) p.tap_shift16[t] = static_cast<uint32_t>(t * dilation * 8);
  p.raw_out = a.out_raw ? 1 : 0;
  p.act_out = a.out_act ? 1 : 0;
  const size_t a_bytes = static_cast<size_t>(p.nbox) * p.RB * 128, b_bytes = kRuC * 128;
  if (!a.stream_f16) { err = "fused RU: needs the fp16 residual stream"; return false; }
  const int sdt = 2;
  const size_t budget = 227 * 1024 - 2048 - kRuHBytes - kRuEpiWarps * static_cast<size_t>(ru_stage_bytes_per_warp(p.act_out));
  p.SA = 2;
  if (2 * a_bytes + 3 * b_bytes > budget) { err = "fused RU does not fit shared memory"; return false; }
  p.SB = static_cast<int>(std::min<size_t>(8, (budget - 2 * a_bytes) / b_bytes));
  p.q_tiles = (T + 255) / 256;
  p.total_tiles = p.q_tiles * B;
  p.bias7 = a.bias7; p.s2_a = a.s2_a; p.s2_inv_b = a.s2_inv_b; p.bias1 = a.bias1;
  p.sn_a = a.sn_a; p.sn_inv_b = a.sn_inv_b;
  p.act_f16 = a.act_f16;
  if (!make_act_tmap(&L.tmA, a.a, B, sg ? sg->in_rows : T, kRuC, 1, p.RB, err, sg ? sg->in_pitch : 0)) return false;
  if (!make_w_tmap(&L.tmW7, a.w7, 7, kRuC, kRuC, kRuC, err)) return false;
  if (!make_w_tmap(&L.tmW1, a.w1, 1, kRuC, kRuC, kRuC, err)) return false;
  if (!make_out_tmap(&L.tmX, a.x, B, T, kRuC, 1, sdt, err, 16, sg ? sg->res_pitch : 0)) return false;
  if (a.out_raw) { if (!make_out_tmap(&L.tmR, a.out_raw, B, T, kRuC, 1, sdt, err, 16, sg ? sg->raw_pitch : 0)) return false; } else L.tmR = L.tmX;
  if (a.out_act) { if (!make_out_tmap(&L.tmO, a.out_act, B, T, kRuC, 1, false, err, 16, sg ? sg->act_pitch : 0)) return false; } else L.tmO = L.tmX;
  L.grid = std::min(p.total_tiles, sm_count());
  if (const char* e = getenv("KVAE_RU_GRID")) L.grid = std::max(1, std::min(L.grid, atoi(e)));   // tests: many tiles per CTA
  L.smem = ru_smem_bytes(p);
  return true;
}

inline cudaError_t launch_conv_ru(const RuLaunch& L, cudaStream_t stream) {
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(conv_ru2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set[dev & 63] = true;
  }
  return launch_pdl(conv_ru2_kernel, dim3(L.grid), dim3(kRuThreads), L.smem, stream, L.tmA, L.tmW7, L.tmW1, L.tmR, L.tmO, L.tmX, L.p);
}

// ------------------------------------------------------------------ tensor-core weight gradient (wgrad_umma.cuh)
struct WgradLaunch {
  CUtensorMap tmD, tmS;
  WgradUmmaParams p;
  dim3 grid;
  size_t smem = 0;
};

// dense [B, Td, Cd] and strided [B, Ts, Cs] are bf16 channels-last; dWp is the packed [K][Cd][Cs] fp32 accumulator.
// (stride, dil, pad) are the FORWARD convolution's: the strided tensor is read at t*stride + k*dil - pad.
inline bool prepare_wgrad_umma(const __nv_bfloat16* dense, int Td, int Cd, const __nv_bfloat16* strided, int Ts, int Cs,
                               int B, int K, int stride, int dil, int pad, float* dWp, WgradLaunch& L, std::string& err) {
  if (Cd % 64 || Cs % 64) { err = "wgrad: channel counts not multiples of 64"; return false; }
  if (stride > 1 && dil != 1) { err = "wgrad: strided conv with dilation unsupported"; return false; }
  if (Ts % stride) { err = "wgrad: strided length not divisible by stride"; return false; }
  if (K > kWgMaxTaps * kWgMaxGroups) { err = "wgrad: too many taps"; return false; }
  WgradUmmaParams& p = L.p;
  std::memset(&p, 0, sizeof(p));
  struct T3 { int phase, delta, k; };
  std::vector<T3> taps;
  for (int k = 0; k < K; ++k) {
    const int off = k * dil - pad;
    taps.push_back({posmod(off, stride), floordiv(off, stride), k});
  }
  std::stable_sort(taps.begin(), taps.end(), [](const T3& a, const T3& b) {
    return a.phase != b.phase ? a.phase < b.phase : a.delta < b.delta;
  });
  p.n_groups = (K + kWgMaxTaps - 1) / kWgMaxTaps;
  int span = 0, max_slabs = 1;
  for (int g = 0; g < p.n_groups; ++g) {
    const int lo = g * kWgMaxTaps, hi = std::min(K, lo + kWgMaxTaps);
    p.g_ntaps[g] = hi - lo;
    int nslabs = 0;
    for (int t = lo; t < hi; ++t) {
      int slab = -1;
      for (int s2 = 0; s2 < nslabs; ++s2)
        if (p.s_phase[g][s2] == taps[t].phase) slab = s2;
      if (slab < 0) {          // taps are sorted by (phase, delta): the first tap of a phase has its smallest delta
        slab = nslabs++;
        p.s_phase[g][slab] = taps[t].phase;
        p.s_row0[g][slab] = taps[t].delta;
      }
      p.g_k[g][t - lo] = taps[t].k;
      p.g_slab[g][t - lo] = slab;
      p.g_shift[g][t - lo] = taps[t].delta - p.s_row0[g][slab];
      span = std::max(span, p.g_shift[g][t - lo]);
    }
    p.g_nslabs[g] = nslabs;
    max_slabs = std::max(max_slabs, nslabs);
  }
  const size_t budget = 227 * 1024 - 2048;
  bool ok = false;
  for (int R : {128, 64, 32, 16}) {
    const int RS = (R + span + 7) & ~7;
    if (RS > 256) continue;
    const size_t stage = wgrad_umma_stage_bytes(R, RS, max_slabs);
    const int NS = static_cast<int>(std::min<size_t>(4, budget / stage));
    if (NS < 2) continue;
    if (NS < 3 && R > 32) continue;       // prefer a deeper pipeline over a taller stage
    p.R = R; p.RS = RS; p.NS = NS;
    ok = true;
    break;
  }
  if (!ok) {
    for (int R : {64, 32, 16}) {
      const int RS = (R + span + 7) & ~7;
      if (RS > 256) continue;
      const size_t stage = wgrad_umma_stage_bytes(R, RS, max_slabs);
      if (budget / stage < 2) continue;
      p.R = R; p.RS = RS; p.NS = 2;
      ok = true;
      break;
    }
  }
  if (!ok) { err = "wgrad: tile does not fit shared memory"; return false; }
  p.B = B; p.Td = Td; p.Cd = Cd; p.Cs = Cs; p.K = K;
  p.chunks_per_clip = (Td + p.R - 1) / p.R;
  p.n_cd = (Cd + 127) / 128;
  p.n_cs = (Cs + 127) / 128;
  const long long combos = static_cast<long long>(p.n_groups) * p.n_cd * p.n_cs;
  const long long items = static_cast<long long>(B) * p.chunks_per_clip;
  long long nsplit = std::max<long long>(1, (3ll * sm_count() + combos - 1) / combos);
  nsplit = std::min(nsplit, items);
  long long ips = (items + nsplit - 1) / nsplit;
  nsplit = (items + ips - 1) / ips;
  if (nsplit > 65535) { err = "wgrad: too many splits"; return false; }
  p.items_per_split = static_cast<int>(ips);
  p.dWp = dWp;
  if (!make_act_tmap(&L.tmD, dense, B, Td, Cd, 1, p.R, err)) return false;
  if (!make_act_tmap(&L.tmS, strided, B, Ts, Cs, stride, p.RS, err)) return false;
  L.grid = dim3(static_cast<unsigned>(combos), static_cast<unsigned>(nsplit));
  L.smem = 1024 + 1024 + static_cast<size_t>(p.NS) * wgrad_umma_stage_bytes(p.R, p.RS, max_slabs);
  return true;
}

inline cudaError_t launch_wgrad_umma(const WgradLaunch& L, cudaStream_t stream) {
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!attr_set[dev & 63]) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    attr_set[dev & 63] = true;
  }
  wgrad_umma_kernel<<<L.grid, 256, L.smem, stream>>>(L.tmD, L.tmS, L.p);
  return cudaGetLastError();
}

}  // namespace kvae
