// HBM-bound helper kernels: SnakeBeta on the API layout, layout changes at the model boundary,
// weight-norm folding and weight packing at load time, and the latent sampling steps.
#pragma once
#include <cuda_bf16.h>
#include <cstdint>

#include "conv_common.cuh"  // snake_beta

namespace kvae {

__device__ __forceinline__ float ld_elem(const void* p, size_t i, int f32) {
  return f32 ? static_cast<const float*>(p)[i] : __bfloat162float(static_cast<const __nv_bfloat16*>(p)[i]);
}
__device__ __forceinline__ void st_elem(void* p, size_t i, int f32, float v) {
  if (f32) static_cast<float*>(p)[i] = v;
  else static_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16(v);
}

// ---------------------------------------------------------------- SnakeBeta, [B, C, T] layout
// reference blocks.py:301-339: alpha' = exp(alpha), beta' = exp(beta) when logscale;
// y = x + 1/(beta' + 1e-9) * sin(x*alpha')^2.   grid: (ceil(T/ (256*4)), B*C)
__global__ void snake_cf_kernel(const void* x, void* y, const float* alpha, const float* beta,
                                int logscale, int C, long long T, int f32) {
  const int c = blockIdx.y % C;
  float a = alpha[c], bt = beta[c];
  if (logscale) { a = expf(a); bt = expf(bt); }
  const float inv_b = 1.0f / (bt + 1e-9f);
  const size_t row = static_cast<size_t>(blockIdx.y) * T;
  const long long t0 = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long t = t0 + i;
    if (t < T) {
      const float v = ld_elem(x, row + t, f32);
      const float s = sinf(v * a);
      st_elem(y, row + t, f32, v + inv_b * (s * s));
    }
  }
}

// a = exp(alpha) (or alpha), inv_b = 1/(exp(beta)+1e-9): per-channel constants used by the fused
// prologues/epilogues.
__global__ void snake_params_kernel(const float* alpha, const float* beta, int logscale, int C, float* a,
                                    float* inv_b) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    float av = alpha[c], bv = beta[c];
    if (logscale) { av = expf(av); bv = expf(bv); }
    a[c] = av;
    inv_b[c] = 1.0f / (bv + 1e-9f);
  }
}

// ---------------------------------------------------------------- [B, C, T] -> [B, T, C] bf16
// 32x32 shared-memory tile transpose.  grid: (ceil(T/32), ceil(C/32), B), block (32, 8)
// split = 1: y is [B, T, 2C] with the bf16 (hi | lo) halves of the fp32 value (fp32-mode tensor-core operand)
// y_pitch (0 = T): rows between clips in y (the streaming decoder writes into a window buffer)
// [x_lo, x_hi) (x_hi < 0: T): the rows read from x; the other rows of y are written as zeros (the zero rows of a
// strided window rounded up to whole stride groups, and rows past the stream end)
__global__ void cf_to_cl_bf16_kernel(const void* x, int f32, __nv_bfloat16* y, int C, int T, int split,
                                     long long y_pitch = 0, long long x_pitch = 0, int x_lo = 0, int x_hi = -1) {
  const long long YP = y_pitch ? y_pitch : T;
  const long long XP = x_pitch ? x_pitch : T;          // elements between channel rows of x
  const int t_hi = x_hi < 0 ? T : x_hi;
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, t = t0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && t >= x_lo && t < t_hi) ? ld_elem(x, (static_cast<size_t>(b) * C + c) * XP + t, f32) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int t = t0 + i, c = c0 + threadIdx.x;
    if (c < C && t < T) {
      const float v = tile[threadIdx.x][i];
      const __nv_bfloat16 hi = __float2bfloat16(v);
      if (split) {
        y[(static_cast<size_t>(b) * YP + t) * 2 * C + c] = hi;
        y[(static_cast<size_t>(b) * YP + t) * 2 * C + C + c] = __float2bfloat16(v - __bfloat162float(hi));
      } else {
        y[(static_cast<size_t>(b) * YP + t) * C + c] = hi;
      }
    }
  }
}

// fp32-mode tensor-core weights: w_direct [K][Cin][Cout] fp32 -> [K][Cout][2*Cin] bf16, (hi | lo) halves per row
__global__ void split_pack_kernel(const float* w_direct, int K, int Cin, int Cout, __nv_bfloat16* w_split) {
  const size_t n = static_cast<size_t>(K) * Cin * Cout;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ci = static_cast<int>(i % Cin);
    const size_t r = i / Cin;                       // k*Cout + co
    const int co = static_cast<int>(r % Cout), k = static_cast<int>(r / Cout);
    const float v = w_direct[(static_cast<size_t>(k) * Cin + ci) * Cout + co];
    const __nv_bfloat16 hi = __float2bfloat16(v);
    w_split[r * 2 * Cin + ci] = hi;
    w_split[r * 2 * Cin + Cin + ci] = __float2bfloat16(v - __bfloat162float(hi));
  }
}

// ---------------------------------------------------------------- weight norm fold
// w[i, :] = v[i, :] * (g[i] / ||v[i, :]||_2)   (old-style torch weight_norm, dim=0).  One block per i.
__global__ void weight_norm_fold_kernel(const float* v, const float* g, float* w, int inner) {
  __shared__ float red[32];
  const size_t base = static_cast<size_t>(blockIdx.x) * inner;
  float s = 0.f;
  for (int i = threadIdx.x; i < inner; i += blockDim.x) { const float x = v[base + i]; s = fmaf(x, x, s); }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  const float scale = g[blockIdx.x] / sqrtf(red[0]);
  for (int i = threadIdx.x; i < inner; i += blockDim.x) w[base + i] = v[base + i] * scale;
}

// ---------------------------------------------------------------- weight packing
// torch Conv1d weight [Cout][Cin][K] (transposed=0) or ConvTranspose1d weight [Cin][Cout][K]
// (transposed=1) -> tensor-core operand [K][Cout][Cin] bf16 and CUDA-core operand [K][Cin][Cout] fp32.
// kFlipTaps: tap k of w lands at K - 1 - k (the data gradient of a Conv1d, kvae_conv1d_win_bwd).
template <bool kFlipTaps = false>
__global__ void pack_weights_kernel(const float* w, int transposed, int Cout, int Cin, int K,
                                    __nv_bfloat16* w_umma, float* w_direct) {
  const size_t n = static_cast<size_t>(Cout) * Cin * K;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int k = kFlipTaps ? K - 1 - static_cast<int>(i % K) : static_cast<int>(i % K);
    const size_t r = i / K;
    int co, ci;
    if (transposed) { co = static_cast<int>(r % Cout); ci = static_cast<int>(r / Cout); }
    else { ci = static_cast<int>(r % Cin); co = static_cast<int>(r / Cin); }
    const float v = w[i];
    if (w_umma) w_umma[(static_cast<size_t>(k) * Cout + co) * Cin + ci] = __float2bfloat16(v);
    if (w_direct) w_direct[(static_cast<size_t>(k) * Cin + ci) * Cout + co] = v;
  }
}

// ---------------------------------------------------------------- fold + pack from a flat parameter buffer
// scale[i] = g[i] / ||v[i, :]||  (one block per dim-0 row); the tiled kernel below applies it while packing.
__global__ void weight_norm_scale_kernel(const float* v, const float* g, float* scale, int inner) {
  __shared__ float red[32];
  const size_t base = static_cast<size_t>(blockIdx.x) * inner;
  float s = 0.f;
  for (int i = threadIdx.x; i < inner; i += blockDim.x) { const float x = v[base + i]; s = fmaf(x, x, s); }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) scale[blockIdx.x] = g[blockIdx.x] / sqrtf(t);
  }
}

// v [R][Cc][K] fp32 (torch layout: Conv1d R = Cout, Cc = Cin; ConvTranspose1d R = Cin, Cc = Cout), scaled per
// row, written in both index orders and both precisions through a shared-memory tile so that reads and
// writes are coalesced:  out1[(k*R + r)*Cc + c]   and   out2[(k*Cc + c)*R + r].
// grid (ceil(R/16), ceil(Cc/32)), block 256, K <= 16.
constexpr int kPackTR = 16, kPackTC = 32, kPackMaxK = 16;
__device__ __forceinline__ void fold_pack_tile(float (*tile)[kPackTC * (kPackMaxK + 1)], const float* v, const float* scale,
                                               int R, int Cc, int K, int bx, int by, __nv_bfloat16* out1_bf16,
                                               float* out1_f32, __nv_bfloat16* out2_bf16, float* out2_f32) {
  // Second form (round 2): no division per element (a per-block table maps the row-contiguous index j = c K + k to
  // its tile slot) and two elements per store (bf16x2 / float2) in both output orders.  The first form spent three
  // runtime div/mod pairs per element and wrote 2-byte elements: 0.98 ms per optimizer step for 156 M weights, five
  // times its HBM floor.
  __shared__ uint16_t slot[kPackTC * kPackMaxK];
  const int r0 = bx * kPackTR, c0 = by * kPackTC;
  const int w = kPackTC * K;                 // contiguous floats per row of the tile
  const int Kp = K | 1;                      // odd per-column stride in shared memory: the transposed reads below
                                             // walk columns, which would be a K-way bank conflict for even K
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = threadIdx.x; j < w; j += 256) {
    const int c = j / K;
    slot[j] = static_cast<uint16_t>(c * Kp + (j - c * K));
  }
  __syncthreads();
  const int cmax = min(kPackTC, Cc - c0);    // valid columns of this tile
  for (int r = warp; r < kPackTR; r += 8) {
    const bool rv = r0 + r < R;
    const float sc = rv ? scale[r0 + r] : 0.f;
    const float* src = v + (static_cast<size_t>(r0 + r) * Cc + c0) * K;
    for (int j = lane; j < w; j += 32) tile[r][slot[j]] = (rv && j < cmax * K) ? src[j] * sc : 0.f;
  }
  __syncthreads();
  // out1[(k R + r) Cc + c]: c fastest; 16 lanes x 2 columns cover a (k, r) row of the tile, a warp two of them
  const bool pair1 = (Cc & 1) == 0;
  for (int pr = warp * 2 + (lane >> 4); pr < K * kPackTR; pr += 16) {
    const int k = pr / kPackTR, r = pr % kPackTR;          // kPackTR = 16: shifts
    const int c = 2 * (lane & 15);
    if (r0 + r >= R || c >= cmax) continue;
    const float a = tile[r][c * Kp + k], b = (c + 1 < cmax) ? tile[r][(c + 1) * Kp + k] : 0.f;
    const size_t o = (static_cast<size_t>(k) * R + r0 + r) * Cc + c0 + c;
    if (pair1 && c + 1 < cmax) {
      if (out1_bf16) *reinterpret_cast<__nv_bfloat162*>(out1_bf16 + o) = __floats2bfloat162_rn(a, b);
      if (out1_f32) *reinterpret_cast<float2*>(out1_f32 + o) = make_float2(a, b);
    } else {
      if (out1_bf16) { out1_bf16[o] = __float2bfloat16(a); if (c + 1 < cmax) out1_bf16[o + 1] = __float2bfloat16(b); }
      if (out1_f32) { out1_f32[o] = a; if (c + 1 < cmax) out1_f32[o + 1] = b; }
    }
  }
  // out2[(k Cc + c) R + r]: r fastest; 8 lanes x 2 rows cover a (k, c) column of the tile, a warp four of them
  const bool pair2 = (R & 1) == 0;
  const int rmax = min(kPackTR, R - r0);
  for (int pc = warp * 4 + (lane >> 3); pc < K * kPackTC; pc += 32) {
    const int k = pc / kPackTC, c = pc % kPackTC;          // kPackTC = 32: shifts
    const int r = 2 * (lane & 7);
    if (c >= cmax || r >= rmax) continue;
    const float a = tile[r][c * Kp + k], b = (r + 1 < rmax) ? tile[r + 1][c * Kp + k] : 0.f;
    const size_t o = (static_cast<size_t>(k) * Cc + c0 + c) * R + r0 + r;
    if (pair2 && r + 1 < rmax) {
      if (out2_bf16) *reinterpret_cast<__nv_bfloat162*>(out2_bf16 + o) = __floats2bfloat162_rn(a, b);
      if (out2_f32) *reinterpret_cast<float2*>(out2_f32 + o) = make_float2(a, b);
    } else {
      if (out2_bf16) { out2_bf16[o] = __float2bfloat16(a); if (r + 1 < rmax) out2_bf16[o + 1] = __float2bfloat16(b); }
      if (out2_f32) { out2_f32[o] = a; if (r + 1 < rmax) out2_f32[o + 1] = b; }
    }
  }
}

__global__ void __launch_bounds__(256)
fold_pack_kernel(const float* v, const float* scale, int R, int Cc, int K, __nv_bfloat16* out1_bf16, float* out1_f32,
                 __nv_bfloat16* out2_bf16, float* out2_f32) {
  __shared__ float tile[kPackTR][kPackTC * (kPackMaxK + 1)];
  fold_pack_tile(tile, v, scale, R, Cc, K, blockIdx.x, blockIdx.y, out1_bf16, out1_f32, out2_bf16, out2_f32);
}

// ---------------------------------------------------------------- the same for ALL layers of a plan in two launches
// One optimizer step re-folds ~75 weight tensors; as one scale + one pack launch per layer (plus a bias copy and a
// SnakeBeta-constant launch per activation) that is ~300 stream operations of a few microseconds of work each --
// 2.9 ms of a 35 ms training step (profiles/r01_train_step_launches.txt).  Here a block finds its layer by binary
// search in a prefix table.
struct FoldDesc {
  long long off_v, off_g, off_bias;   // floats into the flat parameter buffer; off_bias < 0: no bias
  int R, Cc, K, Cout;
  int row0;                           // first block of the layer in weight_norm_scale_all_kernel = offset into scale[]
  int tile0, tiles_x;                 // first block in fold_pack_all_kernel, tiles along R
  __nv_bfloat16* o1b; float* o1f; __nv_bfloat16* o2b; float* o2f;
  float* bias;
};
struct SnakeDesc { long long off_alpha, off_beta; int C; float* a; float* inv_b; };

__device__ __forceinline__ int find_layer_by_row(const FoldDesc* d, int n, int block) {
  int lo = 0, hi = n - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (d[mid].row0 <= block) lo = mid; else hi = mid - 1; }
  return lo;
}
__device__ __forceinline__ int find_layer_by_tile(const FoldDesc* d, int n, int block) {
  int lo = 0, hi = n - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (d[mid].tile0 <= block) lo = mid; else hi = mid - 1; }
  return lo;
}

// grid = sum of dim-0 rows over the layers; the block of a layer's first row also copies its bias
__global__ void __launch_bounds__(256)
weight_norm_scale_all_kernel(const float* params, const FoldDesc* d, int n_layers, float* scale) {
  __shared__ float red[32];
  const FoldDesc L = d[find_layer_by_row(d, n_layers, blockIdx.x)];
  const int row = blockIdx.x - L.row0;
  const int inner = L.Cc * L.K;
  const float* v = params + L.off_v + static_cast<size_t>(row) * inner;
  float s = 0.f;
  for (int i = threadIdx.x; i < inner; i += blockDim.x) { const float x = v[i]; s = fmaf(x, x, s); }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) scale[blockIdx.x] = params[L.off_g + row] / sqrtf(t);
  }
  if (row == 0 && L.off_bias >= 0)
    for (int i = threadIdx.x; i < L.Cout; i += blockDim.x) L.bias[i] = params[L.off_bias + i];
}

__global__ void __launch_bounds__(256)
fold_pack_all_kernel(const float* params, const FoldDesc* d, int n_layers, const float* scale) {
  __shared__ float tile[kPackTR][kPackTC * (kPackMaxK + 1)];
  const FoldDesc L = d[find_layer_by_tile(d, n_layers, blockIdx.x)];
  const int t = blockIdx.x - L.tile0;
  fold_pack_tile(tile, params + L.off_v, scale + L.row0, L.R, L.Cc, L.K, t % L.tiles_x, t / L.tiles_x, L.o1b, L.o1f, L.o2b,
                 L.o2f);
}

// one block per SnakeBeta layer
__global__ void snake_params_all_kernel(const float* params, const SnakeDesc* d, int logscale) {
  const SnakeDesc L = d[blockIdx.x];
  for (int c = threadIdx.x; c < L.C; c += blockDim.x) {
    float av = params[L.off_alpha + c], bv = params[L.off_beta + c];
    if (logscale) { av = expf(av); bv = expf(bv); }
    L.a[c] = av;
    L.inv_b[c] = 1.0f / (bv + 1e-9f);
  }
}

// ---------------------------------------------------------------- waveform -> int16 PCM
// The tail every caller of the decoder repeats (infer_0828_sigma.py:298, train_offline.py:302,319):
//   audio.to(float32).div(max|audio|).clamp(-1, 1).mul(32767).to(int16)
// two passes: peak (bit pattern of a non-negative float orders like an unsigned integer), then the same
// separately rounded div / mul and the truncating conversion torch performs.
__global__ void absmax_kernel(const void* x, size_t n, int f32, unsigned int* peak_bits) {
  float m = 0.f;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    m = fmaxf(m, fabsf(ld_elem(x, i, f32)));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(peak_bits, __float_as_uint(m));
}
__global__ void pcm16_kernel(const void* x, size_t n, int f32, const unsigned int* peak_bits, int16_t* out) {
  const float peak = __uint_as_float(*peak_bits);
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float v = __fdiv_rn(ld_elem(x, i, f32), peak);
    v = fminf(fmaxf(v, -1.f), 1.f);
    out[i] = static_cast<int16_t>(__float2int_rz(__fmul_rn(v, 32767.f)));
  }
}

__global__ void f32_to_bf16_kernel(const float* x, __nv_bfloat16* y, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    y[i] = __float2bfloat16(x[i]);
}

// ---------------------------------------------------------------- ragged batches
// A batch whose clips have different valid lengths is run at the padded length; after every layer the rows of each
// clip beyond ITS valid length are set to zero in the layer's output tensors, so the next convolution sees exactly
// the zero padding the reference's per-clip call would have applied at that clip's end (SnakeBeta(0) = 0, so a zero
// stream row is a zero operand row).  v[b] = valid rows of clip b in this tensor.
constexpr int kRaggedMaxClips = 64;
struct RaggedLens { int v[kRaggedMaxClips]; };
// grid: (blocks over the longest tail, clips of this group); base -> first clip of the group, channels-last rows
__global__ void zero_tail_rows_kernel(uint8_t* base, long long clip_bytes, int row_bytes, long long rows, RaggedLens lens) {
  const int b = blockIdx.y;
  long long valid = lens.v[b];
  if (valid >= rows) return;
  if (valid < 0) valid = 0;
  uint8_t* p0 = base + static_cast<size_t>(b) * clip_bytes + static_cast<size_t>(valid) * row_bytes;
  const size_t nbytes = static_cast<size_t>(rows - valid) * row_bytes;
  const size_t i0 = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x, step = static_cast<size_t>(gridDim.x) * blockDim.x;
  if (((reinterpret_cast<uintptr_t>(p0) | nbytes) & 15) == 0) {
    uint4* q = reinterpret_cast<uint4*>(p0);
    for (size_t i = i0; i < nbytes / 16; i += step) q[i] = make_uint4(0, 0, 0, 0);
  } else {   // row_bytes is always even (2- or 4-byte elements)
    uint16_t* q = reinterpret_cast<uint16_t*>(p0);
    for (size_t i = i0; i < nbytes / 2; i += step) q[i] = 0;
  }
}
// Channels-first, pitched sibling (the BigVGANFlowVAE ragged path): y[b, c, t] lives at y + (b * C + c) * ldy + t and is
// set to 0 for t in [v[b], T).  grid: (blocks over the longest tail, C, clips)
__global__ void zero_tail_cf_kernel(void* y, int C, long long T, long long ldy, RaggedLens lens, int f32) {
  const int b = blockIdx.z;
  const size_t row = (static_cast<size_t>(b) * C + blockIdx.y) * ldy;
  const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long t = lens.v[b] + blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < T; t += step)
    st_elem(y, row + t, f32, 0.f);
}

// twj_dataset.py:231-235 for a batch of mono clips: librosa.util.normalize(wav) * 0.95 (peak normalisation, clips
// whose peak is below float32 tiny stay as they are), duplicated to two channels, zero-padded to the batch length.
//   pass 1 (grid: (blocks, B)): per-clip absolute peak;  pass 2: out[b, 0 | 1, t] = wav_b[t] / peak_b * 0.95
__global__ void clip_peak_kernel(const float* wav, const long long* offsets, const int* lens, unsigned int* peak_bits) {
  const int b = blockIdx.y;
  const float* x = wav + offsets[b];
  const int n = lens[b];
  float m = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(peak_bits + b, __float_as_uint(m));
}
__global__ void clip_normalize_dup_kernel(const float* wav, const long long* offsets, const int* lens,
                                          const unsigned int* peak_bits, float gain, float* out, long long L_pad,
                                          int channels) {
  const int b = blockIdx.y;
  const float* x = wav + offsets[b];
  const int n = lens[b];
  const float peak = __uint_as_float(peak_bits[b]);
  const bool scale = peak > 1.17549435e-38f;            // librosa: norms below tiny are left alone (fill=None)
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < L_pad;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float v = 0.f;
    if (i < n) {
      v = x[i];
      if (scale) v = __fdiv_rn(v, peak);
      v = __fmul_rn(v, gain);
    }
    for (int c = 0; c < channels; ++c) out[(static_cast<size_t>(b) * channels + c) * L_pad + i] = v;
  }
}

// ---------------------------------------------------------------- latent sampling
// sample(mean, 'fix') of model_sigmaVAE.py:153-178,187-213: mean + std * noise, evaluated as torch
// does -- two separately rounded operations (mul then add), never an FMA -- so the result is
// bit-identical to the reference given the same noise tensor.  per_batch_std != nullptr is the
// 'gaussian' branch: std_b = std_noise[b] * (0.5 / 0.8), broadcast over the other dims.
__global__ void sigma_sample_kernel(const void* mean, const void* noise, void* out, size_t n, int f32, float std,
                                    const void* std_noise, float value, size_t per_batch) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float s = std;
    if (std_noise) {
      s = __fmul_rn(ld_elem(std_noise, i / per_batch, f32), value);
      if (!f32) s = __bfloat162float(__float2bfloat16(s));
    }
    float t = __fmul_rn(s, ld_elem(noise, i, f32));
    if (!f32) t = __bfloat162float(__float2bfloat16(t));
    st_elem(out, i, f32, __fadd_rn(ld_elem(mean, i, f32), t));
  }
}

// vae_sample of bottleneck.py:51-62 (as edited in the reference): latents = noise*scale + mean with
// the two roundings of torch; kl = (mean^2 + var - log var - 1).sum(1).mean() with
// stdev = softplus(scale) + 1e-4.  Per-block partial sums of the KL terms go to kl_partial
// (deterministic two-pass reduction; kvae_vae_sample finishes it).
__global__ void vae_sample_kernel(const void* mean, const void* scale, const void* noise, void* out, size_t n,
                                  int f32, double* kl_partial) {
  __shared__ double red[32];
  double acc = 0.0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float m = ld_elem(mean, i, f32), sc = ld_elem(scale, i, f32);
    float t = __fmul_rn(ld_elem(noise, i, f32), sc);
    if (!f32) t = __bfloat162float(__float2bfloat16(t));
    st_elem(out, i, f32, __fadd_rn(t, m));
    const float sp = (sc > 20.f) ? sc : log1pf(expf(sc));
    const float stdev = sp + 1e-4f;
    const float var = stdev * stdev;
    acc += static_cast<double>(m * m + var - logf(var) - 1.f);
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.0;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) kl_partial[blockIdx.x] = t;
  }
}
__global__ void kl_finish_kernel(const double* partial, int n, double denom, float* kl) {
  __shared__ double red[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) acc += partial[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (blockDim.x >> 5); ++i) t += red[i];
    *kl = static_cast<float>(t / denom);
  }
}

}  // namespace kvae
