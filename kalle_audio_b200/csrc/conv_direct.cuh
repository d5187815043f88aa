// Generic fp32 convolution on the CUDA cores.  Serves what the tensor-core kernel cannot:
//   * layers whose channel counts are not multiples of 64 -- the decoder's last conv
//     (128 -> io_channels, autoencoders.py:184) and the encoder's first (io_channels -> 128, :133),
//   * every layer in fp32 mode (<= 1e-5 budget), and small test architectures.
// Same tap decomposition as the tensor-core path (conv_umma_host.cuh::build_taps); input and
// raw output are addressed through element strides so the API layout [B, C, T] and the internal
// channels-last layout [B, T, C] are both read/written in place (no separate transposes).
// SnakeBeta can run as a prologue (applied once per staged element, not per tap) and/or as an
// epilogue producing the bf16 operand of a following tensor-core conv.
#pragma once
#include <cuda_bf16.h>
#include <cstdint>

#include "conv_common.cuh"  // Tap, kMaxTaps, kMaxPhases, snake_beta

namespace kvae {

struct DirectParams {
  int B, Tq_out, T_out, P_out, P_in, T_in, Cin, Cout, span;  // Tq_out = ceil(T_out / P_out)
  int tap_begin[kMaxPhases + 1];
  Tap taps[kMaxTaps];
  const void* x;
  int x_f32;
  long long x_sB, x_sT, x_sC;     // element strides of the input
  const float* pro_a;             // prologue SnakeBeta exp(alpha) [Cin] or nullptr
  const float* pro_inv_b;
  const float* w;                 // [K][Cin][Cout] fp32
  const float* bias;              // [Cout] or nullptr
  const void* residual;           // channels-last [B, T_out, Cout] or nullptr
  int residual_f32;
  void* out_raw;
  int out_raw_f32;
  long long o_sB, o_sT, o_sC;     // element strides of out_raw
  __nv_bfloat16* out_act;         // channels-last bf16 (SnakeBeta applied if snake_a)
  int act_split;                  // 1: out_act is [B, T, 2*Cout], bf16 (hi | lo) halves (fp32-mode tensor-core consumer)
  const float* snake_a;
  const float* snake_inv_b;
  int tanh_out;
  int q_base;                     // window form: first output row index q computed (blocks start there)
  int t_lo;                       // window form: outputs t < t_lo are not stored; out_raw holds t - t_lo
};

constexpr int kDirectKC = 16;

template <int BT, int BN, int TM, int TN>
__global__ void __launch_bounds__((BT / TM) * (BN / TN))
conv_direct_kernel(const __grid_constant__ DirectParams p) {
  constexpr int NTHREADS = (BT / TM) * (BN / TN);
  constexpr int KC = kDirectKC;
  extern __shared__ float smem_f[];
  const int slab_rows = BT + p.span;
  float* slab = smem_f;                              // [slab_rows][KC + 1]
  float* wt = smem_f + slab_rows * (KC + 1);         // [KC][BN]

  const int tid = threadIdx.x;
  const int tx = tid % (BN / TN);
  const int ty = tid / (BN / TN);
  const int phi = blockIdx.x % p.P_out;
  const int q0 = (blockIdx.x / p.P_out) * BT + p.q_base;
  const int n0 = blockIdx.y * BN;
  const int b = blockIdx.z;
  const int t_lo = p.tap_begin[phi], t_hi = p.tap_begin[phi + 1];

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  const bool time_fast = (p.x_sT == 1);  // API layout: walk time fastest for coalescing
  for (int c0 = 0; c0 < p.Cin; c0 += KC) {
    for (int t = t_lo; t < t_hi; ++t) {
      const Tap tap = p.taps[t];
      if (tap.first) {
        __syncthreads();
        for (int idx = tid; idx < slab_rows * KC; idx += NTHREADS) {
          const int r = time_fast ? idx % slab_rows : idx / KC;
          const int ci = time_fast ? idx / slab_rows : idx % KC;
          const int qi = q0 + tap.a_row + r;
          const long long ti = static_cast<long long>(qi) * p.P_in + tap.a_phase;
          float v = 0.f;
          if (qi >= 0 && ti < p.T_in && c0 + ci < p.Cin) {
            const long long off = b * p.x_sB + ti * p.x_sT + (c0 + ci) * p.x_sC;
            v = p.x_f32 ? static_cast<const float*>(p.x)[off]
                        : __bfloat162float(static_cast<const __nv_bfloat16*>(p.x)[off]);
            if (p.pro_a) v = snake_beta<false>(v, p.pro_a[c0 + ci], p.pro_inv_b[c0 + ci]);
          }
          slab[r * (KC + 1) + ci] = v;
        }
      }
      __syncthreads();
      for (int idx = tid; idx < KC * BN; idx += NTHREADS) {
        const int ci = idx / BN, co = idx % BN;
        float v = 0.f;
        if (c0 + ci < p.Cin && n0 + co < p.Cout)
          v = p.w[(static_cast<size_t>(tap.w_slab) * p.Cin + c0 + ci) * p.Cout + n0 + co];
        wt[ci * BN + co] = v;
      }
      __syncthreads();
#pragma unroll 4
      for (int ci = 0; ci < KC; ++ci) {
        float a[TM], w[TN];
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] = slab[(ty * TM + i + tap.shift) * (KC + 1) + ci];
#pragma unroll
        for (int j = 0; j < TN; ++j) w[j] = wt[ci * BN + tx * TN + j];
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
          for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
      }
    }
  }

  const int T_out = p.T_out;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int q = q0 + ty * TM + i;
    if (q >= p.Tq_out) continue;
    const long long t_out = static_cast<long long>(q) * p.P_out + phi;
    if (t_out >= T_out || t_out < p.t_lo) continue;
    const size_t cl_row = (static_cast<size_t>(b) * T_out + t_out) * p.Cout;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int co = n0 + tx * TN + j;
      if (co >= p.Cout) continue;
      float v = acc[i][j];
      if (p.bias) v += p.bias[co];
      if (p.residual)
        v += p.residual_f32 ? static_cast<const float*>(p.residual)[cl_row + co]
                            : __bfloat162float(static_cast<const __nv_bfloat16*>(p.residual)[cl_row + co]);
      if (p.tanh_out) v = tanhf(v);
      if (p.out_raw) {
        const long long off = b * p.o_sB + (t_out - p.t_lo) * p.o_sT + co * p.o_sC;
        if (p.out_raw_f32) static_cast<float*>(p.out_raw)[off] = v;
        else static_cast<__nv_bfloat16*>(p.out_raw)[off] = __float2bfloat16(v);
      }
      if (p.out_act) {
        float a = v;
        if (p.snake_a) a = snake_beta<false>(v, p.snake_a[co], p.snake_inv_b[co]);
        if (p.act_split) {
          const __nv_bfloat16 hi = __float2bfloat16(a);
          p.out_act[2 * cl_row + co] = hi;
          p.out_act[2 * cl_row + p.Cout + co] = __float2bfloat16(a - __bfloat162float(hi));
        } else {
          p.out_act[cl_row + co] = __float2bfloat16(a);
        }
      }
    }
  }
}

}  // namespace kvae
