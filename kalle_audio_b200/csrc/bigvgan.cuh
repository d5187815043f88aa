// Leaf kernels of the BigVGANFlowVAE inference path (reference /root/reference/backup/flows.py:396-529): the
// anti-aliased periodic activation of its AMP blocks and the small elementwise steps between the convolutions.
// The convolutions themselves run through the generic conv kernels (kvae_conv1d_fwd).
#pragma once
#include <cuda_bf16.h>
#include <cstdint>

#include "elementwise.cuh"

namespace kvae {

// Activation1d (alias_free_torch, used at flows.py:266, 312, 443): upsample x2 with a 12-tap Kaiser-sinc filter
// (replicate padding), Snake / SnakeBeta at the doubled rate, low-pass + decimate x2 with the same kind of filter.
// ONE pass over [B, C, T]: a block stages a row segment of x with its halo, builds the activated double-rate signal
// in shared memory and decimates it -- the reference runs pad + conv_transpose + crop + activation + pad + conv
// (six eager kernels, four full-size intermediates at twice the rate).
//   u[n]  = 2 * sum_i xp[i] * fu[n + 15 - 2 i]      xp[i] = x[clamp(i - 5, 0, T-1)], 0 <= n + 15 - 2 i < 12,  n in [0, 2T)
//   v[n]  = u[n] + inv_b * sin(a * u[n])^2
//   y[t]  = sum_m vp[2 t + m] * fd[m]               vp[j] = v[clamp(j - 5, 0, 2T-1)],  m in [0, 12)
constexpr int kAaTile = 1024;                        // outputs per block
constexpr int kAaK = 12;
constexpr int kAaHalo = 5;                           // y[t] reads x[t - 5 .. t + 5]
constexpr long long kAaNoEnd = 1ll << 60;            // t_end of a window whose stream has not ended
// Window form (the streaming decoder's unit of work; the whole-row call is the case x0 = o0 = 0, o1 = t_end = T):
// x holds the absolute rows [x0, x0 + nx) of every (b, c) row at pitch ldx, outputs t in [o0, o1) go to
// y[(b, c) * ldy + t - o0].  Replicate padding applies at absolute row 0 and at the stream end t_end (kAaNoEnd: none),
// so a window away from both edges computes exactly what the whole row computes there.  The caller guarantees that
// rows [max(0, o0 - 5), min(o1 + 5, t_end)) are inside the window; halo rows outside it are never used by a stored
// output and are staged as 0.
// Everything inside a tile is indexed relative to the tile start in 32 bits; 64-bit arithmetic only places the tile
// and clamps at the two ends of the row (the first version did every tap's index in 64 bits and spent ~60 % of its
// instructions there: 21 of the 60 ms of the bench decode).  Same operations in the same order per sample.
__global__ void __launch_bounds__(256) aa_act_kernel(const void* x, long long ldx, long long x0, long long nx, void* y,
                                                     long long ldy, long long o0, long long o1, long long t_end,
                                                     const float* alpha, const float* beta, int logscale,
                                                     const float* fu, const float* fd, int C, int f32) {
  __shared__ float xs[kAaTile + 16];
  __shared__ float vs[2 * kAaTile + kAaK];
  __shared__ float f_up[kAaK], f_dn[kAaK];
  const int c = blockIdx.y % C;
  const size_t row_x = static_cast<size_t>(blockIdx.y) * ldx, row_y = static_cast<size_t>(blockIdx.y) * ldy;
  const long long t0 = o0 + static_cast<long long>(blockIdx.x) * kAaTile;   // absolute
  if (threadIdx.x < kAaK) { f_up[threadIdx.x] = fu[threadIdx.x]; f_dn[threadIdx.x] = fd[threadIdx.x]; }
  float a = alpha[c], bt = beta ? beta[c] : alpha[c];          // Snake: 1/alpha; SnakeBeta: 1/beta
  if (logscale) { a = expf(a); bt = expf(bt); }
  const float inv_b = 1.0f / (bt + 1e-9f);
  // rows still inside the stream, relative to the tile: x index i_rel = t - t0 in [lo_x, hi_x], v index n - 2 t0 in [lo_v, hi_v]
  const int lo_x = static_cast<int>(-min(t0, 64ll)), hi_x = static_cast<int>(min(t_end - 1 - t0, static_cast<long long>(kAaTile + 64)));
  const int lo_v = 2 * lo_x, hi_v = static_cast<int>(min(2 * t_end - 1 - 2 * t0, static_cast<long long>(2 * kAaTile + 64)));
  // x rows t0 - 8 .. t0 + TT + 7 (clamped = replicate padding)
  for (int i = threadIdx.x; i < kAaTile + 16; i += 256) {
    const long long r = t0 + max(lo_x, min(hi_x, i - 8)) - x0;
    xs[i] = (r >= 0 && r < nx) ? ld_elem(x, row_x + r, f32) : 0.f;
  }
  __syncthreads();
  // activated double-rate samples n = 2 t0 - 5 .. 2 t0 + 2 TT + 6, the index clamped to [0, 2 t_end) (replicate padding of v)
  for (int j = threadIdx.x; j < 2 * kAaTile + kAaK; j += 256) {
    const int n = max(lo_v, min(hi_v, j - 5));                  // relative to 2 t0
    // taps i with 0 <= n + 15 - 2 i <= 11: six of them, from i_lo = floor((n + 5) / 2)
    const int i_lo = (n + 5) >> 1;
    const int k0 = n + 15 - 2 * i_lo;                           // 10 or 11
    const float* xp = xs + i_lo + 3;                            // xs index of x[i - 5] = (i - 5) + 8
    float u = 0.f;
#pragma unroll
    for (int q = 0; q < 6; ++q) u = fmaf(xp[q], f_up[k0 - 2 * q], u);
    u *= 2.f;
    const float s = sinf(u * a);
    vs[j] = u + inv_b * (s * s);
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kAaTile / 256; ++r) {
    const int tl = threadIdx.x + 256 * r;
    if (t0 + tl < o1) {
      float acc = 0.f;
#pragma unroll
      for (int m = 0; m < kAaK; ++m) acc = fmaf(vs[2 * tl + m], f_dn[m], acc);
      st_elem(y, row_y + (t0 + tl - o0), f32, acc);
    }
  }
}

// op 0: leaky_relu(x, slope = param); op 1: tanh
__global__ void unary_kernel(const void* x, void* y, size_t n, int op, float param, int f32) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float v = ld_elem(x, i, f32);
    st_elem(y, i, f32, op == 0 ? (v >= 0.f ? v : v * param) : tanhf(v));
  }
}
// out = alpha * a + beta * b (residual adds, the average over the AMP blocks of a stage)
__global__ void axpby_kernel(const void* a, const void* b, void* out, size_t n, float alpha, float beta, int f32) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    st_elem(out, i, f32, __fadd_rn(__fmul_rn(alpha, ld_elem(a, i, f32)), __fmul_rn(beta, ld_elem(b, i, f32))));
}
// z = mean + noise * exp(logs) (flows.py:500-501), the three torch roundings kept separate
__global__ void gauss_sample_kernel(const void* mean, const void* logs, const void* noise, void* out, size_t n, int f32) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float e = expf(ld_elem(logs, i, f32));
    if (!f32) e = __bfloat162float(__float2bfloat16(e));
    float t = __fmul_rn(ld_elem(noise, i, f32), e);
    if (!f32) t = __bfloat162float(__float2bfloat16(t));
    st_elem(out, i, f32, __fadd_rn(ld_elem(mean, i, f32), t));
  }
}

}  // namespace kvae
