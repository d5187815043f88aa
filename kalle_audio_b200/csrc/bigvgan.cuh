// Leaf kernels of the BigVGANFlowVAE inference path (reference /root/reference/backup/flows.py:396-529): the
// anti-aliased periodic activation of its AMP blocks and the small elementwise steps between the convolutions, and
// their backward (BigVGANFlowVAE.decode_with_grad).  The convolutions themselves run through the layer-level conv
// (kvae_conv1d_pack + kvae_conv1d_win_fwd; backward kvae_conv1d_win_bwd).
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
// kRagged (a batch of clips of different lengths): clip b = row / C ends at its own lens.v[b] instead of t_end, and
// outputs t >= lens.v[b] are stored as 0, so a following conv reads the zero padding the clip's own call would have.
// Otherwise lens is not read; the window and whole-row calls compile to the code they had before.
template <bool kRagged>
__global__ void __launch_bounds__(256) aa_act_kernel(const void* x, long long ldx, long long x0, long long nx, void* y,
                                                     long long ldy, long long o0, long long o1, long long t_end,
                                                     const float* alpha, const float* beta, int logscale,
                                                     const float* fu, const float* fd, int C, int f32, RaggedLens lens) {
  __shared__ float xs[kAaTile + 16];
  __shared__ float vs[2 * kAaTile + kAaK];
  __shared__ float f_up[kAaK], f_dn[kAaK];
  const int c = blockIdx.y % C;
  const size_t row_x = static_cast<size_t>(blockIdx.y) * ldx, row_y = static_cast<size_t>(blockIdx.y) * ldy;
  const long long t0 = o0 + static_cast<long long>(blockIdx.x) * kAaTile;   // absolute
  if constexpr (kRagged) {
    t_end = lens.v[blockIdx.y / C];
    if (t0 >= t_end) {                                          // a tile past the clip's end: zeros only
      for (int tl = threadIdx.x; tl < kAaTile && t0 + tl < o1; tl += 256) st_elem(y, row_y + (t0 + tl - o0), f32, 0.f);
      return;
    }
  }
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
      st_elem(y, row_y + (t0 + tl - o0), f32, !kRagged || t0 + tl < t_end ? acc : 0.f);
    }
  }
}

// Backward of aa_act_kernel over whole rows (x0 = o0 = 0, o1 = t_end = T), recomputing u from x tile by tile as the
// forward does: nothing at the double rate is stored between the two passes.  With gvp / gxp the gradients of the
// padded v / x (the adjoints of the decimation and of the up-filter):
//   gvp[j] = sum_t gy[t] fd[j - 2 t]                     0 <= j - 2 t < 12
//   gv[n]  = gvp[n + 5]  (+ gvp[0 .. 4] at n = 0, + gvp[2T + 5 .. 2T + 9] at n = 2T - 1: the replicate padding folded back)
//   gu[n]  = gv[n] (1 + inv_b a sin(2 a u[n]))
//   gxp[i] = 2 sum_n gu[n] fu[n + 15 - 2 i]              0 <= n + 15 - 2 i < 12,  n in [0, 2T)
//   gx[t]  = gxp[t + 5]  (+ gxp[2 .. 4] at t = 0, + gxp[T + 5 .. T + 7] at t = T - 1)
// gx[t] reads gy[t - 5 .. t + 5] and x[t - 8 .. t + 8]: the tile stages both with their halos.  The parameter terms
// dv/da = inv_b u sin(2 a u) and dv/db = -inv_b^2 sin^2(a u) share the per-channel factors, so the block sums
// gv u sin(2 a u) and gv sin^2(a u) over its own double-rate samples n in [2 t0, 2 t1) (in double: the terms cancel)
// and writes them as ONE partial per (row, tile); aa_act_bwd_params_kernel reduces them in a fixed order.
__global__ void __launch_bounds__(256) aa_act_bwd_kernel(const void* x, const void* gy, void* gx, double* part, long long T,
                                                         const float* alpha, const float* beta, int logscale,
                                                         const float* fu, const float* fd, int C, int f32) {
  __shared__ float xs[kAaTile + 16];                 // x rows t0 - 8 .. t0 + TT + 7, replicate padded
  __shared__ float gys[kAaTile + 21];                // gy rows t0 - 10 .. t0 + TT + 10, zero outside [0, T)
  __shared__ float gus[2 * kAaTile + 22];            // gu at n - 2 t0 in [-11, 2 TT + 11)
  __shared__ float gxs[kAaTile + 6];                 // gxp at i - 5 - t0 in [-3, TT + 3)
  __shared__ float f_up[kAaK], f_dn[kAaK];
  __shared__ double red[2][8];
  const int c = blockIdx.y % C;
  const size_t row = static_cast<size_t>(blockIdx.y) * T;
  const long long t0 = static_cast<long long>(blockIdx.x) * kAaTile;
  if (threadIdx.x < kAaK) { f_up[threadIdx.x] = fu[threadIdx.x]; f_dn[threadIdx.x] = fd[threadIdx.x]; }
  float a = alpha[c], bt = beta ? beta[c] : alpha[c];
  if (logscale) { a = expf(a); bt = expf(bt); }
  const float inv_b = 1.0f / (bt + 1e-9f);
  const int lo_x = static_cast<int>(-min(t0, 64ll)), hi_x = static_cast<int>(min(T - 1 - t0, static_cast<long long>(kAaTile + 64)));
  // double-rate samples that exist, relative to 2 t0: [lo_n, hi_n)
  const int lo_n = 2 * lo_x, hi_n = static_cast<int>(min(2 * T - 2 * t0, static_cast<long long>(2 * kAaTile + 64)));
  const int tile_t = static_cast<int>(min(T - t0, static_cast<long long>(kAaTile)));
  for (int i = threadIdx.x; i < kAaTile + 16; i += 256)
    xs[i] = ld_elem(x, row + (t0 + max(lo_x, min(hi_x, i - 8))), f32);
  for (int i = threadIdx.x; i < kAaTile + 21; i += 256) {
    const int r = i - 10;
    gys[i] = (r >= lo_x && r <= hi_x) ? ld_elem(gy, row + (t0 + r), f32) : 0.f;
  }
  __syncthreads();
  auto gvp = [&](int j) {                            // gvp at j - 2 t0: six taps of one parity
    const int m0 = j & 1;
    const float* g = gys + 10 + ((j - m0) >> 1);
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < 6; ++q) acc = fmaf(g[-q], f_dn[m0 + 2 * q], acc);
    return acc;
  };
  double sa = 0.0, sb = 0.0;
  for (int j = threadIdx.x; j < 2 * kAaTile + 22; j += 256) {
    const int n = j - 11;
    float g = 0.f;
    if (n >= lo_n && n < hi_n) {
      float gv = gvp(n + 5);
      if (n == lo_n && t0 == 0)
        for (int q = 0; q < 5; ++q) gv += gvp(q);
      if (n == hi_n - 1 && hi_n < 2 * kAaTile + 64)
        for (int q = 6; q < 11; ++q) gv += gvp(n + q);
      const int i_lo = (n + 5) >> 1;                 // u[n] exactly as aa_act_kernel builds it
      const int k0 = n + 15 - 2 * i_lo;
      const float* xp = xs + i_lo + 3;
      float u = 0.f;
#pragma unroll
      for (int q = 0; q < 6; ++q) u = fmaf(xp[q], f_up[k0 - 2 * q], u);
      u *= 2.f;
      float s, co;
      sincosf(u * a, &s, &co);
      const float s2 = 2.f * s * co;                 // sin(2 a u)
      g = gv * (1.f + inv_b * a * s2);
      if (n >= 0 && n < 2 * tile_t) {
        sa = fma(static_cast<double>(gv), static_cast<double>(u * s2), sa);
        sb = fma(static_cast<double>(gv), static_cast<double>(s * s), sb);
      }
    }
    gus[j] = g;
  }
  __syncthreads();
  for (int r = threadIdx.x; r < kAaTile + 6; r += 256) {
    const float* g = gus + 2 * r;                    // gu at n - 2 t0 = 2 (r - 3) - 5 + m, m in [0, 12)
    float acc = 0.f;
#pragma unroll
    for (int m = 0; m < kAaK; ++m) acc = fmaf(g[m], f_up[m], acc);
    gxs[r] = 2.f * acc;
  }
  for (int o = 16; o > 0; o >>= 1) {
    sa += __shfl_xor_sync(0xffffffffu, sa, o);
    sb += __shfl_xor_sync(0xffffffffu, sb, o);
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = sa; red[1][threadIdx.x >> 5] = sb; }
  __syncthreads();
  if (threadIdx.x == 0 && part) {                  // part == nullptr: no parameter gradient wanted
    double ta = 0.0, tb = 0.0;
    for (int w = 0; w < 8; ++w) { ta += red[0][w]; tb += red[1][w]; }
    const size_t pi = (static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * 2;
    part[pi] = ta;
    part[pi + 1] = tb;
  }
#pragma unroll
  for (int r = 0; r < kAaTile / 256; ++r) {
    const int tl = threadIdx.x + 256 * r;
    if (tl < tile_t) {
      float g = gxs[tl + 3];
      if (t0 + tl == 0) g += gxs[0] + gxs[1] + gxs[2];
      if (t0 + tl == T - 1) g += gxs[tl + 4] + gxs[tl + 5] + gxs[tl + 6];
      st_elem(gx, row + (t0 + tl), f32, g);
    }
  }
}

// d alpha / d beta from aa_act_bwd_kernel's partials [B, C, tiles, 2]: one block per channel, each thread sums its
// partials in index order, then a fixed tree -- the same bits on every call.  Snake (beta == nullptr): a is also the b,
// so both terms go to d alpha.  logscale: a = exp(alpha), b = exp(beta), so each term is multiplied by a or b.
__global__ void aa_act_bwd_params_kernel(const double* part, const float* alpha, const float* beta, int logscale,
                                         float* dalpha, float* dbeta, int B, int C, int tiles) {
  __shared__ double red[2][256];
  const int c = blockIdx.x;
  double sa = 0.0, sb = 0.0;
  for (int i = threadIdx.x; i < B * tiles; i += blockDim.x) {
    const int b = i / tiles, tile = i % tiles;
    const size_t pi = ((static_cast<size_t>(b) * C + c) * tiles + tile) * 2;
    sa += part[pi];
    sb += part[pi + 1];
  }
  red[0][threadIdx.x] = sa;
  red[1][threadIdx.x] = sb;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) {
      red[0][threadIdx.x] += red[0][threadIdx.x + h];
      red[1][threadIdx.x] += red[1][threadIdx.x + h];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    float a = alpha[c], bt = beta ? beta[c] : alpha[c];
    if (logscale) { a = expf(a); bt = expf(bt); }
    const double inv_b = 1.0 / (static_cast<double>(bt) + 1e-9);
    const double da = inv_b * red[0][0] * (logscale ? a : 1.0);
    const double db = -inv_b * inv_b * red[1][0] * (logscale ? bt : 1.0);
    if (beta) { dalpha[c] = static_cast<float>(da); dbeta[c] = static_cast<float>(db); }
    else dalpha[c] = static_cast<float>(da + db);
  }
}

// op 0: leaky_relu(x, slope = param); op 1: tanh
__global__ void unary_kernel(const void* x, void* y, size_t n, int op, float param, int f32) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float v = ld_elem(x, i, f32);
    st_elem(y, i, f32, op == 0 ? (v >= 0.f ? v : v * param) : tanhf(v));
  }
}
// backward of unary_kernel: op 0 reads the forward's input t = x, gx = gy * (x > 0 ? 1 : param) (torch's leaky_relu
// backward); op 1 reads the forward's output t = y, gx = gy * (1 - y^2)
__global__ void unary_bwd_kernel(const void* t, const void* gy, void* gx, size_t n, int op, float param, int f32) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float v = ld_elem(t, i, f32), g = ld_elem(gy, i, f32);
    st_elem(gx, i, f32, op == 0 ? (v > 0.f ? g : g * param) : g * (1.f - v * v));
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
// backward of the sample on the latents x = [B, 2 D, T] (mean | logs, torch.split at flows.py:500): gz and noise are
// [B, D, T] (DT = D * T per clip); gx[:, :D] = gz, gx[:, D:] = gz * noise * exp(logs)
__global__ void gauss_sample_bwd_kernel(const void* x, const void* noise, const void* gz, void* gx, long long DT, size_t n,
                                        int f32) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t b = i / DT, base = b * 2 * DT + (i - b * DT);
    const float g = ld_elem(gz, i, f32);
    st_elem(gx, base, f32, g);
    st_elem(gx, base + DT, f32, g * ld_elem(noise, i, f32) * expf(ld_elem(x, base + DT, f32)));
  }
}

}  // namespace kvae
