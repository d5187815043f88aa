// Elementwise kernels of BigVGANFlowVAE's flow, the VITS ResidualCouplingBlock (reference backup/flows.py:613-792): the
// WaveNet gate (fused_add_tanh_sigmoid_multiply without conditioning), WN's residual / skip update, the mask multiply
// after `pre`, and the coupling update with the channel reversal of `Flip`, each with its backward.  All of them work on
// [B, C, T] tensors of fp32 or bf16 (fp32 arithmetic, one rounding per stored value) with a [B, 1, T] mask of the same
// dtype; a block owns one (b, channel) row segment, so no index division runs per element.  The convolutions of the
// flow (`pre`, `post`, WN's `in_layers` / `res_skip_layers`) run through the layer-level conv; no reduction happens here.
#pragma once
#include <cuda_bf16.h>
#include <cstdint>

#include "elementwise.cuh"

namespace kvae {

constexpr int kFlowThreads = 128;   // rows are short at 12.5 Hz (100 .. 375 frames per clip)

// Split / Flip: xs = x, or x with its channels reversed (flip), and x0 = xs[:, :C/2] as a contiguous copy (the
// coupling layer's `pre` input) when x0 != NULL.  grid (ceil(T / kFlowThreads), B * C)
__global__ void __launch_bounds__(kFlowThreads) flow_split_kernel(const void* x, void* xs, void* x0, int C, long long T,
                                                                  int flip, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / C, c = blockIdx.y - b * C, half = C / 2;
  const int src = flip ? C - 1 - c : c;
  const float v = ld_elem(x, (static_cast<size_t>(b) * C + src) * T + t, f32);
  st_elem(xs, static_cast<size_t>(blockIdx.y) * T + t, f32, v);
  if (x0 && c < half) st_elem(x0, (static_cast<size_t>(b) * half + c) * T + t, f32, v);
}
// backward: gx[src] = gxs[c] + gx0[c] (c < C/2); either gradient may be NULL (an unused output)
__global__ void __launch_bounds__(kFlowThreads) flow_split_bwd_kernel(const void* gxs, const void* gx0, void* gx, int C,
                                                                      long long T, int flip, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / C, c = blockIdx.y - b * C, half = C / 2;
  float g = gxs ? ld_elem(gxs, static_cast<size_t>(blockIdx.y) * T + t, f32) : 0.f;
  if (gx0 && c < half) g += ld_elem(gx0, (static_cast<size_t>(b) * half + c) * T + t, f32);
  st_elem(gx, (static_cast<size_t>(b) * C + (flip ? C - 1 - c : c)) * T + t, f32, g);
}

// y = x * mask (h = pre(x0) * x_mask; its backward is the same product with the output gradient).  grid (.., B * C)
__global__ void __launch_bounds__(kFlowThreads) flow_mask_kernel(const void* x, const void* mask, void* y, int C,
                                                                 long long T, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const size_t i = static_cast<size_t>(blockIdx.y) * T + t;
  st_elem(y, i, f32, ld_elem(x, i, f32) * ld_elem(mask, static_cast<size_t>(blockIdx.y / C) * T + t, f32));
}

// WN gate: acts = tanh(a[:, :H]) * sigmoid(a[:, H:]) from a [B, 2H, T].  grid (.., B * H)
__global__ void __launch_bounds__(kFlowThreads) wn_gate_kernel(const void* a, void* acts, int H, long long T, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / H, c = blockIdx.y - b * H;
  const size_t ia = (static_cast<size_t>(b) * 2 * H + c) * T + t, ib = ia + static_cast<size_t>(H) * T;
  const float th = tanhf(ld_elem(a, ia, f32));
  const float sg = 1.f / (1.f + expf(-ld_elem(a, ib, f32)));
  st_elem(acts, static_cast<size_t>(blockIdx.y) * T + t, f32, th * sg);
}
// backward from the saved a: ga[:, :H] = g s (1 - t^2), ga[:, H:] = g t s (1 - s), both halves in one pass
__global__ void __launch_bounds__(kFlowThreads) wn_gate_bwd_kernel(const void* a, const void* g, void* ga, int H,
                                                                   long long T, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / H, c = blockIdx.y - b * H;
  const size_t ia = (static_cast<size_t>(b) * 2 * H + c) * T + t, ib = ia + static_cast<size_t>(H) * T;
  const float th = tanhf(ld_elem(a, ia, f32));
  const float sg = 1.f / (1.f + expf(-ld_elem(a, ib, f32)));
  const float gv = ld_elem(g, static_cast<size_t>(blockIdx.y) * T + t, f32);
  st_elem(ga, ia, f32, gv * sg * (1.f - th * th));
  st_elem(ga, ib, f32, gv * th * sg * (1.f - sg));
}

// WN residual / skip update of layer i from rs = res_skip_layers[i](acts) and the running skip sum (skip == NULL: the
// first layer, skip = 0).  Not the last layer (rs [B, 2H, T]): x_out = (x + rs[:, :H]) * mask, skip_out = skip +
// rs[:, H:].  The last layer (rs [B, H, T]): skip_out = (skip + rs) * mask, WN's output; x and x_out are not used.
// grid (.., B * H)
__global__ void __launch_bounds__(kFlowThreads) wn_update_kernel(const void* x, const void* rs, const void* skip,
                                                                 const void* mask, void* x_out, void* skip_out, int H,
                                                                 int last, long long T, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / H, c = blockIdx.y - b * H;
  const size_t i = static_cast<size_t>(blockIdx.y) * T + t;
  const float mk = ld_elem(mask, static_cast<size_t>(b) * T + t, f32);
  const float s = skip ? ld_elem(skip, i, f32) : 0.f;
  if (last) {
    st_elem(skip_out, i, f32, (s + ld_elem(rs, i, f32)) * mk);
    return;
  }
  const size_t ir = (static_cast<size_t>(b) * 2 * H + c) * T + t;
  st_elem(x_out, i, f32, (ld_elem(x, i, f32) + ld_elem(rs, ir, f32)) * mk);
  st_elem(skip_out, i, f32, s + ld_elem(rs, ir + static_cast<size_t>(H) * T, f32));
}
// backward.  Not the last layer: gx = g_xout * mask, grs[:, :H] = g_xout * mask, grs[:, H:] = g_skipout (the skip
// input's gradient is g_skipout itself; gskip, when given, gets a copy).  The last layer: grs = gskip = g_skipout *
// mask.  A NULL output gradient reads as 0.
__global__ void __launch_bounds__(kFlowThreads) wn_update_bwd_kernel(const void* g_xout, const void* g_skipout,
                                                                     const void* mask, void* gx, void* grs, void* gskip,
                                                                     int H, int last, long long T, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / H, c = blockIdx.y - b * H;
  const size_t i = static_cast<size_t>(blockIdx.y) * T + t;
  const float mk = ld_elem(mask, static_cast<size_t>(b) * T + t, f32);
  const float gs = g_skipout ? ld_elem(g_skipout, i, f32) : 0.f;
  if (last) {
    st_elem(grs, i, f32, gs * mk);
    if (gskip) st_elem(gskip, i, f32, gs * mk);
    return;
  }
  const float gxm = (g_xout ? ld_elem(g_xout, i, f32) : 0.f) * mk;
  const size_t ir = (static_cast<size_t>(b) * 2 * H + c) * T + t;
  st_elem(gx, i, f32, gxm);
  st_elem(grs, ir, f32, gxm);
  st_elem(grs, ir + static_cast<size_t>(H) * T, f32, gs);
  if (gskip) st_elem(gskip, i, f32, gs);
}

// Coupling (ResidualCouplingLayer with mean_only, logs = 0) from the layer input x [B, C, T] and m = post(h) [B, C/2, T]:
// with mm = m * mask, x1' = mm + x1 * mask (forward) or (x1 - mm) * mask (reverse); y = cat(x0, x1'), written with its
// channels reversed when flip (the Flip that follows the layer), and y0 = y[:, :C/2] as a contiguous copy when y0 !=
// NULL (the next layer's `pre` input).  grid (.., B * C/2)
__global__ void __launch_bounds__(kFlowThreads) flow_coupling_kernel(const void* x, const void* m, const void* mask,
                                                                     void* y, void* y0, int half, long long T, int flip,
                                                                     int reverse, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / half, c = blockIdx.y - b * half;
  const size_t row0 = static_cast<size_t>(b) * 2 * half;
  const float mk = ld_elem(mask, static_cast<size_t>(b) * T + t, f32);
  const float x0 = ld_elem(x, (row0 + c) * T + t, f32), x1 = ld_elem(x, (row0 + half + c) * T + t, f32);
  const float mm = ld_elem(m, static_cast<size_t>(blockIdx.y) * T + t, f32) * mk;
  const float x1n = reverse ? (x1 - mm) * mk : mm + x1 * mk;
  const int c0 = flip ? 2 * half - 1 - c : c, c1 = flip ? half - 1 - c : half + c;
  st_elem(y, (row0 + c0) * T + t, f32, x0);
  st_elem(y, (row0 + c1) * T + t, f32, x1n);
  if (y0) {          // y's first half: x1' reversed under flip, x0 otherwise
    const int cc = flip ? c1 : c;
    st_elem(y0, (static_cast<size_t>(b) * half + cc) * T + t, f32, flip ? x1n : x0);
  }
}
// backward: gx[:, :C/2] = the gradient of y's x0 channels (+ gy0 without flip), gx[:, C/2:] = g1 * mask and gm = g1 *
// mask (forward) or -g1 * mask^2 (reverse), with g1 the gradient of the x1' channels (+ gy0 under flip).  gy or gy0 NULL:
// an unused output.  Neither x nor m is read.
__global__ void __launch_bounds__(kFlowThreads) flow_coupling_bwd_kernel(const void* gy, const void* gy0,
                                                                         const void* mask, void* gx, void* gm, int half,
                                                                         long long T, int flip, int reverse, int f32) {
  const long long t = blockIdx.x * static_cast<long long>(kFlowThreads) + threadIdx.x;
  if (t >= T) return;
  const int b = blockIdx.y / half, c = blockIdx.y - b * half;
  const size_t row0 = static_cast<size_t>(b) * 2 * half;
  const float mk = ld_elem(mask, static_cast<size_t>(b) * T + t, f32);
  const int c0 = flip ? 2 * half - 1 - c : c, c1 = flip ? half - 1 - c : half + c;
  float g0 = gy ? ld_elem(gy, (row0 + c0) * T + t, f32) : 0.f;
  float g1 = gy ? ld_elem(gy, (row0 + c1) * T + t, f32) : 0.f;
  if (gy0) {
    const float gg = ld_elem(gy0, (static_cast<size_t>(b) * half + (flip ? c1 : c)) * T + t, f32);
    if (flip) g1 += gg; else g0 += gg;
  }
  st_elem(gx, (row0 + c) * T + t, f32, g0);
  st_elem(gx, (row0 + half + c) * T + t, f32, g1 * mk);
  st_elem(gm, static_cast<size_t>(blockIdx.y) * T + t, f32, reverse ? -(g1 * mk) * mk : g1 * mk);
}

}  // namespace kvae
