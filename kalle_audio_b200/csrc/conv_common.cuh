// Pieces shared by the convolution kernels: the tap table of the implicit-GEMM convs and the SnakeBeta
// activation in the forms the epilogues use.
//
// A "tap" is (input phase, row shift, weight slab); taps that read the same input phase share ONE staged A slab and
// address it through row-shifted shared-memory descriptors, so the activations are fetched once per chunk instead of
// once per tap.
#pragma once
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>

#include "ptx.cuh"

namespace kvae {

constexpr int kMaxTaps = 32;
constexpr int kMaxPhases = 8;

struct Tap {
  int16_t a_phase;  // phase of the input view (strided conv), else 0
  int16_t a_row;    // slab start row relative to the tile's first output row (valid if first)
  int16_t shift;    // row offset of this tap inside the staged slab (>= 0)
  int16_t w_slab;   // packed-weight slab index
  int16_t first;    // 1: a new A slab is staged before this tap
  int16_t last;     // 1: last tap reading the current A slab
};

// sin(x) for the bf16-mode epilogues: the MUFU approximation as is (one FMUL by 1/(2*pi) + MUFU.SIN; the unit
// works on the fractional number of revolutions, so it is periodic by construction).  Its error is
// ~4e-7 + |x| * 2^-24 (the rounding of x/(2*pi)), i.e. < 1e-5 for |x| < 100 -- far below the bf16 rounding
// applied right after.  An explicit range reduction in front cost five more FMA-pipe instructions per
// element, and the fused epilogues at C = 128 are bound by exactly that pipe (64 lanes/clk/SM), see
// profiles/r01_conv_umma2_swap_k7_c128_B4.ncu-rep.
__device__ __forceinline__ float sin_fast(float x) { return __sinf(x); }

template <bool kFastSin>
__device__ __forceinline__ float snake_beta(float v, float a, float inv_b) {
  // reference blocks.py:301-302: x + (1/(beta + 1e-9)) * sin(x*alpha)^2
  const float s = kFastSin ? sin_fast(v * a) : sinf(v * a);
  return fmaf(inv_b * s, s, v);
}

// fp32-mode SnakeBeta inside the tensor-core epilogues: sinf costs ~40 instructions per element in epilogues that are
// issue-bound, so reduce the argument to [-pi, pi] with a two-constant Cody-Waite step (exact to ~1e-7 for |x| < 1e4)
// and use the MUFU sine there, where its absolute error is ~4e-7 -- an order of magnitude inside the 1e-5 budget.
__device__ __forceinline__ float snake_beta_rr(float v, float a, float inv_b) {
  const float t = v * a;
  const float k = rintf(t * 0.15915494309189535f);
  float r = fmaf(k, -6.2831854820251465f, t);          // 2*pi rounded to fp32
  r = fmaf(k, 1.7484555314695172e-7f, r);              // 2*pi - fp32(2*pi) = -1.7484555e-7, sign folded in
  const float s = __sinf(r);
  return fmaf(inv_b * s, s, v);
}

}  // namespace kvae
