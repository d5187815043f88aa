// Kernels of the training step (BASELINE config 5; the reference gets these from autograd through
// stable_audio_tools/models/autoencoders.py:39-191, blocks.py:301-339, bottleneck.py:51-62 and
// torch.nn.utils.weight_norm -- there is no hand-written backward in the reference):
//   snake_bwd_kernel      G_prev = dA * SnakeBeta'(x) (+ skip-connection gradient); per-channel sums for
//                         d alpha, d beta and the producing conv's bias gradient, all in one HBM pass
//   wgrad_direct_kernel   fp32 CUDA-core weight gradient of Conv1d / ConvTranspose1d (fp32 mode, edge convs)
//   weight_norm_bwd       (dg, dv) from dw for torch.nn.utils.weight_norm(dim=0)
//   vae_sample_bwd / gaussian_nll / adamw   latent sampling gradient, the sigma-VAE loss, the optimizer
// All activations are channels-last [B, T, C]; gradients of the stream are fp32, with a bf16 copy as the
// tensor-core operand of the data-/weight-gradient GEMMs.
#pragma once
#include "ptx.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "conv_common.cuh"  // snake_beta
#include "elementwise.cuh"  // ld_elem / st_elem

namespace kvae {

// ---------------------------------------------------------------- [B, C, T] -> [B, T, C] fp32
// grid (ceil(T/32), ceil(C/32), B), block (32, 8)
__global__ void cf_to_cl_f32_kernel(const void* x, int f32, float* y, int C, long long T) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const long long t0 = static_cast<long long>(blockIdx.x) * 32;
  const int c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i;
    const long long t = t0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && t < T) ? ld_elem(x, (static_cast<size_t>(b) * C + c) * T + t, f32) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const long long t = t0 + i;
    const int c = c0 + threadIdx.x;
    if (c < C && t < T) y[(static_cast<size_t>(b) * T + t) * C + c] = tile[threadIdx.x][i];
  }
}

// ---------------------------------------------------------------- bias gradient, [B, C, T] layout
// db[c] = sum_{b,t} gy[b, c, t].  One block per channel.
__global__ void bias_grad_cf_kernel(const void* gy, int f32, float* db, int B, int C, long long T) {
  __shared__ float red[32];
  const int c = blockIdx.x;
  float s = 0.f;
  for (int b = 0; b < B; ++b) {
    const size_t base = (static_cast<size_t>(b) * C + c) * T;
    for (long long t = threadIdx.x; t < T; t += blockDim.x) s += ld_elem(gy, base + t, f32);
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) db[c] = t;
  }
}

// ---------------------------------------------------------------- SnakeBeta backward + reductions
// y = x + inv_b * sin(a x)^2  (blocks.py:301-302), a = exp(alpha), inv_b = 1/(exp(beta) + 1e-9):
//   dy/dx     = 1 + inv_b * a * sin(2 a x)
//   dy/dalpha = inv_b * a * x * sin(2 a x)            (logscale; without it drop the factor a)
//   dy/dbeta  = -inv_b^2 * exp(beta) * sin(a x)^2     (logscale; without it drop exp(beta))
// The per-channel factors are applied once per block to the partial sums.
struct SnakeBwdParams {
  const float* dA;        // [rows, C] gradient w.r.t. the activated tensor (fp32)
  const float* x;         // [rows, C] pre-activation stream saved by the forward pass (nullptr with a == nullptr)
  const float* a;         // SnakeBeta exp(alpha) [C]; nullptr: identity (G = dA + skip)
  const float* inv_b;
  int logscale;
  const float* skip;      // [rows, C] gradient arriving through the ResidualUnit skip connection or nullptr
  float* G;               // [rows, C] fp32 out or nullptr
  __nv_bfloat16* Gb;      // [rows, C] bf16 out or nullptr
  float* d_alpha;         // [C] accumulated (atomicAdd) or nullptr
  float* d_beta;
  float* d_bias;          // [C] column sums of G (bias gradient of the conv that produced x) or nullptr
  long long rows;
  int C;
  int CW;                 // channels per block column (power of two <= 256)
  int rows_per_block;
  int fast;               // 1: MUFU sin/cos (bf16 mode); 0: sincosf (fp32 mode, <= 1e-5 budget)
  // bf16 mode, vectorised kernels only: the data-gradient conv hands dA over as bf16 (its fragment-mapped epilogue,
  // half the bytes), and the skip-connection gradient is read from the bf16 copy Gb of the later step -- the fp32
  // copy of that gradient then has no reader and is not written at all.
  int dA_bf16;            // dA points to bf16
  int skip_bf16;          // skip points to bf16
  int x_f16;              // x points to fp16 (training plans with the fp16 stream); vectorised kernels only
};

__global__ void __launch_bounds__(256) snake_bwd_kernel(const SnakeBwdParams p) {
  __shared__ float red[3][256];
  const int CW = p.CW;
  const int rl = threadIdx.x / CW;          // row lane
  const int nrl = 256 / CW;
  const int c = blockIdx.y * CW + (threadIdx.x % CW);
  const long long r0 = static_cast<long long>(blockIdx.x) * p.rows_per_block;
  const long long r1 = min(r0 + p.rows_per_block, p.rows);
  float s1 = 0.f, s2 = 0.f, sb = 0.f;
  if (c < p.C) {
    float a = 0.f, ib = 0.f;
    if (p.a) { a = p.a[c]; ib = p.inv_b[c]; }
    for (long long r = r0 + rl; r < r1; r += nrl) {
      const size_t i = static_cast<size_t>(r) * p.C + c;
      float g = p.dA[i];
      if (p.a) {
        const float xv = p.x[i];
        float sn, cs;
        sincosf(a * xv, &sn, &cs);
        const float s2x = 2.f * sn * cs;          // sin(2 a x)
        s1 = fmaf(g * xv, s2x, s1);
        s2 = fmaf(g, sn * sn, s2);
        g = g * fmaf(ib * a, s2x, 1.f);
      }
      if (p.skip) g += p.skip[i];
      sb += g;
      if (p.G) p.G[i] = g;
      if (p.Gb) p.Gb[i] = __float2bfloat16(g);
    }
  }
  red[0][threadIdx.x] = s1;
  red[1][threadIdx.x] = s2;
  red[2][threadIdx.x] = sb;
  __syncthreads();
  if (threadIdx.x < CW && c < p.C) {
    float t1 = 0.f, t2 = 0.f, tb = 0.f;
    for (int j = 0; j < nrl; ++j) {
      t1 += red[0][threadIdx.x + j * CW];
      t2 += red[1][threadIdx.x + j * CW];
      tb += red[2][threadIdx.x + j * CW];
    }
    if (p.a && p.d_alpha) {
      const float a = p.a[c], ib = p.inv_b[c];
      const float eb = 1.f / ib - 1e-9f;          // exp(beta)
      atomicAdd(p.d_alpha + c, t1 * ib * (p.logscale ? a : 1.f));
      atomicAdd(p.d_beta + c, -t2 * ib * ib * (p.logscale ? eb : 1.f));
    }
    if (p.d_bias) atomicAdd(p.d_bias + c, tb);
  }
}

// Vectorised form for C % 4 == 0: a thread owns 4 consecutive channels (float4 loads, 8-byte bf16 stores) and
// walks rows; CW here counts float4 columns per block (power of two <= 256).  Same sums, same outputs.
template <bool kFast>
__device__ __forceinline__ void snake_bwd_elem(float& g, float xv, float a, float ib, float& s1, float& s2) {
  float sn, cs;
  if (kFast) { sn = __sinf(a * xv); cs = __cosf(a * xv); } else { sincosf(a * xv, &sn, &cs); }
  const float s2x = 2.f * sn * cs;
  s1 = fmaf(g * xv, s2x, s1);
  s2 = fmaf(g, sn * sn, s2);
  g = g * fmaf(ib * a, s2x, 1.f);
}

template <bool kFast>
__global__ void __launch_bounds__(256) snake_bwd_vec4_kernel(const SnakeBwdParams p) {
  __shared__ float4 red[3][256];
  const int CW = p.CW;                      // float4 columns handled by this block
  const int rl = threadIdx.x / CW;
  const int nrl = 256 / CW;
  const int c4 = blockIdx.y * CW + (threadIdx.x % CW);
  const int C4 = p.C >> 2;
  const long long r0 = static_cast<long long>(blockIdx.x) * p.rows_per_block;
  const long long r1 = min(r0 + p.rows_per_block, p.rows);
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1, sb = s1;
  float4 a = s1, ib = s1;
  if (c4 < C4) {
    if (p.a) {
      a = __ldg(reinterpret_cast<const float4*>(p.a) + c4);
      ib = __ldg(reinterpret_cast<const float4*>(p.inv_b) + c4);
    }
    const float4* dA = reinterpret_cast<const float4*>(p.dA);
    const float4* X = reinterpret_cast<const float4*>(p.x);
    const float4* SK = reinterpret_cast<const float4*>(p.skip);
    float4* G = reinterpret_cast<float4*>(p.G);
    uint2* Gb = reinterpret_cast<uint2*>(p.Gb);
    auto ld_bf16x4 = [](const void* base, size_t i) {
      const uint2 q = __ldcs(reinterpret_cast<const uint2*>(base) + i);
      const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.x));
      const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.y));
      return make_float4(lo.x, lo.y, hi.x, hi.y);
    };
#pragma unroll 2
    for (long long r = r0 + rl; r < r1; r += nrl) {
      const size_t i = static_cast<size_t>(r) * C4 + c4;
      float4 g = p.dA_bf16 ? ld_bf16x4(p.dA, i) : __ldcs(dA + i);
      if (p.a) {
        float4 xv;
        if (p.x_f16) {
          const uint2 q = __ldcs(reinterpret_cast<const uint2*>(p.x) + i);
          const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&q.x));
          const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&q.y));
          xv = make_float4(lo.x, lo.y, hi.x, hi.y);
        } else {
          xv = __ldcs(X + i);
        }
        snake_bwd_elem<kFast>(g.x, xv.x, a.x, ib.x, s1.x, s2.x);
        snake_bwd_elem<kFast>(g.y, xv.y, a.y, ib.y, s1.y, s2.y);
        snake_bwd_elem<kFast>(g.z, xv.z, a.z, ib.z, s1.z, s2.z);
        snake_bwd_elem<kFast>(g.w, xv.w, a.w, ib.w, s1.w, s2.w);
      }
      if (SK) {
        const float4 k4 = p.skip_bf16 ? ld_bf16x4(p.skip, i) : __ldcs(SK + i);
        g.x += k4.x; g.y += k4.y; g.z += k4.z; g.w += k4.w;
      }
      sb.x += g.x; sb.y += g.y; sb.z += g.z; sb.w += g.w;
      if (G) G[i] = g;
      if (Gb) {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(g.x, g.y), h1 = __floats2bfloat162_rn(g.z, g.w);
        Gb[i] = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
      }
    }
  }
  red[0][threadIdx.x] = s1;
  red[1][threadIdx.x] = s2;
  red[2][threadIdx.x] = sb;
  __syncthreads();
  if (threadIdx.x < CW && c4 < C4) {
    float4 t1 = make_float4(0.f, 0.f, 0.f, 0.f), t2 = t1, tb = t1;
    for (int j = 0; j < nrl; ++j) {
      const float4 u1 = red[0][threadIdx.x + j * CW], u2 = red[1][threadIdx.x + j * CW], ub = red[2][threadIdx.x + j * CW];
      t1.x += u1.x; t1.y += u1.y; t1.z += u1.z; t1.w += u1.w;
      t2.x += u2.x; t2.y += u2.y; t2.z += u2.z; t2.w += u2.w;
      tb.x += ub.x; tb.y += ub.y; tb.z += ub.z; tb.w += ub.w;
    }
    const int c = c4 * 4;
    if (p.a && p.d_alpha) {
      const float av[4] = {a.x, a.y, a.z, a.w}, iv[4] = {ib.x, ib.y, ib.z, ib.w};
      const float v1[4] = {t1.x, t1.y, t1.z, t1.w}, v2[4] = {t2.x, t2.y, t2.z, t2.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float eb = 1.f / iv[e] - 1e-9f;
        atomicAdd(p.d_alpha + c + e, v1[e] * iv[e] * (p.logscale ? av[e] : 1.f));
        atomicAdd(p.d_beta + c + e, -v2[e] * iv[e] * iv[e] * (p.logscale ? eb : 1.f));
      }
    }
    if (p.d_bias) {
      atomicAdd(p.d_bias + c, tb.x); atomicAdd(p.d_bias + c + 1, tb.y);
      atomicAdd(p.d_bias + c + 2, tb.z); atomicAdd(p.d_bias + c + 3, tb.w);
    }
  }
}

// ---------------------------------------------------------------- SnakeBeta backward, HBM-streaming form
// Same arithmetic and outputs as snake_bwd_vec4_kernel.  That kernel keeps one or two rows per thread in flight and is
// bound by memory LATENCY, not bytes (ncu, profiles/r02_snake_bwd_vec4_before.txt: 23 % of DRAM peak, 22 stalled warps
// per issue on long_scoreboard), so halving its bytes (bf16 dA / skip) did not shorten it.  Here a producer thread
// streams [R rows x CW4 float4-columns] tiles of the 2-3 input tensors into a 4-stage shared-memory ring with bulk
// async copies (mbarrier full / empty) -- ~100 KB per SM in flight whatever the compute warps are doing -- and 16
// compute warps read the tiles from shared memory and write G / Gb straight to global memory (a warp's 32 threads
// write one contiguous row segment).  Persistent CTAs; per-channel sums stay in registers across all tiles of a CTA.
constexpr int kSbsStages = 4;
constexpr int kSbsCompute = 512;                   // compute threads (warp 16 = producer)
constexpr int kSbsThreads = kSbsCompute + 32;
constexpr int kSbsTileVec = 1024;                  // float4 vectors per tile and tensor (16 KB fp32 / 8 KB bf16)

struct SnakeBwdStreamGeom {
  int CW4;              // float4 columns per tile (power of two, <= 512, divides 512)
  int ncol;             // column blocks (C4 / CW4)
  int R;                // rows per tile (kSbsTileVec / CW4)
  long long row_tiles;  // ceil(rows / R)
};

inline size_t snake_bwd_stream_smem() { return 1024 + static_cast<size_t>(kSbsStages) * 3 * kSbsTileVec * 16 + 3 * kSbsCompute * 16; }

template <bool kFast>
__global__ void __launch_bounds__(kSbsThreads, 1) snake_bwd_stream_kernel(const SnakeBwdParams p, const SnakeBwdStreamGeom gm) {
  extern __shared__ uint8_t sbs_raw[];
  const uint32_t raw_addr = ptx::smem_u32(sbs_raw);
  uint8_t* smem = sbs_raw + (((raw_addr + 127u) & ~127u) - raw_addr);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + kSbsStages;
  uint8_t* ring = smem + 128;
  float4* red = reinterpret_cast<float4*>(ring + static_cast<size_t>(kSbsStages) * 3 * kSbsTileVec * 16);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C4 = p.C >> 2;
  const long long total = gm.row_tiles * gm.ncol;
  const int cb = blockIdx.x % gm.ncol;                   // this CTA's column block (fixed: grid is a multiple of ncol)
  const long long t_first = blockIdx.x / gm.ncol, t_step = gridDim.x / gm.ncol;
  const bool has_a = p.a != nullptr, has_sk = p.skip != nullptr;
  const int esz_dA = p.dA_bf16 ? 8 : 16, esz_sk = p.skip_bf16 ? 8 : 16, esz_x = p.x_f16 ? 8 : 16;   // bytes per 4 channels
  if (threadIdx.x == 0) {
    for (int i = 0; i < kSbsStages; ++i) { ptx::mbar_init(&full[i], 1); ptx::mbar_init(&empty[i], kSbsCompute / 32); }
    ptx::fence_mbar_init();
  }
  __syncthreads();
  (void)total;
  if (warp == kSbsCompute / 32) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (long long rt = t_first; rt < gm.row_tiles; rt += t_step) {
        const long long r0 = rt * gm.R;
        const int nr = static_cast<int>(min(static_cast<long long>(gm.R), p.rows - r0));
        ptx::mbar_wait(&empty[s], ph ^ 1u);
        uint8_t* st = ring + static_cast<size_t>(s) * 3 * kSbsTileVec * 16;
        const uint32_t bytes = static_cast<uint32_t>(nr) * gm.CW4 * (esz_dA + (has_a ? esz_x : 0) + (has_sk ? esz_sk : 0));
        ptx::mbar_expect_tx(&full[s], bytes);
        const size_t e0 = static_cast<size_t>(r0) * C4 + static_cast<size_t>(cb) * gm.CW4;     // first float4 index
        if (gm.ncol == 1) {                                // whole rows: one contiguous range per tensor
          const uint32_t nv = static_cast<uint32_t>(nr) * gm.CW4;
          ptx::bulk_load_1d(st, reinterpret_cast<const uint8_t*>(p.dA) + e0 * esz_dA, nv * esz_dA, &full[s]);
          if (has_a) ptx::bulk_load_1d(st + kSbsTileVec * 16, reinterpret_cast<const uint8_t*>(p.x) + e0 * esz_x, nv * esz_x, &full[s]);
          if (has_sk) ptx::bulk_load_1d(st + 2 * kSbsTileVec * 16, reinterpret_cast<const uint8_t*>(p.skip) + e0 * esz_sk, nv * esz_sk, &full[s]);
        } else {
          for (int r = 0; r < nr; ++r) {
            const size_t e = e0 + static_cast<size_t>(r) * C4;
            ptx::bulk_load_1d(st + static_cast<size_t>(r) * gm.CW4 * esz_dA, reinterpret_cast<const uint8_t*>(p.dA) + e * esz_dA,
                              gm.CW4 * esz_dA, &full[s]);
            if (has_a) ptx::bulk_load_1d(st + kSbsTileVec * 16 + static_cast<size_t>(r) * gm.CW4 * esz_x,
                                         reinterpret_cast<const uint8_t*>(p.x) + e * esz_x, gm.CW4 * esz_x, &full[s]);
            if (has_sk) ptx::bulk_load_1d(st + 2 * kSbsTileVec * 16 + static_cast<size_t>(r) * gm.CW4 * esz_sk,
                                          reinterpret_cast<const uint8_t*>(p.skip) + e * esz_sk, gm.CW4 * esz_sk, &full[s]);
          }
        }
        if (++s == kSbsStages) { s = 0; ph ^= 1u; }
      }
    }
    return;
  }
  // ------------------------------------------------------------ compute warps
  const int c4l = threadIdx.x % gm.CW4;                 // column inside the tile (CW4 <= 512 divides 512)
  const int rl = threadIdx.x / gm.CW4, nrl = kSbsCompute / gm.CW4;
  const int c4 = cb * gm.CW4 + c4l;
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1, sb = s1, a = s1, ib = s1;
  if (has_a) {
    a = __ldg(reinterpret_cast<const float4*>(p.a) + c4);
    ib = __ldg(reinterpret_cast<const float4*>(p.inv_b) + c4);
  }
  float4* G = reinterpret_cast<float4*>(p.G);
  uint2* Gb = reinterpret_cast<uint2*>(p.Gb);
  auto bf4 = [](uint2 q) {
    const float2 lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.x));
    const float2 hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&q.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
  };
  int s = 0;
  uint32_t ph = 0;
  for (long long rt = t_first; rt < gm.row_tiles; rt += t_step) {
    const long long r0 = rt * gm.R;
    const int nr = static_cast<int>(min(static_cast<long long>(gm.R), p.rows - r0));
    ptx::mbar_wait(&full[s], ph);
    const uint8_t* st = ring + static_cast<size_t>(s) * 3 * kSbsTileVec * 16;
#pragma unroll 2
    for (int r = rl; r < nr; r += nrl) {
      const int v = r * gm.CW4 + c4l;
      float4 g = p.dA_bf16 ? bf4(reinterpret_cast<const uint2*>(st)[v]) : reinterpret_cast<const float4*>(st)[v];
      if (has_a) {
        float4 xv;
        if (p.x_f16) {
          const uint2 q = reinterpret_cast<const uint2*>(st + kSbsTileVec * 16)[v];
          const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&q.x));
          const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&q.y));
          xv = make_float4(lo.x, lo.y, hi.x, hi.y);
        } else {
          xv = reinterpret_cast<const float4*>(st + kSbsTileVec * 16)[v];
        }
        snake_bwd_elem<kFast>(g.x, xv.x, a.x, ib.x, s1.x, s2.x);
        snake_bwd_elem<kFast>(g.y, xv.y, a.y, ib.y, s1.y, s2.y);
        snake_bwd_elem<kFast>(g.z, xv.z, a.z, ib.z, s1.z, s2.z);
        snake_bwd_elem<kFast>(g.w, xv.w, a.w, ib.w, s1.w, s2.w);
      }
      if (has_sk) {
        const float4 k4 = p.skip_bf16 ? bf4(reinterpret_cast<const uint2*>(st + 2 * kSbsTileVec * 16)[v])
                                      : reinterpret_cast<const float4*>(st + 2 * kSbsTileVec * 16)[v];
        g.x += k4.x; g.y += k4.y; g.z += k4.z; g.w += k4.w;
      }
      sb.x += g.x; sb.y += g.y; sb.z += g.z; sb.w += g.w;
      const size_t i = static_cast<size_t>(r0 + r) * C4 + c4;
      if (G) __stcs(G + i, g);
      if (Gb) {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(g.x, g.y), h1 = __floats2bfloat162_rn(g.z, g.w);
        __stcs(Gb + i, make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1)));
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&empty[s]);
    if (++s == kSbsStages) { s = 0; ph ^= 1u; }
  }
  // per-channel sums: reduce over the row lanes of this CTA, then one atomic per channel and CTA
  red[threadIdx.x] = s1;
  red[kSbsCompute + threadIdx.x] = s2;
  red[2 * kSbsCompute + threadIdx.x] = sb;
  ptx::named_bar_sync(1, kSbsCompute);
  if (threadIdx.x < gm.CW4) {
    float4 t1 = make_float4(0.f, 0.f, 0.f, 0.f), t2 = t1, tb = t1;
    for (int j = 0; j < nrl; ++j) {
      const float4 u1 = red[threadIdx.x + j * gm.CW4], u2 = red[kSbsCompute + threadIdx.x + j * gm.CW4],
                   ub = red[2 * kSbsCompute + threadIdx.x + j * gm.CW4];
      t1.x += u1.x; t1.y += u1.y; t1.z += u1.z; t1.w += u1.w;
      t2.x += u2.x; t2.y += u2.y; t2.z += u2.z; t2.w += u2.w;
      tb.x += ub.x; tb.y += ub.y; tb.z += ub.z; tb.w += ub.w;
    }
    const int c = c4 * 4;
    if (has_a && p.d_alpha) {
      const float av[4] = {a.x, a.y, a.z, a.w}, iv[4] = {ib.x, ib.y, ib.z, ib.w};
      const float v1[4] = {t1.x, t1.y, t1.z, t1.w}, v2[4] = {t2.x, t2.y, t2.z, t2.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float eb = 1.f / iv[e] - 1e-9f;
        atomicAdd(p.d_alpha + c + e, v1[e] * iv[e] * (p.logscale ? av[e] : 1.f));
        atomicAdd(p.d_beta + c + e, -v2[e] * iv[e] * iv[e] * (p.logscale ? eb : 1.f));
      }
    }
    if (p.d_bias) {
      atomicAdd(p.d_bias + c, tb.x); atomicAdd(p.d_bias + c + 1, tb.y);
      atomicAdd(p.d_bias + c + 2, tb.z); atomicAdd(p.d_bias + c + 3, tb.w);
    }
  }
}

// geometry of the streaming form, or false when the shape needs the plain kernels (C4 not a power of two / multiple of 512)
inline bool snake_bwd_stream_geom(const SnakeBwdParams& p, SnakeBwdStreamGeom& g) {
  if (p.C % 8) return false;
  const int C4 = p.C / 4;
  int cw = C4;
  if (C4 > 512) { if (C4 % 512) return false; cw = 512; }
  if (cw & (cw - 1)) return false;
  if (cw < 8) return false;
  if (p.rows < 4096) return false;                       // tiny tensors: the plain kernel's many small blocks do better
  g.CW4 = cw;
  g.ncol = C4 / cw;
  g.R = kSbsTileVec / cw;
  g.row_tiles = (p.rows + g.R - 1) / g.R;
  // 16-byte alignment of every bulk copy: bf16 rows of CW4 * 8 bytes, pointers from the workspace (1 KB aligned)
  return true;
}

// ---------------------------------------------------------------- weight gradient of the waveform-edge convs
// Conv1d(k, stride 1) between a wide tensor (C channels, channels-last fp32) and a thin one (NT <= 2 channels):
//   out[c][j][k] = sum_{b,t} W[b, t + sigma*(k*dil - pad), c] * N[b, t, j]
// sigma = +1: decoder tail (wide = SnakeBeta(stream) = conv input, thin = output gradient)  -> dW[j][c][k]
// sigma = -1: encoder head (wide = output gradient, thin = the waveform = conv input)        -> dW[c][j][k]
// HBM-bound (the wide tensor is read once); thread = channel, 7 x NT accumulators in registers, the thin rows a
// block needs are staged in shared memory.  grid (nblocks), block 256 = (256 / C) row lanes x C channels.
struct EdgeWgradParams {
  const float* W;            // [B, T, C] fp32 (fp16 with W_f16: the saved stream of a training plan)
  int W_f16;
  const float* W_a;          // SnakeBeta prologue on W (nullptr: none)
  const float* W_inv_b;
  const void* N;             // thin tensor, element strides below
  int N_f32;
  long long N_sB, N_sT, N_sC;
  float* dW;                 // torch layout; out_wide_first = 1: [C][NT][K], 0: [NT][C][K]
  int out_wide_first;
  int sigma;
  int B, T, C, K, dil, pad;
  int rows_per_block;        // rows of one clip per block (blocks never straddle clips)
  int blocks_per_clip;
  int fast_sin;              // bf16-mode plans: MUFU sine in the SnakeBeta prologue, as the forward pass computed it
};

constexpr int kEdgeMaxK = 8;

template <int NT>
__global__ void __launch_bounds__(256) wgrad_edge_kernel(const EdgeWgradParams p) {
  extern __shared__ float thin[];            // [rows_per_block + 2*halo][NT]
  const int b = blockIdx.x / p.blocks_per_clip;
  const int t0 = (blockIdx.x % p.blocks_per_clip) * p.rows_per_block;
  const int t1 = min(t0 + p.rows_per_block, p.T);
  const int halo = max(p.pad, (p.K - 1) * p.dil - p.pad);
  const int nthin = (t1 - t0) + 2 * halo;
  for (int i = threadIdx.x; i < nthin * NT; i += 256) {
    const int r = i / NT, j = i % NT;
    const int t = t0 - halo + r;
    thin[i] = (t >= 0 && t < p.T) ? ld_elem(p.N, static_cast<size_t>(b * p.N_sB + t * p.N_sT + j * p.N_sC), p.N_f32) : 0.f;
  }
  __syncthreads();
  const int lanes = 256 / p.C;               // row lanes (C <= 256, power of two)
  const int c = threadIdx.x % p.C, rl = threadIdx.x / p.C;
  float acc[kEdgeMaxK][NT];
#pragma unroll
  for (int k = 0; k < kEdgeMaxK; ++k)
#pragma unroll
    for (int j = 0; j < NT; ++j) acc[k][j] = 0.f;
  float a = 0.f, ib = 0.f;
  if (p.W_a) { a = p.W_a[c]; ib = p.W_inv_b[c]; }
  // wide row u pairs with thin row t = u - sigma*(k*dil - pad); four rows per iteration so that four
  // independent 512-byte row loads are in flight per warp (one load per iteration was latency-bound)
  if (rl < lanes) {
    const int u_lo = max(0, t0 - halo), u_hi = min(p.T, t1 + halo);
    const float* Wc = p.W + static_cast<size_t>(b) * p.T * p.C + c;
    for (int u0 = u_lo + rl; u0 < u_hi; u0 += 4 * lanes) {
      float w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int u = u0 + q * lanes;
        w[q] = (u < u_hi) ? __ldcs(Wc + static_cast<size_t>(u) * p.C) : 0.f;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int u = u0 + q * lanes;
        if (u >= u_hi) break;
        float wv = w[q];
        if (p.W_a) wv = snake_beta<false>(wv, a, ib);
#pragma unroll
        for (int k = 0; k < kEdgeMaxK; ++k) {
          if (k < p.K) {
            const int t = u - p.sigma * (k * p.dil - p.pad);
            if (t >= t0 && t < t1) {
#pragma unroll
              for (int j = 0; j < NT; ++j) acc[k][j] = fmaf(wv, thin[(t - t0 + halo) * NT + j], acc[k][j]);
            }
          }
        }
      }
    }
  }
  __syncthreads();
  // reduce over row lanes through shared memory (re-using the thin buffer is not safe in size: use atomics per lane)
#pragma unroll
  for (int k = 0; k < kEdgeMaxK; ++k) {
    if (k < p.K) {
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        float v = acc[k][j];
        if (rl < lanes && v != 0.f) {
          const size_t o = p.out_wide_first ? (static_cast<size_t>(c) * NT + j) * p.K + k
                                            : (static_cast<size_t>(j) * p.C + c) * p.K + k;
          atomicAdd(p.dW + o, v);
        }
      }
    }
  }
}

// Vectorised form (C % 4 == 0, C / 4 a power of two <= 256): a thread owns FOUR consecutive channels, so a warp reads
// whole 512-byte rows with 16-byte loads (four rows in flight per thread), and the row lanes of a block are reduced
// through shared memory before ONE atomic per weight and block.  The scalar kernel above issued 4-byte loads
// (128 bytes per warp request), kept ~4 KB per block in flight and sent every lane's partial sums to the same 1 792
// addresses: 0.8 ms per launch for 453 MB (0.57 TB/s; profiles/r02_train_step_launches.txt).
template <int NT>
__global__ void __launch_bounds__(256, 2) wgrad_edge_vec4_kernel(const EdgeWgradParams p) {
  extern __shared__ float thin[];            // [rows_per_block + 2*halo][NT], then the reduction scratch
  const int b = blockIdx.x / p.blocks_per_clip;
  const int t0 = (blockIdx.x % p.blocks_per_clip) * p.rows_per_block;
  const int t1 = min(t0 + p.rows_per_block, p.T);
  const int halo = max(p.pad, (p.K - 1) * p.dil - p.pad);
  const int nthin = (t1 - t0) + 2 * halo;
  for (int i = threadIdx.x; i < nthin * NT; i += 256) {
    const int r = i / NT, j = i % NT;
    const int t = t0 - halo + r;
    thin[i] = (t >= 0 && t < p.T) ? ld_elem(p.N, static_cast<size_t>(b * p.N_sB + t * p.N_sT + j * p.N_sC), p.N_f32) : 0.f;
  }
  __syncthreads();
  const int C4 = p.C >> 2;
  const int lanes = 256 / C4;
  const int c4 = threadIdx.x % C4, rl = threadIdx.x / C4;
  float acc[kEdgeMaxK][NT][4];
#pragma unroll
  for (int k = 0; k < kEdgeMaxK; ++k)
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[k][j][e] = 0.f;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f), ib = a;
  if (p.W_a) {
    a = __ldg(reinterpret_cast<const float4*>(p.W_a) + c4);
    ib = __ldg(reinterpret_cast<const float4*>(p.W_inv_b) + c4);
  }
  const int u_lo = max(0, t0 - halo), u_hi = min(p.T, t1 + halo);
  const float4* Wc = reinterpret_cast<const float4*>(p.W + static_cast<size_t>(b) * p.T * p.C) + c4;
  const uint2* Wh = reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(p.W) + static_cast<size_t>(b) * p.T * p.C) + c4;
  for (int u0 = u_lo + rl; u0 < u_hi; u0 += 4 * lanes) {
    float4 w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int u = u0 + q * lanes;
      if (u >= u_hi) { w[q] = make_float4(0.f, 0.f, 0.f, 0.f); continue; }
      if (p.W_f16) {
        const uint2 hq = __ldcs(Wh + static_cast<size_t>(u) * C4);
        const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&hq.x));
        const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&hq.y));
        w[q] = make_float4(lo.x, lo.y, hi.x, hi.y);
      } else {
        w[q] = __ldcs(Wc + static_cast<size_t>(u) * C4);
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int u = u0 + q * lanes;
      if (u >= u_hi) break;
      float wv[4] = {w[q].x, w[q].y, w[q].z, w[q].w};
      if (p.W_a) {
        if (p.fast_sin) {
          wv[0] = snake_beta<true>(wv[0], a.x, ib.x); wv[1] = snake_beta<true>(wv[1], a.y, ib.y);
          wv[2] = snake_beta<true>(wv[2], a.z, ib.z); wv[3] = snake_beta<true>(wv[3], a.w, ib.w);
        } else {
          wv[0] = snake_beta<false>(wv[0], a.x, ib.x); wv[1] = snake_beta<false>(wv[1], a.y, ib.y);
          wv[2] = snake_beta<false>(wv[2], a.z, ib.z); wv[3] = snake_beta<false>(wv[3], a.w, ib.w);
        }
      }
#pragma unroll
      for (int k = 0; k < kEdgeMaxK; ++k) {
        if (k < p.K) {
          const int t = u - p.sigma * (k * p.dil - p.pad);
          if (t >= t0 && t < t1) {
#pragma unroll
            for (int j = 0; j < NT; ++j) {
              const float tv = thin[(t - t0 + halo) * NT + j];
#pragma unroll
              for (int e = 0; e < 4; ++e) acc[k][j][e] = fmaf(wv[e], tv, acc[k][j][e]);
            }
          }
        }
      }
    }
  }
  // reduce the row lanes through shared memory, one tap at a time: scratch [lanes][C4][NT * 4]
  float* red = thin + ((nthin * NT + 3) & ~3);
#pragma unroll
  for (int k = 0; k < kEdgeMaxK; ++k) {
    if (k < p.K) {
      __syncthreads();
#pragma unroll
      for (int j = 0; j < NT; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e) red[(rl * C4 + c4) * (NT * 4) + j * 4 + e] = acc[k][j][e];
      __syncthreads();
      for (int i = threadIdx.x; i < C4 * NT * 4; i += 256) {
        float v = 0.f;
        for (int l = 0; l < lanes; ++l) v += red[l * C4 * NT * 4 + i];
        const int cc = (i / (NT * 4)) * 4 + (i & 3), j = (i >> 2) % NT;
        if (v != 0.f) {
          const size_t o = p.out_wide_first ? (static_cast<size_t>(cc) * NT + j) * p.K + k
                                            : (static_cast<size_t>(j) * p.C + cc) * p.K + k;
          atomicAdd(p.dW + o, v);
        }
      }
    }
  }
}

// ---------------------------------------------------------------- data gradient of the decoder tail
// Conv1d(C -> NT <= 2, k, stride 1): dA[b, u, c] = sum_{k,j} w[k][c][j] * gy[b, u - (k*dil - pad), j].
// The wide side is the output here (HBM-bound write of [B, T, C] fp32); thread = channel with its k x NT weights
// in registers, the thin gradient rows of a block staged in shared memory.  Same grid as wgrad_edge_kernel.
struct EdgeDgradParams {
  const float* gy;           // [B, T, NT] fp32 channels-last
  const float* w;            // [K][C][NT] fp32 (forward CUDA-core packing)
  float* dA;                 // [B, T, C] fp32
  int B, T, C, K, dil, pad;
  int rows_per_block, blocks_per_clip;
};

template <int NT>
__global__ void __launch_bounds__(256) dgrad_edge_kernel(const EdgeDgradParams p) {
  extern __shared__ float thin[];            // [rows_per_block + 2*halo][NT]
  const int b = blockIdx.x / p.blocks_per_clip;
  const int t0 = (blockIdx.x % p.blocks_per_clip) * p.rows_per_block;
  const int t1 = min(t0 + p.rows_per_block, p.T);
  const int halo = max(p.pad, (p.K - 1) * p.dil - p.pad);
  const int nthin = (t1 - t0) + 2 * halo;
  for (int i = threadIdx.x; i < nthin * NT; i += 256) {
    const int t = t0 - halo + i / NT;
    thin[i] = (t >= 0 && t < p.T) ? p.gy[(static_cast<size_t>(b) * p.T + t) * NT + i % NT] : 0.f;
  }
  __syncthreads();
  const int lanes = 256 / p.C;
  const int c = threadIdx.x % p.C, rl = threadIdx.x / p.C;
  if (rl >= lanes) return;
  float w[kEdgeMaxK][NT];
#pragma unroll
  for (int k = 0; k < kEdgeMaxK; ++k)
#pragma unroll
    for (int j = 0; j < NT; ++j) w[k][j] = (k < p.K) ? __ldg(p.w + (static_cast<size_t>(k) * p.C + c) * NT + j) : 0.f;
  float* out = p.dA + static_cast<size_t>(b) * p.T * p.C + c;
  for (int u = t0 + rl; u < t1; u += lanes) {
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < kEdgeMaxK; ++k) {
      if (k < p.K) {
        const int r = u - (k * p.dil - p.pad) - t0 + halo;     // staged thin row (zero outside the clip)
#pragma unroll
        for (int j = 0; j < NT; ++j) v = fmaf(w[k][j], thin[r * NT + j], v);
      }
    }
    __stcs(out + static_cast<size_t>(u) * p.C, v);
  }
}

// ---------------------------------------------------------------- weight gradient, CUDA cores
// dW[cd][cs][k] += sum_{b,t} D[b, t, cd] * S[b, t*stride + k*dil - pad, cs]
//   Conv1d:          D = dY [B, T_out, Cout], S = a [B, T_in, Cin]   -> dW[Cout][Cin][K]  (torch layout)
//   ConvTranspose1d: D = a  [B, T_in, Cin],   S = dY [B, T_out, Cout] -> dW[Cin][Cout][K] (torch layout)
// where a = SnakeBeta(x) is either the bf16 operand the forward pass saved or recomputed from the fp32
// stream on load.  grid (ceil(Cd/64) * ceil(Cs/64), K, nsplit), block 256; each block reduces a slice of
// the B*Td rows into a 64x64 tile (4x4 per thread) and adds it with atomics.
struct WgradParams {
  const void* D;
  int D_f32;
  long long D_sB, D_sT, D_sC;   // element strides (so the API layout [B, C, T] can be read in place)
  const float* D_a;             // SnakeBeta prologue on D (nullptr: none)
  const float* D_inv_b;
  const void* S;
  int S_f32;
  long long S_sB, S_sT, S_sC;
  const float* S_a;
  const float* S_inv_b;
  float* dW;                    // [Cd][Cs][K]
  int B, Td, Ts, Cd, Cs, K, stride, dil, pad;
  long long rows_per_split;     // of the B*Td rows
};

constexpr int kWgRows = 16;

__global__ void __launch_bounds__(256) wgrad_direct_kernel(const WgradParams p) {
  __shared__ float sd[kWgRows][64 + 1];
  __shared__ float ss[kWgRows][64 + 1];
  const int n_cs = (p.Cs + 63) / 64;
  const int cd0 = (blockIdx.x / n_cs) * 64, cs0 = (blockIdx.x % n_cs) * 64;
  const int k = blockIdx.y;
  const long long rows = static_cast<long long>(p.B) * p.Td;
  const long long r_begin = static_cast<long long>(blockIdx.z) * p.rows_per_split;
  const long long r_end = min(r_begin + p.rows_per_split, rows);
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;   // tx -> cs, ty -> cd
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (long long r0 = r_begin; r0 < r_end; r0 += kWgRows) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < kWgRows * 64; idx += 256) {
      // walk the contiguous dimension fastest: channels for channels-last tensors, time for the API layout
      int rr, cc;
      if (p.D_sC == 1) { rr = idx / 64; cc = idx % 64; } else { rr = idx % kWgRows; cc = idx / kWgRows; }
      const long long r = r0 + rr;
      float v = 0.f;
      if (r < r_end && cd0 + cc < p.Cd) {
        const long long b = r / p.Td, t = r % p.Td;
        v = ld_elem(p.D, static_cast<size_t>(b * p.D_sB + t * p.D_sT + (cd0 + cc) * p.D_sC), p.D_f32);
        if (p.D_a) v = snake_beta<false>(v, p.D_a[cd0 + cc], p.D_inv_b[cd0 + cc]);
      }
      sd[rr][cc] = v;
      if (p.S_sC == 1) { rr = idx / 64; cc = idx % 64; } else { rr = idx % kWgRows; cc = idx / kWgRows; }
      const long long r2 = r0 + rr;
      v = 0.f;
      if (r2 < r_end && cs0 + cc < p.Cs) {
        const long long b = r2 / p.Td, t = r2 % p.Td;
        const long long u = t * p.stride + static_cast<long long>(k) * p.dil - p.pad;
        if (u >= 0 && u < p.Ts) {
          v = ld_elem(p.S, static_cast<size_t>(b * p.S_sB + u * p.S_sT + (cs0 + cc) * p.S_sC), p.S_f32);
          if (p.S_a) v = snake_beta<false>(v, p.S_a[cs0 + cc], p.S_inv_b[cs0 + cc]);
        }
      }
      ss[rr][cc] = v;
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < kWgRows; ++rr) {
      float dv[4], sv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) dv[i] = sd[rr][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) sv[j] = ss[rr][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], sv[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cd = cd0 + ty * 4 + i;
    if (cd >= p.Cd) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cs = cs0 + tx * 4 + j;
      if (cs < p.Cs) atomicAdd(p.dW + (static_cast<size_t>(cd) * p.Cs + cs) * p.K + k, acc[i][j]);
    }
  }
}

// ---------------------------------------------------------------- weight norm backward
// w[i,:] = v[i,:] * g[i] / n_i,  n_i = ||v[i,:]||:
//   dg[i] = <dw_i, v_i> / n_i ;  dv_i = (g_i / n_i) * (dw_i - v_i * <dw_i, v_i> / n_i^2)
// One block per row i.  dw and dv may alias (in place).
__device__ __forceinline__ void weight_norm_bwd_row(float (*red)[32], const float* v, const float* g, const float* dw,
                                                    float* dv, float* dg, int inner, int row) {
  const size_t base = static_cast<size_t>(row) * inner;
  float nn = 0.f, dot = 0.f;
  for (int i = threadIdx.x; i < inner; i += blockDim.x) {
    const float x = v[base + i];
    nn = fmaf(x, x, nn);
    dot = fmaf(dw[base + i], x, dot);
  }
  for (int o = 16; o > 0; o >>= 1) {
    nn += __shfl_xor_sync(0xffffffffu, nn, o);
    dot += __shfl_xor_sync(0xffffffffu, dot, o);
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = nn; red[1][threadIdx.x >> 5] = dot; }
  __syncthreads();
  if (threadIdx.x < 32) {
    float a = (threadIdx.x < (blockDim.x >> 5)) ? red[0][threadIdx.x] : 0.f;
    float b = (threadIdx.x < (blockDim.x >> 5)) ? red[1][threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (threadIdx.x == 0) { red[0][0] = a; red[1][0] = b; }
  }
  __syncthreads();
  nn = red[0][0];
  dot = red[1][0];
  const float n = sqrtf(nn);
  const float gi = g[row];
  const float s = gi / n, q = dot / nn;
  for (int i = threadIdx.x; i < inner; i += blockDim.x) dv[base + i] = s * (dw[base + i] - v[base + i] * q);
  if (threadIdx.x == 0) dg[row] = dot / n;
}
__global__ void weight_norm_bwd_kernel(const float* v, const float* g, const float* dw, float* dv, float* dg,
                                       int inner) {
  __shared__ float red[2][32];
  weight_norm_bwd_row(red, v, g, dw, dv, dg, inner, blockIdx.x);
}

// Same, with dw in the packed layout [K][R][Cc] the tensor-core weight-gradient kernel accumulates into
// (v, dv in the torch layout [R][Cc][K]).  g == nullptr: no weight norm, dv = dw re-ordered.
__device__ __forceinline__ void weight_norm_bwd_packed_row(float (*red)[32], const float* v, const float* g,
                                                           const float* dwp, float* dv, float* dg, int R, int Cc, int K,
                                                           int i) {
  const int inner = Cc * K;
  const size_t base = static_cast<size_t>(i) * inner;
  // walk the packed layout in its own order (c fastest) for coalesced reads of dw
  float nn = 0.f, dot = 0.f;
  if (g) {
    // (k, c) of j = k Cc + c advance by the block size without a division per element
    const int dk1 = blockDim.x / Cc, dc1 = blockDim.x % Cc;
    int k = threadIdx.x / Cc, c = threadIdx.x % Cc;
    for (int j = threadIdx.x; j < inner; j += blockDim.x) {
      const float x = v[base + static_cast<size_t>(c) * K + k];
      nn = fmaf(x, x, nn);
      dot = fmaf(dwp[(static_cast<size_t>(k) * R + i) * Cc + c], x, dot);
      k += dk1; c += dc1;
      if (c >= Cc) { c -= Cc; ++k; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      nn += __shfl_xor_sync(0xffffffffu, nn, o);
      dot += __shfl_xor_sync(0xffffffffu, dot, o);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = nn; red[1][threadIdx.x >> 5] = dot; }
    __syncthreads();
    if (threadIdx.x < 32) {
      float a = (threadIdx.x < (blockDim.x >> 5)) ? red[0][threadIdx.x] : 0.f;
      float b = (threadIdx.x < (blockDim.x >> 5)) ? red[1][threadIdx.x] : 0.f;
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
      }
      if (threadIdx.x == 0) { red[0][0] = a; red[1][0] = b; }
    }
    __syncthreads();
    nn = red[0][0];
    dot = red[1][0];
  }
  const float n = g ? sqrtf(nn) : 1.f;
  const float s = g ? g[i] / n : 1.f, q = g ? dot / nn : 0.f;
  const int dc2 = blockDim.x / K, dk2 = blockDim.x % K;
  int c2 = threadIdx.x / K, k2 = threadIdx.x % K;
  for (int j = threadIdx.x; j < inner; j += blockDim.x) {     // torch order (j = c K + k) for coalesced writes of dv
    const float d = dwp[(static_cast<size_t>(k2) * R + i) * Cc + c2];
    dv[base + j] = g ? s * (d - v[base + j] * q) : d;
    c2 += dc2; k2 += dk2;
    if (k2 >= K) { k2 -= K; ++c2; }
  }
  if (g && threadIdx.x == 0) dg[i] = dot / n;
}

// One layer (kvae_conv1d_win_bwd): one block per dim-0 row, 256 threads.
__global__ void __launch_bounds__(256) weight_norm_bwd_packed_kernel(const float* v, const float* g, const float* dwp,
                                                                     float* dv, float* dg, int R, int Cc, int K) {
  __shared__ float red[2][32];
  weight_norm_bwd_packed_row(red, v, g, dwp, dv, dg, R, Cc, K, blockIdx.x);
}

// All layers of a plan in ONE launch (72 launches of ~16 us each before): grid = sum of dim-0 rows, a block finds its
// layer by binary search in the prefix table.  params == nullptr: packed gradients are only re-ordered.
struct WnBwdDesc {
  long long off_v, off_g, off_dwp;    // floats; off_dwp < 0: dW sits in the weight_v slot of grads (in place)
  int R, Cc, K, row0;
};
__global__ void __launch_bounds__(256)
weight_norm_bwd_all_kernel(const float* params, float* grads, const float* dwp, const WnBwdDesc* d, int n_layers) {
  __shared__ float red[2][32];
  int lo = 0, hi = n_layers - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (d[mid].row0 <= static_cast<int>(blockIdx.x)) lo = mid; else hi = mid - 1; }
  const WnBwdDesc L = d[lo];
  const int row = blockIdx.x - L.row0;
  if (L.off_dwp >= 0)
    weight_norm_bwd_packed_row(red, params ? params + L.off_v : nullptr, params ? params + L.off_g : nullptr, dwp + L.off_dwp,
                               grads + L.off_v, grads + L.off_g, L.R, L.Cc, L.K, row);
  else if (params)
    weight_norm_bwd_row(red, params + L.off_v, params + L.off_g, grads + L.off_v, grads + L.off_v, grads + L.off_g,
                        L.Cc * L.K, row);
}

// ---------------------------------------------------------------- vae_sample backward (bottleneck.py:51-62)
// latents = noise*scale + mean ; kl = (mean^2 + var - log var - 1).sum(1).mean(), stdev = softplus(scale)+1e-4.
//   d mean  = gz + gkl * 2 mean / (B*T)
//   d scale = gz * noise + gkl * (2 stdev - 2/stdev) * sigmoid(scale) / (B*T)
__global__ void vae_sample_bwd_kernel(const void* mean, const void* scale, const void* noise, const void* gz,
                                      const float* gkl, float inv_bt, void* gmean, void* gscale, size_t n, int f32) {
  const float gk = gkl ? (*gkl) * inv_bt : 0.f;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float m = ld_elem(mean, i, f32), sc = ld_elem(scale, i, f32);
    const float g = gz ? ld_elem(gz, i, f32) : 0.f;
    const float sp = (sc > 20.f) ? sc : log1pf(expf(sc));
    const float stdev = sp + 1e-4f;
    const float sig = 1.f / (1.f + expf(-sc));
    st_elem(gmean, i, f32, g + gk * 2.f * m);
    st_elem(gscale, i, f32, g * ld_elem(noise, i, f32) + gk * (2.f * stdev - 2.f / stdev) * sig);
  }
}

// ---------------------------------------------------------------- sigma-VAE Gaussian NLL
// nll = sum_i [ 0.5 ((x_i - xhat_i)/sigma)^2 + log sigma + 0.5 log(2 pi) ] / B ; d nll / d xhat = (xhat - x)/(sigma^2 B)
// (no in-tree definition in the reference: SURVEY.md section 8c).  partial: per-block double sums.
__global__ void gaussian_nll_kernel(const void* x, const void* xhat, size_t n, int f32, float inv_var, float inv_b,
                                    void* gxhat, double* partial) {
  __shared__ double red[32];
  double acc = 0.0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float d = ld_elem(xhat, i, f32) - ld_elem(x, i, f32);
    acc += static_cast<double>(d * d);
    if (gxhat) st_elem(gxhat, i, f32, d * inv_var * inv_b);
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.0;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) partial[blockIdx.x] = t;
  }
}
__global__ void gaussian_nll_finish_kernel(const double* partial, int nblocks, double n, double inv_var, double log_sigma,
                                           double inv_b, float* loss) {
  __shared__ double red[32];
  double acc = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += blockDim.x) acc += partial[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (blockDim.x >> 5); ++i) t += red[i];
    *loss = static_cast<float>((0.5 * inv_var * t + n * (log_sigma + 0.9189385332046727)) * inv_b);
  }
}

// ---------------------------------------------------------------- AdamW over a flat fp32 buffer
// torch.optim.AdamW semantics (decoupled weight decay, bias-corrected moments); grad is scaled first
// (1/world_size after a summing all-reduce).
__global__ void adamw_kernel(float* p, const float* g, float* m, float* v, size_t n, float lr, float b1, float b2,
                             float eps, float wd, float bc1, float bc2_sqrt, float grad_scale) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * grad_scale;
    float pi = p[i];
    pi -= lr * wd * pi;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

}  // namespace kvae
