// wgrad_umma: weight gradient of Conv1d / ConvTranspose1d on the tcgen05 tensor cores.
//
//   dW[k][cd][cs] += sum_{b,t} D[b, t, cd] * S[b, t*stride + k*dil - pad, cs]
//     Conv1d:          D = dY (bf16 copy of the stream gradient), S = a = SnakeBeta(x) (saved bf16 operand)
//     ConvTranspose1d: D = a,                                     S = dY
// (autograd of F.conv1d / F.conv_transpose1d in the reference, autoencoders.py:49-53,76,98.)
//
// The contraction runs over TIME, which is the slow dimension of the channels-last tensors -- so both
// operands are fed to the MMA in **MN-major** form: a TMA box {64 channels, R rows} with SWIZZLE_128B is
// already the canonical MN-major SW128 image (one 128-byte line per time row = 64 channels; 8 rows per
// swizzle atom, SBO = 1024 B between atoms along K; LBO = distance between the two 64-channel halves of a
// 128-wide tile).  No transpose is ever materialised.  A tap is a row shift of the S slab, addressed through
// the descriptor start address exactly as in the forward kernel (conv_umma2.cuh), so one staged slab serves
// every tap of its input phase.
//
// Tile: 128 (cd) x 128 (cs) x up to 4 taps per CTA = 4 accumulators of 128 TMEM columns.  The B*Td rows are
// split over gridDim.y CTAs per tile (split-K); CTAs of the same split run side by side (tile index is the
// fast grid dimension), so the D / S rows they share come from L2.  Partial sums are added to a packed fp32
// buffer [K][Cd][Cs] with vector reductions (red.global.add.v4.f32); the weight-norm backward reads that
// layout directly (train.cuh::weight_norm_bwd_packed_row).
//
// Warp roles (256 threads): warp 0 TMA producer, warp 1 UMMA issuer, warp 2 TMEM allocator, warps 4-7 epilogue.
#pragma once
#include <cuda_bf16.h>
#include <cstdint>

#include "ptx.cuh"

namespace kvae {

constexpr int kWgMaxTaps = 4;    // taps (accumulators) per CTA
constexpr int kWgMaxGroups = 8;  // tap groups per layer (K <= 32)

struct WgradUmmaParams {
  int B, Td, Cd, Cs, K;
  int R;                         // dense rows per pipeline stage (multiple of 16)
  int NS;                        // pipeline stages
  int chunks_per_clip;           // ceil(Td / R)
  int n_cd, n_cs, n_groups;      // tiles; blockIdx.x = (group * n_cd + cd_tile) * n_cs + cs_tile
  int items_per_split;           // chunks (over B * chunks_per_clip) per gridDim.y slice
  // per tap group
  int g_ntaps[kWgMaxGroups];
  int g_nslabs[kWgMaxGroups];
  int g_k[kWgMaxGroups][kWgMaxTaps];       // kernel index of each tap
  int g_slab[kWgMaxGroups][kWgMaxTaps];    // which staged S slab the tap reads
  int g_shift[kWgMaxGroups][kWgMaxTaps];   // row shift inside that slab
  int s_phase[kWgMaxGroups][kWgMaxTaps];   // per slab: input phase of the strided tensor
  int s_row0[kWgMaxGroups][kWgMaxTaps];    // per slab: first row relative to the chunk's first dense row
  int RS;                        // rows per S slab box (R + largest shift span, multiple of 8)
  float* dWp;                    // packed [K][Cd][Cs] fp32
};

__host__ __device__ inline size_t wgrad_umma_stage_bytes(int R, int RS, int nslabs) {
  return static_cast<size_t>(2) * R * 128 + static_cast<size_t>(nslabs) * 2 * RS * 128;
}

__global__ void __launch_bounds__(256, 1)
wgrad_umma_kernel(const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmS,
                  const __grid_constant__ WgradUmmaParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + 8;
  uint64_t* acc_full = full + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full + 17);
  uint8_t* ring = smem + 1024;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  const int cs_t = tile % p.n_cs;
  const int cd_t = (tile / p.n_cs) % p.n_cd;
  const int grp = tile / (p.n_cs * p.n_cd);
  const int ntaps = p.g_ntaps[grp];
  const int nslabs = p.g_nslabs[grp];
  const int cd0 = cd_t * 128, cs0 = cs_t * 128;
  const uint32_t d_half = static_cast<uint32_t>(p.R) * 128;       // one 64-channel half of the D slab
  const uint32_t s_half = static_cast<uint32_t>(p.RS) * 128;
  const uint32_t stage_bytes = 2 * d_half + static_cast<uint32_t>(nslabs) * 2 * s_half;
  const long long total_items = static_cast<long long>(p.B) * p.chunks_per_clip;
  const long long it0 = static_cast<long long>(blockIdx.y) * p.items_per_split;
  const long long it1 = min(it0 + p.items_per_split, total_items);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmD);
    ptx::prefetch_tmap(&tmS);
    for (int i = 0; i < p.NS; ++i) { ptx::mbar_init(&full[i], 1); ptx::mbar_init(&empty[i], 1); }
    ptx::mbar_init(acc_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // (warp-uniform loop, one elected lane issues: the loop state stays in uniform registers -- conv_umma2.cuh)
    {
      int st = 0;
      uint32_t ph = 0;
      for (long long it = it0; it < it1; ++it) {
        const int b = __shfl_sync(0xffffffffu, static_cast<int>(it / p.chunks_per_clip), 0);
        const int r0 = __shfl_sync(0xffffffffu, static_cast<int>(it % p.chunks_per_clip) * p.R, 0);
        ptx::mbar_wait(&empty[st], ph ^ 1u);
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(&full[st], stage_bytes);
          uint8_t* dst = ring + static_cast<size_t>(st) * stage_bytes;
          ptx::tma_load_4d(dst, &tmD, &full[st], cd0, 0, r0, b);
          ptx::tma_load_4d(dst + d_half, &tmD, &full[st], cd0 + 64, 0, r0, b);
          dst += 2 * d_half;
          for (int s = 0; s < nslabs; ++s) {
            const int row = r0 + p.s_row0[grp][s];
            ptx::tma_load_4d(dst, &tmS, &full[st], cs0, p.s_phase[grp][s], row, b);
            ptx::tma_load_4d(dst + s_half, &tmS, &full[st], cs0 + 64, p.s_phase[grp][s], row, b);
            dst += 2 * s_half;
          }
        }
        __syncwarp();
        if (++st == p.NS) { st = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ UMMA issuer
    {   // warp-uniform loop, one elected lane issues
      const uint32_t idesc = ptx::idesc_bf16_f32_mn(128, 128);
      // MN-major SW128 descriptors: LBO = distance between 64-channel halves, SBO = 1024 B (8 time rows)
      const uint64_t hi_common = (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      const uint64_t d_hi = hi_common | (static_cast<uint64_t>(d_half >> 4) << 16);
      const uint64_t s_hi = hi_common | (static_cast<uint64_t>(s_half >> 4) << 16);
      const uint32_t ring_lo = (ptx::smem_u32(ring) & 0x3FFFFu) >> 4;
      const int ksteps = p.R / 16;
      // lane t holds tap t's (slab offset + shift rows) >> 4, relative to the stage's S area; read back by shuffle
      const int tl = lane < ntaps ? lane : 0;
      const uint32_t my_tap_off = (static_cast<uint32_t>(p.g_slab[grp][tl]) * 2 * s_half + static_cast<uint32_t>(p.g_shift[grp][tl]) * 128) >> 4;
      uint32_t toff[kWgMaxTaps];
#pragma unroll
      for (int t = 0; t < kWgMaxTaps; ++t) toff[t] = __shfl_sync(0xffffffffu, my_tap_off, t);
      int st = 0;
      uint32_t ph = 0, accum = 0;
      for (long long it = it0; it < it1; ++it) {
        ptx::mbar_wait(&full[st], ph);
        ptx::tc_fence_after();
        const uint32_t d_lo = ring_lo + ((static_cast<uint32_t>(st) * stage_bytes) >> 4);
        const uint32_t s_lo = d_lo + ((2 * d_half) >> 4);
        if (ptx::elect_one()) {
          for (int j = 0; j < ksteps; ++j) {
            const uint32_t koff = static_cast<uint32_t>(j) * (2048 >> 4);       // 16 time rows
#pragma unroll
            for (int t = 0; t < kWgMaxTaps; ++t)
              if (t < ntaps)
                ptx::umma_f16(tmem_base + t * 128, d_hi | ((d_lo + koff) & 0x3FFFu), s_hi | ((s_lo + toff[t] + koff) & 0x3FFFu),
                              idesc, (j | static_cast<int>(accum)) ? 1u : 0u);
          }
          ptx::umma_commit(&empty[st]);
        }
        __syncwarp();
        accum = 1u;
        if (++st == p.NS) { st = 0; ph ^= 1u; }
      }
      if (ptx::elect_one()) ptx::umma_commit(acc_full);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue: accumulators -> packed dW (reductions)
    const int quad = warp & 3;
    const int cd = cd0 + quad * 32 + lane;
    if (it1 > it0) {
      ptx::mbar_wait(acc_full, 0);
      ptx::tc_fence_after();
      for (int t = 0; t < ntaps; ++t) {
        const int k = p.g_k[grp][t];
        float* row = p.dWp + (static_cast<size_t>(k) * p.Cd + cd) * p.Cs + cs0;
#pragma unroll 1
        for (int cb = 0; cb < 4; ++cb) {
          uint32_t r[32];
          __syncwarp();
          ptx::tmem_ld_32x32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + t * 128 + cb * 32, r);
          ptx::tmem_ld_wait();
          if (cd < p.Cd) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              if (cs0 + cb * 32 + j < p.Cs)
                ptx::red_add_v4(row + cb * 32 + j, __uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
          }
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}

}  // namespace kvae
