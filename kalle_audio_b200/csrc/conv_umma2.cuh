// conv_umma2: persistent, double-buffered version of the tcgen05 implicit-GEMM convolution.
//
// Implicit-GEMM 1-D convolution on the sm_100a tensor cores (tcgen05.mma, TMEM accumulators, TMA-fed operands).  One
// kernel serves the three weight-normalised convolution shapes of the Oobleck stack (reference:
// stable_audio_tools/models/autoencoders.py:39-114): Conv1d stride 1 dilation d, Conv1d stride s kernel 2s, and
// ConvTranspose1d stride s (polyphase).  Activations are channels-last [B, T, C] bf16, so a tap shift is a whole
// 128-byte-row offset of a K-major operand tile; weights are pre-packed [tap][Cout][Cin] bf16.  GEMM view per tile:
// D[M, N] += A[time rows, 64 ch] * W[out-channels, 64 ch]^T summed over (64-channel chunk) x (tap); taps that read the
// same input phase share one staged A slab (conv_common.cuh, Tap).  The schedule:
//   * one CTA per SM loops over output tiles (static round-robin), so operand loads of tile i+1 are
//     in flight while tile i is still being multiplied / written out;
//   * the accumulator lives in TMEM twice (2 x MT*NT columns) when that fits in 512 columns: the UMMA
//     issuer starts tile i+1 as soon as its operands land while the epilogue drains tile i;
//   * three instantiations.  <0>: 8 epilogue warps (two warpgroups, each covering the 128 TMEM lanes), every warp its own
//     little pipeline over 32-row x 32-channel blocks with no block-level barrier -- the generic epilogue (fp32
//     streams, bf16x3 split, channels-first output, time-on-M tiles).  <1> / <2>: 16 epilogue warps (four per TMEM lane
//     quadrant) on 16-row x 32-channel items with a specialised fragment-mapped epilogue -- <1> the forward launches
//     in the swap orientation with 2-byte stream / operand blocks (every tensor-core conv of an inference plan and of
//     the training forward), <2> the data-gradient launches with the fused SnakeBeta backward;
//   * in every epilogue one elected lane prefetches the item's ResidualUnit skip block with a TMA load one item
//     ahead, every lane adds its part, writes the result IN PLACE into the same swizzled shared-memory block
//     (conflict-free) plus the SnakeBeta-activated bf16 block, and the elected lane hands both to TMA stores; the
//     bulk-group mechanism recycles the blocks.  Every HBM access is a full line and no thread waits on a store.
//
// Warp roles (384 threads in <0>, 640 in <1> / <2>): warp 0 weight TMA producer, warp 1 UMMA issuer, warp 2 TMEM
// allocator, warp 3 activation-slab TMA producer, warps 4.. epilogue.  Producers and issuer run WARP-UNIFORM loops with
// an elected lane doing the issue (loop state in uniform registers).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "conv_common.cuh"
#include "ptx.cuh"

namespace kvae {

struct ConvParams2 {
  int B, Tq_out, P_out, Cout;
  int n_chunks;
  int MT, NT;
  int RB, nbox;
  int SA, SB;
  int swap;                // 1: out-channels on the MMA M side (TMEM lanes), time on the N side (see kernel)
  int acc_stages;          // 1 or 2 accumulator buffers in TMEM
  int tmem_cols;           // power of two >= acc_stages*MT*NT
  int q_tiles, n_tiles, total_tiles;
  int tap_begin[kMaxPhases + 1];
  // taps packed one word each so the single-thread producer / UMMA issue loops stay short:
  //   tap_mma[t]: bits 0-15 (row shift * 128 B) >> 4, bit 16 first tap of a slab, bit 17 last tap of a slab
  //   tap_ld[t] : bits 0-7 input phase, bits 8-15 weight slab, bits 16-31 slab start row (signed)
  uint32_t tap_mma[kMaxTaps];
  uint32_t tap_ld[kMaxTaps];
  // epilogue
  const float* bias;
  const float* residual;   // fp32 channels-last [B, T_out, Cout] or nullptr
  int raw_mode;            // 0 none, 1 channels-last stream via TMA (tmR), 2 channels-first direct store
  int raw_f16;             // 1: the residual stream (raw_mode 1 output and the skip-connection input) is fp16 in HBM
                           //    (fp32 in registers and TMEM); 0: fp32.  Inference plans use fp16: it halves the
                           //    stream traffic of the HBM-bound 128-channel stages for +4e-5 of the 1e-3 budget
  void* out_cf;            // raw_mode 2: [B, Cout, T_out]
  long long cf_ld;         // raw_mode 2: elements between channel rows of out_cf (0: T_out)
  int out_cf_f32;
  int act_mode;            // 0 none, 1 bf16 channels-last via TMA (tmO)
  int fast;                // 1: conv_umma2_kernel<1> -- 16 epilogue warps on 16-row x 32-channel items (forward, swap orientation,
                           //    2-byte stream / operand blocks only; see the kFast branch of the kernel);
                           // 2: conv_umma2_kernel<2> -- the same epilogue with the fused SnakeBeta backward (bwd below)
  int split3;              // fp32-mode arithmetic on the tensor cores: both operands are stored as bf16 (hi | lo)
                           // halves -- activations [.., 2*Cin], weights [tap][Cout][2*Cin] -- and every K chunk is
                           // multiplied three times: hi*hi + lo*hi + hi*lo (the lo*lo term is below fp32 rounding).
                           // The kernel just sees 3x the chunks, with different operand columns per chunk.
  int Cin;                 // input channels (split3: column of the lo halves)
  int act_split;           // 1: the bf16 operand output is written as (hi | lo) halves, lo at channel Cout + c
  int precise;             // 1: SnakeBeta with sinf (fp32 mode), 0: MUFU sin
  const float* snake_a;    // SnakeBeta folded into the activated output (nullptr: plain cast)
  const float* snake_inv_b;
  // raw_mode 2 only: the sigma-VAE sample fused into the encoder's last conv (model_sigmaVAE.py:187-213 'fix' on the
  // mean half of the latents, twj-style chunk(2, dim=1)): for channels c < samp_D,
  //   samp_out[b, c, t] = mean + samp_std * samp_noise[b, c, t], two separately rounded operations on the value AS STORED
  // (rounded to the output dtype first), i.e. bit-identical to torch on the stored latents.  Same dtype as out_cf.
  // Training backward, data-gradient launches (conv_umma2_kernel<2> only): the SnakeBeta derivative and the
  // skip-connection add of the layer BEFORE this conv are applied to the accumulator in the epilogue,
  //   G = dA * (1 + a * inv_b * sin(2 a x)) + skip        (dA = this conv's output, x = that layer's saved fp16 stream)
  // G leaves as bf16 through the operand path (act_mode 1), and the per-channel sums d alpha, d beta and the bias
  // gradient of the producing conv (column sums of G) accumulate in registers and go out with one atomic per channel,
  // warp and tile.  Replaces a separate HBM pass over dA, x, skip and G (snake_bwd_stream_kernel).
  int bwd;                 // 1: this mode; tmX maps x (fp16), tmR maps skip (bf16) when bwd_skip
  int bwd_skip;
  int bwd_logscale;
  const float* bwd_a;      // exp(alpha) / 1/(exp(beta)+1e-9) of that SnakeBeta
  const float* bwd_inv_b;
  float* d_alpha;          // [Cout] accumulated
  float* d_beta;
  float* d_bias;           // [Cout] accumulated or nullptr
  const void* samp_noise;  // [B, samp_D, T_out] or nullptr
  void* samp_out;          // [B, samp_D, T_out]
  int samp_D;
  float samp_std;
};

__device__ __forceinline__ void fused_sigma_sample(const ConvParams2& p, int b, int c, size_t t_out, int T_out, float v) {
  if (p.samp_noise && c < p.samp_D) {
    const size_t o = (static_cast<size_t>(b) * p.samp_D + c) * T_out + t_out;
    if (p.out_cf_f32) {
      const float n = static_cast<const float*>(p.samp_noise)[o];
      static_cast<float*>(p.samp_out)[o] = __fadd_rn(v, __fmul_rn(p.samp_std, n));
    } else {
      const float m = __bfloat162float(__float2bfloat16(v));
      const float n = __bfloat162float(static_cast<const __nv_bfloat16*>(p.samp_noise)[o]);
      const float t = __bfloat162float(__float2bfloat16(__fmul_rn(p.samp_std, n)));
      static_cast<__nv_bfloat16*>(p.samp_out)[o] = __float2bfloat16(__fadd_rn(m, t));
    }
  }
}

constexpr int kRawBlkBytes = 32 * 128;   // 32 rows x 32 fp32, SWIZZLE_128B
constexpr int kActBlkBytes = 32 * 64;    // 32 rows x 32 bf16 (or fp16 stream), SWIZZLE_64B
constexpr int kFastBlk = 16 * 64;        // conv_umma2_kernel<1>: 16 rows x 32 bf16 / fp16, SWIZZLE_64B
__host__ __device__ inline int conv_umma2_raw_blk(int raw_f16) { return raw_f16 ? kActBlkBytes : kRawBlkBytes; }
// per-epilogue-warp staging: a ring of fp32 blocks (3 deep when the skip connection is prefetched into
// it, else 2) and two bf16 blocks; only what a layer needs is carved out
__host__ __device__ inline int conv_umma2_raw_slots(int raw_mode, bool residual) {
  return (raw_mode == 1 || residual) ? (residual ? 3 : 2) : 0;
}
__host__ __device__ inline int conv_umma2_stage_bytes_per_warp(int raw_mode, int act_mode, bool residual, int raw_f16,
                                                               int act_split = 0, int bwd = 0, int fast = 0) {
  if (bwd) return 2 * (2 * kFastBlk) + 2 * kFastBlk;            // <2>: two slots of [x block | skip block], two bf16 output blocks
  if (fast) return conv_umma2_raw_slots(raw_mode, residual) * kFastBlk + (act_mode == 1 ? 2 * kFastBlk : 0);
  return conv_umma2_raw_slots(raw_mode, residual) * conv_umma2_raw_blk(raw_f16) +
         (act_mode == 1 ? 2 * kActBlkBytes * (act_split ? 2 : 1) : 0);
}

__host__ __device__ inline size_t conv_umma2_smem_bytes(const ConvParams2& p) {
  return 1024 + 1024 + static_cast<size_t>(p.SA) * p.nbox * p.RB * 128 + static_cast<size_t>(p.SB) * p.NT * 128 +
         (p.fast ? 16 : 8) * conv_umma2_stage_bytes_per_warp(p.raw_mode, p.act_mode, p.residual != nullptr, p.raw_f16,
                                                             p.act_split, p.bwd, p.fast);
}

template <int kFast>
__global__ void __launch_bounds__(kFast ? 640 : 384, 1)
conv_umma2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                  const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmO,
                  const __grid_constant__ CUtensorMap tmX, const __grid_constant__ ConvParams2 p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* a_empty = a_full + 8;
  uint64_t* b_full = a_full + 16;
  uint64_t* b_empty = a_full + 32;
  uint64_t* t_full = a_full + 48;    // [2] accumulator ready
  uint64_t* t_empty = a_full + 50;   // [2] accumulator drained (8 epilogue warps arrive)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 52);
  uint64_t* res_full = a_full + 56;  // [8 or 16 warps][3 slots] skip-connection block landed
  uint8_t* a_ring = smem + 1024;
  const uint32_t a_bytes = static_cast<uint32_t>(p.nbox) * p.RB * 128;
  const uint32_t b_bytes = static_cast<uint32_t>(p.NT) * 128;
  uint8_t* b_ring = a_ring + static_cast<size_t>(p.SA) * a_bytes;
  uint8_t* stage_base = b_ring + static_cast<size_t>(p.SB) * b_bytes;

  const int warp = ptx::warp_idx();
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW);
    if (p.raw_mode == 1 || p.bwd_skip) ptx::prefetch_tmap(&tmR);
    if (p.act_mode == 1) ptx::prefetch_tmap(&tmO);
    for (int i = 0; i < p.SA; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < p.SB; ++i) { ptx::mbar_init(&b_full[i], 1); ptx::mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&t_full[i], 1); ptx::mbar_init(&t_empty[i], kFast ? 16 : 8); }
    for (int i = 0; i < (kFast ? 48 : 24); ++i) ptx::mbar_init(&res_full[i], 1);
    if (p.residual || p.bwd) ptx::prefetch_tmap(&tmX);
    ptx::fence_mbar_init();
  }
  ptx::pdl_launch_dependents();
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  ptx::pdl_wait();                 // everything above overlapped the previous kernel's tail; its outputs are visible from here
  const uint32_t tmem_base = *tmem_slot;
  // Two operand assignments.  swap = 0: M = 128 time rows (x MT sub-tiles), N = NT out-channels.
  // swap = 1 (NT == 128): M = 128 out-channels, N = 128*MT time rows.  With N = 256 one instruction does the
  // work of two, and per 128 cycles the tensor core reads 4 KB (weights) + 8 KB (activations) of shared
  // memory instead of 2 x (4 + 4) KB -- at M = N = 128 the operand reads alone saturate the 128 B/cycle
  // shared-memory port, which capped the C = 128 layers at ~55 % tensor utilisation.
  const int acc_cols = p.swap ? 128 * p.MT : p.MT * p.NT;

  // tile id -> (batch, q tile, output phase, n tile); n fastest so CTAs sharing an A slab run together
  auto decode = [&](int tile, int& b, int& q0, int& phi, int& n0) {
    n0 = (tile % p.n_tiles) * p.NT;
    int r = tile / p.n_tiles;
    phi = r % p.P_out;
    r /= p.P_out;
    q0 = (r % p.q_tiles) * (128 * p.MT);
    b = r / p.q_tiles;
  };

  // Two TMA producer threads.  In ONE FIFO with the weight slabs an activation slab was requested only SB weight
  // stages (about a microsecond) before its first MMA -- less than an HBM round trip -- although its ring stage had
  // been free for much longer; on its own thread a slab is requested the moment its stage is released.
  if (warp == 0 || warp == 3) {
    // (warp-uniform loops, one elected lane issues -- see the UMMA issuer below)
    {
      const bool do_a = warp == 3;
      const bool do_w = warp == 0;
      const int SA = p.SA, SB = p.SB, nbox = p.nbox, RB = p.RB;
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        int b, q0, phi, n0;
        decode(tile, b, q0, phi, n0);
        const int t_lo = p.tap_begin[phi], t_hi = p.tap_begin[phi + 1];
        const int n_vc = p.split3 ? 3 * p.n_chunks : p.n_chunks;
        for (int ch = 0; ch < n_vc; ++ch) {
          // operand columns of this (virtual) chunk: plain, or hi*hi / lo*hi / hi*lo of the bf16x3 split
          int a_col = ch * 64, w_col = ch * 64;
          if (p.split3) {
            const int c = ch % p.n_chunks, part = ch / p.n_chunks;
            a_col = c * 64 + (part == 1 ? p.Cin : 0);
            w_col = c * 64 + (part == 2 ? p.Cin : 0);
          }
          for (int t = t_lo; t < t_hi; ++t) {
            const uint32_t tl = p.tap_ld[t];
            if (do_a && (p.tap_mma[t] & 0x10000u)) {
              ptx::mbar_wait(&a_empty[as], aph ^ 1u);
              if (ptx::elect_one()) {
                ptx::mbar_expect_tx(&a_full[as], a_bytes);
                const int row = q0 + (static_cast<int32_t>(tl) >> 16);
                for (int bx = 0; bx < nbox; ++bx)
                  ptx::tma_load_4d(a_ring + static_cast<size_t>(as) * a_bytes + bx * RB * 128, &tmA, &a_full[as],
                                   a_col, tl & 0xff, row + bx * RB, b);
              }
              __syncwarp();
              if (++as == SA) { as = 0; aph ^= 1u; }
            }
            if (do_w) {
              ptx::mbar_wait(&b_empty[bs], bph ^ 1u);
              if (ptx::elect_one()) {
                ptx::mbar_expect_tx(&b_full[bs], b_bytes);
                ptx::tma_load_3d(b_ring + static_cast<size_t>(bs) * b_bytes, &tmW, &b_full[bs], w_col, n0,
                                 (tl >> 8) & 0xff);
              }
              __syncwarp();
              if (++bs == SB) { bs = 0; bph ^= 1u; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ UMMA issuer
    // The WHOLE warp walks the (tile, chunk, tap) loop and the barriers; one elected lane issues the MMAs and commits.
    // With the loop inside `if (elect_one())` (the first form) every loop variable lived in a vector register of a
    // divergent thread: 79 instructions per weight stage with an indexed constant load, six R2UR transfers and the
    // parameter block re-read each iteration -- ~540 cycles per stage of four MMAs, which 256-row tiles hide (512 tensor
    // cycles) but 128-row tiles do not: the batch-1 streaming layers ran their tensor pipe at 16 %
    // (profiles/r02_o12_b1_k7_c1024.ncu-rep).  Warp-uniform, the loop state sits in uniform registers next to the descriptors.
    {
      const uint32_t idesc = ptx::idesc_bf16_f32(128, p.NT);
      const uint32_t idesc_swap = ptx::idesc_bf16_f32(128, 128 * p.MT);
      const uint64_t desc_hi = (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      const uint32_t a_lo0 = ((ptx::smem_u32(a_ring) & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t b_lo0 = ((ptx::smem_u32(b_ring) & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t a_stage16 = a_bytes >> 4, b_stage16 = b_bytes >> 4;
      const bool two = (p.MT == 2);
      const bool swap = p.swap != 0;
      const int SA = p.SA, SB = p.SB, acc_stages = p.acc_stages;
      const int n_vc = p.split3 ? 3 * p.n_chunks : p.n_chunks;
      const uint32_t NT16 = p.NT;
      int as = 0, bs = 0, cur = 0, acc = 0;
      uint32_t aph = 0, bph = 0, accph = 0, cur_lo = a_lo0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int phi = (tile / p.n_tiles) % p.P_out;
        const int t_lo = p.tap_begin[phi], t_hi = p.tap_begin[phi + 1];
        ptx::mbar_wait(&t_empty[acc], accph ^ 1u);   // epilogue has drained this accumulator buffer
        ptx::tc_fence_after();
        const uint32_t d0 = tmem_base + acc * acc_cols;
        const uint32_t d1 = d0 + NT16;
        uint32_t accum = 0;                          // first MMA of a tile overwrites the accumulator
        for (int ch = 0; ch < n_vc; ++ch) {
          uint32_t tw = p.tap_mma[t_lo];
          for (int t = t_lo; t < t_hi; ++t) {
            const uint32_t tw_next = p.tap_mma[t + 1 < t_hi ? t + 1 : t_lo];   // fetched under this stage's MMAs
            if (tw & 0x10000u) {
              ptx::mbar_wait(&a_full[as], aph);
              cur = as;
              cur_lo = a_lo0 + as * a_stage16;
              if (++as == SA) { as = 0; aph ^= 1u; }
            }
            ptx::mbar_wait(&b_full[bs], bph);
            ptx::tc_fence_after();
            const uint32_t al = cur_lo + (tw & 0xffffu);
            const uint32_t bl = b_lo0 + bs * b_stage16;
            if (ptx::elect_one()) {
              if (swap) {
                ptx::umma_f16(d0, desc_hi | bl, desc_hi | al, idesc_swap, accum);
                ptx::umma_f16(d0, desc_hi | (bl + 2), desc_hi | (al + 2), idesc_swap, 1u);
                ptx::umma_f16(d0, desc_hi | (bl + 4), desc_hi | (al + 4), idesc_swap, 1u);
                ptx::umma_f16(d0, desc_hi | (bl + 6), desc_hi | (al + 6), idesc_swap, 1u);
              } else {
                ptx::umma_f16(d0, desc_hi | al, desc_hi | bl, idesc, accum);
                ptx::umma_f16(d0, desc_hi | (al + 2), desc_hi | (bl + 2), idesc, 1u);
                ptx::umma_f16(d0, desc_hi | (al + 4), desc_hi | (bl + 4), idesc, 1u);
                ptx::umma_f16(d0, desc_hi | (al + 6), desc_hi | (bl + 6), idesc, 1u);
                if (two) {
                  const uint32_t al1 = al + 1024;        // second 128-row sub-tile: +128 rows * 128 B >> 4
                  ptx::umma_f16(d1, desc_hi | al1, desc_hi | bl, idesc, accum);
                  ptx::umma_f16(d1, desc_hi | (al1 + 2), desc_hi | (bl + 2), idesc, 1u);
                  ptx::umma_f16(d1, desc_hi | (al1 + 4), desc_hi | (bl + 4), idesc, 1u);
                  ptx::umma_f16(d1, desc_hi | (al1 + 6), desc_hi | (bl + 6), idesc, 1u);
                }
              }
              ptx::umma_commit(&b_empty[bs]);
              if (tw & 0x20000u) ptx::umma_commit(&a_empty[cur]);
            }
            __syncwarp();
            accum = 1u;
            if (++bs == SB) { bs = 0; bph ^= 1u; }
            tw = tw_next;
          }
        }
        if (ptx::elect_one()) ptx::umma_commit(&t_full[acc]);
        __syncwarp();
        if (++acc == acc_stages) { acc = 0; accph ^= 1u; }
      }
    }
  } else if (warp >= 4 && kFast) {
    // ------------------------------------------------------------ epilogue, kFast: 16 warps (4 per TMEM lane quadrant) on
    // 16-row x 32-channel items -- the EPI2 mapping of conv_ru2.cuh.  The generic epilogue below spends ~860 warp
    // instructions per 32 x 32 item, most of them control (integer divisions for the prefetch coordinates, generic ->
    // shared address conversions, ring geometry recomputed per item, run-time mode branches) executed as one dependent
    // chain with two warps per scheduler (profiles/r02_k1_c256_before_after.txt: the k = 1 / transposed / strided convs ran at the
    // epilogue's item rate, 60 % of their HBM floor).  Here the tile decode happens once per tile, every address is a
    // loop-invariant 32-bit shared-memory offset, and four warps per scheduler hide each other's latencies.
    const int e = warp - 4, quad = warp & 3, sub = e >> 2;
    const int g8 = lane >> 2, rr = lane & 7, mj = lane >> 3;
    constexpr bool kBwd = (kFast == 2);   // fused SnakeBeta backward of the data-gradient launches (ConvParams2::bwd)
    const bool has_res = kBwd || p.residual != nullptr;
    const bool raw_out = !kBwd && p.raw_mode == 1, act_out = kBwd || p.act_mode == 1, has_snake = p.snake_a != nullptr;
    const int R = kBwd ? 2 : conv_umma2_raw_slots(p.raw_mode, has_res);
    const uint32_t slot_bytes = kBwd ? 2 * kFastBlk : kFastBlk;
    const uint32_t res_tx = (kBwd && p.bwd_skip) ? 2 * kFastBlk : kFastBlk;
    uint8_t* ring = stage_base + e * conv_umma2_stage_bytes_per_warp(p.raw_mode, p.act_mode, has_res, 1, 0, kBwd ? 1 : 0, 1);
    uint8_t* aring = ring + R * slot_bytes;
    const int brow = (mj >> 1) * 8 + rr;     // ldmatrix / stmatrix: this lane addresses row brow of a [16 x 64 B] block
    const uint32_t blk_lane = brow * 64 + (((mj & 1) ^ ((brow >> 1) & 3)) << 4);
    const uint32_t ring_lane = ptx::smem_u32(ring) + blk_lane;
    const uint32_t aring_lane = ring_lane + R * slot_bytes;
    uint64_t* my_res_full = res_full + e * 3;
    const int n_items = 8 * p.MT;            // 16-row items per quadrant and tile
    const uint32_t acc_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    auto dup = [](float f) { return ptx::f2_pack(f, f); };
    auto issue_skip = [&](int cb, int ph, int row, int bb, int slot) {   // lane 0 only
      ptx::mbar_expect_tx(&my_res_full[slot], res_tx);
      ptx::tma_load_4d(ring + slot * slot_bytes, &tmX, &my_res_full[slot], cb, ph, row, bb);
      if (kBwd && p.bwd_skip) ptx::tma_load_4d(ring + slot * slot_bytes + kFastBlk, &tmR, &my_res_full[slot], cb, ph, row, bb);
    };
    // decode() divides in the vector ALU; the lane-0 broadcast tells ptxas the results are warp-uniform, so the TMA
    // coordinates built from them sit in uniform registers instead of going through an R2UR waterfall loop per issue
    auto decode_u = [&](int t, int& ob, int& oq0, int& ophi, int& on0) {
      decode(t, ob, oq0, ophi, on0);
      ob = __shfl_sync(0xffffffffu, ob, 0);
      oq0 = __shfl_sync(0xffffffffu, oq0, 0);
      ophi = __shfl_sync(0xffffffffu, ophi, 0);
      on0 = __shfl_sync(0xffffffffu, on0, 0);
    };
    int tile = blockIdx.x;
    int b = 0, q0 = 0, phi = 0, n0 = 0;
    if (tile < p.total_tiles) decode_u(tile, b, q0, phi, n0);
    if (has_res && tile < p.total_tiles && ptx::elect_one()) issue_skip(n0 + quad * 32, phi, q0 + sub * 16, b, 0);
    int acc = 0, jr = 0, ja = 0;
    uint32_t accph = 0, res_ph = 0;
    float acc_da[4] = {0.f, 0.f, 0.f, 0.f}, acc_db[4] = {0.f, 0.f, 0.f, 0.f}, acc_bias[4] = {0.f, 0.f, 0.f, 0.f};
    for (; tile < p.total_tiles; tile += gridDim.x) {
      const int ntile = tile + gridDim.x;    // this CTA's next tile: its first skip block is prefetched during the last item
      int nb = 0, nq0 = 0, nphi = 0, nn0 = 0;
      if (ntile < p.total_tiles) decode_u(ntile, nb, nq0, nphi, nn0);
      const int cbase = n0 + quad * 32;
      uint64_t kb[4], ka[4], kib[4];         // index 2 * lane half + hi: channel cbase + 16 L + 8 hi + g8
      float bw_a[4], bw_ib[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ch = cbase + (i >> 1) * 16 + (i & 1) * 8 + g8;
        if constexpr (kBwd) {
          bw_a[i] = __ldg(p.bwd_a + ch);
          bw_ib[i] = __ldg(p.bwd_inv_b + ch);
        } else {
          kb[i] = p.bias ? dup(__ldg(p.bias + ch)) : 0ull;
          ka[i] = has_snake ? dup(__ldg(p.snake_a + ch)) : 0ull;
          kib[i] = has_snake ? dup(__ldg(p.snake_inv_b + ch)) : 0ull;
        }
      }
      ptx::mbar_wait_parked(&t_full[acc], accph);
      ptx::tc_fence_after();
      const uint32_t acc_tmem = acc_lane + acc * acc_cols;
#pragma unroll 1
      for (int item = sub; item < n_items; item += 4) {
        const int r0 = q0 + item * 16;
        const int sn = (jr + 1 == R) ? 0 : jr + 1;
        if (ptx::elect_one()) {
          // all but the newest store group have read their blocks: slot sn (last used two items ago) and the other
          // operand block are free; fetch the NEXT item's skip block
          ptx::bulk_wait_read<1>();
          if (has_res) {
            if (item + 4 < n_items) issue_skip(cbase, phi, r0 + 64, b, sn);
            else if (ntile < p.total_tiles) issue_skip(nn0 + quad * 32, nphi, nq0 + sub * 16, nb, sn);
          }
        }
        uint32_t r[16], sk[8];
        __syncwarp();
        const uint32_t t2 = acc_tmem + item * 16;
        ptx::tmem_ld_16x256b_x2(t2, r);
        ptx::tmem_ld_16x256b_x2(t2 + (16u << 16), r + 8);
        const uint32_t rb = ring_lane + jr * slot_bytes;
        if (has_res) {
          ptx::mbar_wait_parked(&my_res_full[jr], (res_ph >> jr) & 1u);
          res_ph ^= (1u << jr);
          ptx::ldmatrix_x4_trans(rb, sk[0], sk[1], sk[2], sk[3]);
          ptx::ldmatrix_x4_trans(rb ^ 32u, sk[4], sk[5], sk[6], sk[7]);
        }
        if constexpr (kBwd) {
          uint32_t gs[8];
          if (p.bwd_skip) {
            ptx::ldmatrix_x4_trans(rb + kFastBlk, gs[0], gs[1], gs[2], gs[3]);
            ptx::ldmatrix_x4_trans((rb + kFastBlk) ^ 32u, gs[4], gs[5], gs[6], gs[7]);
          }
          ptx::tmem_ld_wait();
          uint32_t w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {          // q = 4 L + 2 n + hi: time rows r0 + 8 n + 2 (lane & 3) + {0, 1}
            const int ci = (q >> 2) * 2 + (q & 1);
            const float2 xf = __half22float2(*reinterpret_cast<const __half2*>(&sk[q]));
            float d0 = __uint_as_float(r[2 * q]), d1 = __uint_as_float(r[2 * q + 1]);
            // rows past the end of the clip hold whatever the taps that still reach valid input produced: the TMA store
            // clips them, the column sums must not see them
            const int trow = r0 + 8 * ((q >> 1) & 1) + 2 * (lane & 3);
            if (trow >= p.Tq_out) d0 = 0.f;
            if (trow + 1 >= p.Tq_out) d1 = 0.f;
            const float t0 = bw_a[ci] * xf.x, t1 = bw_a[ci] * xf.y;
            const float sn0 = __sinf(t0), cs0 = __cosf(t0), sn1 = __sinf(t1), cs1 = __cosf(t1);
            const float s20 = 2.f * sn0 * cs0, s21 = 2.f * sn1 * cs1;
            acc_da[ci] = fmaf(d0 * xf.x, s20, fmaf(d1 * xf.y, s21, acc_da[ci]));
            acc_db[ci] = fmaf(d0, sn0 * sn0, fmaf(d1, sn1 * sn1, acc_db[ci]));
            const float k = bw_ib[ci] * bw_a[ci];
            d0 *= fmaf(k, s20, 1.f);
            d1 *= fmaf(k, s21, 1.f);
            if (p.bwd_skip) {
              const float2 gf = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&gs[q]));
              d0 += gf.x;
              d1 += gf.y;
            }
            acc_bias[ci] += d0 + d1;
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(d0, d1);
            w[q] = *reinterpret_cast<const uint32_t*>(&h2);
          }
          const uint32_t ab = aring_lane + ja * kFastBlk;
          ptx::stmatrix_x4_trans(ab, w[0], w[1], w[2], w[3]);
          ptx::stmatrix_x4_trans(ab ^ 32u, w[4], w[5], w[6], w[7]);
        } else {
        ptx::tmem_ld_wait();
        uint64_t v[8];                       // q = 4 L + 2 n + hi
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          v[q] = ptx::f2_add(ptx::f2_pack_u(r[2 * q], r[2 * q + 1]), kb[(q >> 2) * 2 + (q & 1)]);
          if (has_res) {
            const float2 sf = __half22float2(*reinterpret_cast<const __half2*>(&sk[q]));
            v[q] = ptx::f2_add(v[q], ptx::f2_pack(sf.x, sf.y));
          }
        }
        if (raw_out) {
          uint32_t w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float y0, y1;
            ptx::f2_unpack(v[q], y0, y1);
            w[q] = ptx::f2h2_sat(y0, y1);
          }
          ptx::stmatrix_x4_trans(rb, w[0], w[1], w[2], w[3]);
          ptx::stmatrix_x4_trans(rb ^ 32u, w[4], w[5], w[6], w[7]);
        }
        if (act_out) {
          uint32_t w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float y0, y1;
            if (has_snake) {
              const int ci = (q >> 2) * 2 + (q & 1);
              float t0, t1;
              ptx::f2_unpack(ptx::f2_mul(v[q], ka[ci]), t0, t1);
              const uint64_t sn2 = ptx::f2_pack(sin_fast(t0), sin_fast(t1));
              ptx::f2_unpack(ptx::f2_fma(ptx::f2_mul(kib[ci], sn2), sn2, v[q]), y0, y1);
            } else {
              ptx::f2_unpack(v[q], y0, y1);
            }
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(y0, y1);
            w[q] = *reinterpret_cast<const uint32_t*>(&h2);
          }
          const uint32_t ab = aring_lane + ja * kFastBlk;
          ptx::stmatrix_x4_trans(ab, w[0], w[1], w[2], w[3]);
          ptx::stmatrix_x4_trans(ab ^ 32u, w[4], w[5], w[6], w[7]);
        }
        }   // !kBwd
        ptx::fence_proxy_async();
        __syncwarp();
        if (ptx::elect_one()) {
          if (raw_out) ptx::tma_store_4d(&tmR, ring + jr * slot_bytes, cbase, phi, r0, b);
          if (act_out) ptx::tma_store_4d(&tmO, aring + ja * kFastBlk, cbase, phi, r0, b);
          ptx::bulk_commit();                // (an empty group when only the skip block was consumed keeps the count uniform)
        }
        if (R > 0) jr = sn;
        ja ^= 1;
      }
      if constexpr (kBwd) {
        // per-channel sums: kept in registers across this CTA's tiles while the channel block stays the same; the four
        // lanes that share a channel (lane & 3 = time columns) combine, then one atomic per channel and warp
        if (ntile >= p.total_tiles || nn0 != n0) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float va = acc_da[i], vb = acc_db[i], vc = acc_bias[i];
            va += __shfl_xor_sync(0xffffffffu, va, 1); va += __shfl_xor_sync(0xffffffffu, va, 2);
            vb += __shfl_xor_sync(0xffffffffu, vb, 1); vb += __shfl_xor_sync(0xffffffffu, vb, 2);
            vc += __shfl_xor_sync(0xffffffffu, vc, 1); vc += __shfl_xor_sync(0xffffffffu, vc, 2);
            if ((lane & 3) == 0) {
              const int c = cbase + (i >> 1) * 16 + (i & 1) * 8 + g8;
              const float ib = bw_ib[i], a = bw_a[i];
              const float eb = 1.f / ib - 1e-9f;                      // exp(beta)
              atomicAdd(p.d_alpha + c, va * ib * (p.bwd_logscale ? a : 1.f));
              atomicAdd(p.d_beta + c, -vb * ib * ib * (p.bwd_logscale ? eb : 1.f));
              if (p.d_bias) atomicAdd(p.d_bias + c, vc);
            }
            acc_da[i] = 0.f; acc_db[i] = 0.f; acc_bias[i] = 0.f;
          }
        }
      }
      // accumulator buffer fully read: hand it back to the UMMA issuer
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&t_empty[acc]);
      if (++acc == p.acc_stages) { acc = 0; accph ^= 1u; }
      b = nb; q0 = nq0; phi = nphi; n0 = nn0;
    }
    if (lane == 0) ptx::bulk_wait<0>();
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue: 8 independent warp pipelines
    const int e = warp - 4;            // epilogue warp index
    const int g = e >> 2;              // item parity handled by this warp
    const int quad = warp & 3;         // TMEM lane quadrant = rows quad*32 .. +31 of a 128-row sub-tile
    const int T_out = p.Tq_out * p.P_out;
    const bool has_res = p.residual != nullptr;
    const int R = conv_umma2_raw_slots(p.raw_mode, has_res);
    const int rawblk = conv_umma2_raw_blk(p.raw_f16);
    uint8_t* raw_ring = stage_base + e * conv_umma2_stage_bytes_per_warp(p.raw_mode, p.act_mode, has_res, p.raw_f16, p.act_split);
    uint8_t* act_ring = raw_ring + R * rawblk;
    uint64_t* my_res_full = res_full + e * 3;
    // An item is one 32-row x 32-channel output block.  swap = 0: TMEM lane = time row, so a thread owns one
    // row x 32 channels (vector shared-memory accesses).  swap = 1: TMEM lane = channel, so a thread owns one
    // channel x 32 rows (scalar accesses into the same swizzled blocks; per-channel constants live in registers).
    const int ipt = p.swap ? 4 * p.MT : p.MT * (p.NT >> 5);
    // fragment-mapped path of the swap orientation for 2-byte stream / operand blocks: the launches that <1> takes
    // unless KVAE_FAST_EPI=0 sends them here
    const bool frag = p.swap && !p.act_split && !p.precise && p.raw_mode != 2 && (p.raw_f16 || (p.raw_mode == 0 && !has_res));
    // ldmatrix / stmatrix: this lane addresses row (lane & 7) of matrix (lane >> 3) inside a 16-row half of a
    // [32 rows x 64 B] SWIZZLE_64B block (lane half 1: address ^ 32, rows 16..31: + 1024)
    const int frag_row = ((lane >> 4) << 3) + (lane & 7);
    const uint32_t frag_lane = frag_row * 64 + ((((lane >> 3) & 1) ^ ((frag_row >> 1) & 3)) << 4);
    int acc = 0, jr = 0, ja = 0;
    uint32_t accph = 0, res_ph = 0;          // res_ph: one parity bit per ring slot
    // item -> block coordinates: (channel, phase, first row, batch)
    auto coords = [&](int tile, int item, int& cb, int& ph, int& r0, int& bb) {
      int q0, n0;
      decode(tile, bb, q0, ph, n0);
      if (p.swap) {
        cb = n0 + quad * 32;
        r0 = q0 + item * 32;
      } else {
        cb = n0 + (item % (p.NT >> 5)) * 32;
        r0 = q0 + (item / (p.NT >> 5)) * 128 + quad * 32;
      }
    };
    if (has_res && lane == 0 && static_cast<int>(blockIdx.x) < p.total_tiles && g < ipt) {
      int cb, ph, r0, bb;
      coords(blockIdx.x, g, cb, ph, r0, bb);
      ptx::mbar_expect_tx(&my_res_full[0], rawblk);
      ptx::tma_load_4d(raw_ring, &tmX, &my_res_full[0], cb, ph, r0, bb);
    }
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      int b, q0, phi, n0;
      decode(tile, b, q0, phi, n0);
      // swap mode: this thread's channel and its constants
      uint64_t fbias[4] = {0, 0, 0, 0}, fsa[4] = {0, 0, 0, 0}, fsib[4] = {0, 0, 0, 0};   // index 2 L + hi
      if (frag) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int c = n0 + quad * 32 + (i >> 1) * 16 + (i & 1) * 8 + (lane >> 2);
          const float bv = p.bias ? __ldg(p.bias + c) : 0.f;
          fbias[i] = ptx::f2_pack(bv, bv);
          if (p.snake_a) {
            const float a = __ldg(p.snake_a + c), ib = __ldg(p.snake_inv_b + c);
            fsa[i] = ptx::f2_pack(a, a);
            fsib[i] = ptx::f2_pack(ib, ib);
          }
        }
      }
      float bias_s = 0.f, sa_s = 1.f, sib_s = 0.f;
      if (p.swap && !frag) {
        const int c = n0 + quad * 32 + lane;
        if (p.bias) bias_s = __ldg(p.bias + c);
        if (p.snake_a) { sa_s = __ldg(p.snake_a + c); sib_s = __ldg(p.snake_inv_b + c); }
      }
      ptx::mbar_wait(&t_full[acc], accph);
      ptx::tc_fence_after();
      const uint32_t acc_tmem = tmem_base + acc * acc_cols + (static_cast<uint32_t>(quad * 32) << 16);
      for (int item = g; item < ipt; item += 2) {
        int cbase, r0, tcol;
        if (p.swap) {
          cbase = n0 + quad * 32;
          r0 = q0 + item * 32;
          tcol = item * 32;
        } else {
          const int m = item / (p.NT >> 5);
          const int c0 = (item % (p.NT >> 5)) * 32;
          cbase = n0 + c0;
          r0 = q0 + m * 128 + quad * 32;   // first row of this warp's block
          tcol = m * p.NT + c0;
        }
        // lane 0: recycle the oldest blocks, then prefetch the NEXT item's skip-connection block
        if (lane == 0 && (R > 0 || p.act_mode == 1)) ptx::bulk_wait_read<1>();
        if (has_res) {
          if (lane == 0) {
            int nt = tile, ni = item + 2;
            if (ni >= ipt) { nt = tile + gridDim.x; ni = g; }
            if (nt < p.total_tiles && ni < ipt) {
              int cb, ph, rr, bb;
              coords(nt, ni, cb, ph, rr, bb);
              const int sn = (jr + 1) % R;
              ptx::mbar_expect_tx(&my_res_full[sn], rawblk);
              ptx::tma_load_4d(raw_ring + sn * rawblk, &tmX, &my_res_full[sn], cb, ph, rr, bb);
            }
          }
          ptx::mbar_wait(&my_res_full[jr], (res_ph >> jr) & 1u);
          res_ph ^= (1u << jr);
        }
        uint8_t* const rblk = raw_ring + jr * rawblk;
        const int actblk = kActBlkBytes * (p.act_split ? 2 : 1);       // (hi | lo) blocks back to back
        uint8_t* const ablk = act_ring + ja * actblk;
        if (frag) {
          // ---- swap orientation, 2-byte stream / operand blocks: fragment mapping (see conv_ru2.cuh).  tcgen05.ld
          // .16x256b hands a thread (time, time+1) PAIRS of one channel; bias, skip and SnakeBeta run on packed fp32
          // pairs, a converted pair is one stmatrix.trans register and the skip block comes in through ldmatrix.trans,
          // so the [32 rows x 64 B] SWIZZLE_64B blocks are touched in 16-byte rows instead of 2 bytes per element.
          uint32_t r[32];                                    // r[16 L + 4 n + 2 hi + {0,1}]: lane half L, column group n
          __syncwarp();
          ptx::tmem_ld_16x256b_x4(acc_tmem + tcol, r);
          ptx::tmem_ld_16x256b_x4(acc_tmem + tcol + (16u << 16), r + 16);
          uint32_t sk[16];                                   // sk[8 L + 4 m + j]: rows 16 m + 8 (j >> 1) .., channel group 2 L + (j & 1)
          const uint32_t rb = ptx::smem_u32(rblk) + frag_lane;
          if (has_res) {
#pragma unroll
            for (int L = 0; L < 2; ++L)
#pragma unroll
              for (int m = 0; m < 2; ++m)
                ptx::ldmatrix_x4_trans((rb + m * 1024) ^ (L * 32u), sk[8 * L + 4 * m], sk[8 * L + 4 * m + 1],
                                       sk[8 * L + 4 * m + 2], sk[8 * L + 4 * m + 3]);
          }
          ptx::tmem_ld_wait();
          uint64_t v[16];                                    // v[8 L + 4 m + j], j = 2 (n & 1) + hi, n = 2 m + (j >> 1)
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const int L = q >> 3, ci = 2 * L + (q & 1);      // channel cbase + 16 L + 8 hi + (lane >> 2)
            const int ri = 16 * L + 4 * (2 * ((q >> 2) & 1) + ((q >> 1) & 1)) + 2 * (q & 1);
            v[q] = ptx::f2_add(ptx::f2_pack_u(r[ri], r[ri + 1]), fbias[ci]);
            if (has_res) {
              const float2 sf = __half22float2(*reinterpret_cast<const __half2*>(&sk[q]));
              v[q] = ptx::f2_add(v[q], ptx::f2_pack(sf.x, sf.y));
            }
          }
          if (p.raw_mode == 1) {
            uint32_t w[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              float y0, y1;
              ptx::f2_unpack(v[q], y0, y1);
              w[q] = ptx::f2h2_sat(y0, y1);
            }
#pragma unroll
            for (int L = 0; L < 2; ++L)
#pragma unroll
              for (int m = 0; m < 2; ++m)
                ptx::stmatrix_x4_trans((rb + m * 1024) ^ (L * 32u), w[8 * L + 4 * m], w[8 * L + 4 * m + 1],
                                       w[8 * L + 4 * m + 2], w[8 * L + 4 * m + 3]);
          }
          if (p.act_mode == 1) {
            uint32_t w[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              float y0, y1;
              if (p.snake_a) {
                const int ci = 2 * (q >> 3) + (q & 1);
                float t0, t1;
                ptx::f2_unpack(ptx::f2_mul(v[q], fsa[ci]), t0, t1);
                const uint64_t sn = ptx::f2_pack(sin_fast(t0), sin_fast(t1));
                ptx::f2_unpack(ptx::f2_fma(ptx::f2_mul(fsib[ci], sn), sn, v[q]), y0, y1);
              } else {
                ptx::f2_unpack(v[q], y0, y1);
              }
              const __nv_bfloat162 h2 = __floats2bfloat162_rn(y0, y1);
              w[q] = *reinterpret_cast<const uint32_t*>(&h2);
            }
            const uint32_t ab = ptx::smem_u32(ablk) + frag_lane;
#pragma unroll
            for (int L = 0; L < 2; ++L)
#pragma unroll
              for (int m = 0; m < 2; ++m)
                ptx::stmatrix_x4_trans((ab + m * 1024) ^ (L * 32u), w[8 * L + 4 * m], w[8 * L + 4 * m + 1],
                                       w[8 * L + 4 * m + 2], w[8 * L + 4 * m + 3]);
          }
        } else {
        uint32_t r[32];
        __syncwarp();
        ptx::tmem_ld_32x32(acc_tmem + tcol, r);
        ptx::tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (p.swap) {
          // ---- thread = channel (cbase + lane), v[j] = row r0 + j
          // element (row j, channel lane) of a SWIZZLE_128B fp32 block / SWIZZLE_64B bf16 block
          const uint32_t rcol = (lane & 3) * 4, rchunk = lane >> 2;
          const uint32_t acol = (lane & 7) * 2, achunk = lane >> 3;
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += bias_s;
          uint8_t* rbase[8];     // the 8 distinct swizzle phases of a SWIZZLE_128B block
#pragma unroll
          for (int c = 0; c < 8; ++c) rbase[c] = rblk + ((rchunk ^ c) << 4) + rcol;
          uint8_t* hbase[4];     // fp16 stream block: same shape and swizzle as the bf16 operand block
#pragma unroll
          for (int c = 0; c < 4; ++c) hbase[c] = rblk + ((achunk ^ c) << 4) + acol;
          if (has_res) {
            if (p.raw_f16) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] += __half2float(*reinterpret_cast<const __half*>(hbase[(j >> 1) & 3] + j * 64));
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] += *reinterpret_cast<const float*>(rbase[j & 7] + j * 128);
            }
          }
          if (p.raw_mode == 2) {
            const int c = cbase + lane;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int q = r0 + j;
              if (q < p.Tq_out) {
                const size_t o = (static_cast<size_t>(b) * p.Cout + c) * (p.cf_ld ? p.cf_ld : T_out) + static_cast<size_t>(q) * p.P_out + phi;
                if (p.out_cf_f32) static_cast<float*>(p.out_cf)[o] = v[j];
                else static_cast<__nv_bfloat16*>(p.out_cf)[o] = __float2bfloat16(v[j]);
                fused_sigma_sample(p, b, c, static_cast<size_t>(q) * p.P_out + phi, T_out, v[j]);
              }
            }
          }
          if (p.raw_mode == 1) {
            if (p.raw_f16) {
#pragma unroll
              for (int j = 0; j < 32; ++j) *reinterpret_cast<uint16_t*>(hbase[(j >> 1) & 3] + j * 64) = ptx::f2h_sat(v[j]);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) *reinterpret_cast<float*>(rbase[j & 7] + j * 128) = v[j];
            }
          }
          if (p.act_mode == 1) {
            if (p.snake_a) {   // hoisted: a per-element test would put a branch between the 32 independent chains
              if (p.precise) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = snake_beta_rr(v[j], sa_s, sib_s);
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = snake_beta<true>(v[j], sa_s, sib_s);
              }
            }
            uint8_t* abase[4];   // the 4 distinct swizzle phases of a SWIZZLE_64B block
#pragma unroll
            for (int c = 0; c < 4; ++c) abase[c] = ablk + ((achunk ^ c) << 4) + acol;
            if (p.act_split) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const __nv_bfloat16 hi = __float2bfloat16(v[j]);
                *reinterpret_cast<__nv_bfloat16*>(abase[(j >> 1) & 3] + j * 64) = hi;
                *reinterpret_cast<__nv_bfloat16*>(abase[(j >> 1) & 3] + kActBlkBytes + j * 64) =
                    __float2bfloat16(v[j] - __bfloat162float(hi));
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                *reinterpret_cast<__nv_bfloat16*>(abase[(j >> 1) & 3] + j * 64) = __float2bfloat16(v[j]);
            }
          }
        } else {
        // ---- thread = time row (r0 + lane), v[j] = channel cbase + j
        if (p.bias) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 bb4 = __ldg(reinterpret_cast<const float4*>(p.bias + cbase + j));
            v[j] += bb4.x; v[j + 1] += bb4.y; v[j + 2] += bb4.z; v[j + 3] += bb4.w;
          }
        }
        uint8_t* rt = rblk + lane * 128;
        uint8_t* rt16 = rblk + lane * 64;                 // fp16 stream block row
        if (has_res) {
          if (p.raw_f16) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 q = *reinterpret_cast<const uint4*>(rt16 + ((j ^ ((lane >> 1) & 3)) << 4));
              const __half2* h2 = reinterpret_cast<const __half2*>(&q);
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4) {
                const float2 f = __half22float2(h2[q4]);
                v[8 * j + 2 * q4] += f.x; v[8 * j + 2 * q4 + 1] += f.y;
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 x = *reinterpret_cast<const float4*>(rt + ((j ^ (lane & 7)) << 4));
              v[4 * j] += x.x; v[4 * j + 1] += x.y; v[4 * j + 2] += x.z; v[4 * j + 3] += x.w;
            }
          }
        }
        if (p.raw_mode == 2) {
          // channels-first API output: lanes hold consecutive time steps -> coalesced per channel
          const int q = r0 + lane;
          if (q < p.Tq_out) {
            const size_t t_out = static_cast<size_t>(q) * p.P_out + phi;
            const size_t ld = p.cf_ld ? static_cast<size_t>(p.cf_ld) : static_cast<size_t>(T_out);
            const size_t o0 = (static_cast<size_t>(b) * p.Cout + cbase) * ld + t_out;
            if (p.out_cf_f32) {
              float* op = static_cast<float*>(p.out_cf) + o0;
#pragma unroll
              for (int j = 0; j < 32; ++j) op[static_cast<size_t>(j) * ld] = v[j];
            } else {
              __nv_bfloat16* op = static_cast<__nv_bfloat16*>(p.out_cf) + o0;
#pragma unroll
              for (int j = 0; j < 32; ++j) op[static_cast<size_t>(j) * ld] = __float2bfloat16(v[j]);
            }
            if (p.samp_noise) {
#pragma unroll
              for (int j = 0; j < 32; ++j) fused_sigma_sample(p, b, cbase + j, t_out, T_out, v[j]);
            }
          }
        }
        if (p.raw_mode == 1) {
          if (p.raw_f16) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint32_t w[4];
#pragma unroll
              for (int q4 = 0; q4 < 4; ++q4) {
                w[q4] = ptx::f2h2_sat(v[8 * j + 2 * q4], v[8 * j + 2 * q4 + 1]);
              }
              *reinterpret_cast<uint4*>(rt16 + ((j ^ ((lane >> 1) & 3)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<float4*>(rt + ((j ^ (lane & 7)) << 4)) =
                  make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
        }
        if (p.act_mode == 1) {
          if (p.snake_a) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 a = __ldg(reinterpret_cast<const float4*>(p.snake_a + cbase + j));
              const float4 ib = __ldg(reinterpret_cast<const float4*>(p.snake_inv_b + cbase + j));
              if (p.precise) {
                v[j] = snake_beta_rr(v[j], a.x, ib.x);
                v[j + 1] = snake_beta_rr(v[j + 1], a.y, ib.y);
                v[j + 2] = snake_beta_rr(v[j + 2], a.z, ib.z);
                v[j + 3] = snake_beta_rr(v[j + 3], a.w, ib.w);
              } else {
                v[j] = snake_beta<true>(v[j], a.x, ib.x);
                v[j + 1] = snake_beta<true>(v[j + 1], a.y, ib.y);
                v[j + 2] = snake_beta<true>(v[j + 2], a.z, ib.z);
                v[j + 3] = snake_beta<true>(v[j + 3], a.w, ib.w);
              }
            }
          }
          uint8_t* at = ablk + lane * 64;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint32_t w[4], wl[4];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              __nv_bfloat162 h = __floats2bfloat162_rn(v[8 * j + 2 * q4], v[8 * j + 2 * q4 + 1]);
              w[q4] = *reinterpret_cast<uint32_t*>(&h);
              if (p.act_split) {
                const float2 hf = __bfloat1622float2(h);
                __nv_bfloat162 l = __floats2bfloat162_rn(v[8 * j + 2 * q4] - hf.x, v[8 * j + 2 * q4 + 1] - hf.y);
                wl[q4] = *reinterpret_cast<uint32_t*>(&l);
              }
            }
            *reinterpret_cast<uint4*>(at + ((j ^ ((lane >> 1) & 3)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            if (p.act_split)
              *reinterpret_cast<uint4*>(at + kActBlkBytes + ((j ^ ((lane >> 1) & 3)) << 4)) =
                  make_uint4(wl[0], wl[1], wl[2], wl[3]);
          }
        }
        }
        }   // !frag
        if (R > 0 || p.act_mode == 1) {
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            if (p.raw_mode == 1) ptx::tma_store_4d(&tmR, raw_ring + jr * rawblk, cbase, phi, r0, b);
            if (p.act_mode == 1) {
              ptx::tma_store_4d(&tmO, ablk, cbase, phi, r0, b);
              if (p.act_split) ptx::tma_store_4d(&tmO, ablk + kActBlkBytes, p.Cout + cbase, phi, r0, b);
            }
            ptx::bulk_commit();   // (an empty group when only the skip block was consumed keeps the count uniform)
          }
          if (R > 0) jr = (jr + 1 == R) ? 0 : jr + 1;
          ja ^= 1;
        }
      }
      // accumulator buffer fully read: hand it back to the UMMA issuer
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&t_empty[acc]);
      if (++acc == p.acc_stages) { acc = 0; accph ^= 1u; }
    }
    if (lane == 0) ptx::bulk_wait<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, p.tmem_cols);
}

}  // namespace kvae
