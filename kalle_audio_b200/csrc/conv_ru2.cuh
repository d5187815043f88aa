// conv_ru2: one-kernel ResidualUnit for 128-channel stages (reference autoencoders.py:39-62):
//     x' = x + conv_k1( SnakeBeta2( conv_k7_dil_d( SnakeBeta1(x) ) ) )
// The producer of x already wrote a = SnakeBeta1(x) (bf16 operand) and x (the fp16 residual stream); this kernel never
// materialises the intermediate h = SnakeBeta2(conv_k7(a)) in HBM.  Per output row it moves 256 B (a) + 256 B (x) in and
// 256 B (x') + 256 B (a' = next layer's operand) out = 1024 B instead of the 1536 B of the two-kernel form, which also
// writes and reads h -- these stages are HBM-bound, so that is the speed-up.
//
// Orientation (see conv_umma2.cuh "swap"): out-channels on the MMA M side (TMEM lanes), 256 time rows on N.
//   GEMM1  D1[co, t]  = sum_{tap,ci} W7[tap][co, ci] * a[t + shift(tap), ci]      (14 x 4 MMAs of 128x256x16)
//   EPI1   h[t, c]    = bf16( SnakeBeta2( D1[c, t] + bias7[c] ) )  -> shared memory, K-major, 128-row halves
//   GEMM2  D2[co2, t] = sum_c W1[co2, c] * h[t, c]                                 (2 halves x 2 x 4 MMAs of 128x128x16)
//   EPI2   x'[t, c]   = D2[c, t] + bias1[c] + x[t, c]  -> fp16 stream (TMA store); a' = bf16(SnakeBeta_next(x')) (TMA store)
// Warp roles (640 threads): 0 weight TMA producer, 1 UMMA issuer, 2 TMEM allocator, 3 activation-slab TMA producer, 4-19
// epilogue.  All 16 epilogue warps (4 per TMEM lane quadrant) do BOTH epilogues, one after the other: their EPI1 share of
// a tile, then their EPI2 share (4 of the 16 16-row items); with separate EPI1 / EPI2 warp groups the EPI1 warps idled
// 70 % of the time waiting for GEMM1 (profiles/r01_conv_ru_unified_epilogue_B16.ncu-rep).  Every warp prefetches its
// next skip-connection block by TMA and stores in place.
//
// The tensor pipe is kept busy across tiles.  Run as a serial GEMM1 -> EPI1 -> GEMM2 chain on one accumulator (the
// first two generations of this kernel), the chain alone (no HBM traffic at all) cost 0.35 of the 0.47 ms per launch,
// against 0.19 ms of tensor work (profiles/r01_ru_ablation.txt).  Here:
//   * TMEM holds TWO 256-column accumulators; tile i uses buffer i & 1.  GEMM2 of a half writes D2 IN PLACE over the
//     128 columns of D1 that EPI1 has just consumed, so two tiles are in flight in 512 columns.
//   * The single MMA thread issues GEMM1 of tile i+1 slab by slab and slots the two GEMM2 halves of tile i in at
//     fixed slab positions (kRuK0, kRuK1): the k=1 conv of tile i executes in the middle of the k=7 conv of tile i+1,
//     the pipe never drains while the epilogue warps turn D1 into h, and EPI2 of tile i runs under the rest of GEMM1.
//   * The weight ring is strictly FIFO in that issue order: W7 slabs of tile i+1 with the two W1 chunks of tile i
//     inserted (twice, once per half) at the same positions.
//   * Epilogue warps use the mma-style fragment mapping (tcgen05.ld.16x256b, ldmatrix/stmatrix.trans, packed fp32
//     pairs).
// Shared memory (227 KB): activation slab ring 2 x <=40 KB, weight ring of 16 KB stages (W7 taps, then the two W1
// chunks of the tile), h half 32 KB, epilogue staging 16 x 3 KB.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "conv_umma2.cuh"

namespace kvae {

struct RuParams {
  int B, T;                 // rows per clip (stride-1 conv: T_in == T_out)
  int RB, nbox;             // activation slab = nbox TMA boxes of RB rows (256 + 6*dilation rows)
  int SA, SB;
  int q_tiles, total_tiles; // 256-row tiles
  uint32_t tap_shift16[7];  // (tap*dilation*128 B) >> 4
  int slab_row0;            // slab start row relative to the tile's first row (= -3*dilation)
  const float* bias7;       // [128]
  const float* s2_a;        // SnakeBeta between the two convs
  const float* s2_inv_b;
  const float* bias1;       // [128]
  int raw_out;              // 1: fp16 stream out via tmR
  int act_out;              // 1: bf16 operand out via tmO
  const float* sn_a;        // SnakeBeta folded into the operand output (nullptr: plain cast)
  const float* sn_inv_b;
  int act_f16;              // the operand output is fp16 instead of bf16 (the unit in front of the decoder tail,
                            // whose GEMM is kind::f16 -- conv_edge.cuh, WaveOutTcParams::preact)
};

constexpr int kRuC = 128;
constexpr int kRuHBytes = 2 * 128 * 128;   // h half: 2 K-chunks x [128 rows x 128 B]
constexpr int kRuActBlk = 16 * 64;         // 16 rows x 32 bf16 / fp16, SWIZZLE_64B
constexpr int kRuThreads = 640;
constexpr int kRuEpiWarps = 16;
// GEMM2 half 0 / half 1 of tile i are issued before slab kRuK0 / kRuK1 of tile i+1's GEMM1 (14 slabs: 2 chunks x 7 taps)
constexpr int kRuK0 = 3, kRuK1 = 6;

// per epilogue warp: 2 fp16 stream blocks (skip in / stream out, in place) + 1 bf16 operand block
__host__ __device__ inline int ru_stage_bytes_per_warp(int act_out) { return 2 * kRuActBlk + (act_out ? kRuActBlk : 0); }
__host__ __device__ inline size_t ru_smem_bytes(const RuParams& p) {
  return 1024 + 1024 + static_cast<size_t>(p.SA) * p.nbox * p.RB * 128 + static_cast<size_t>(p.SB) * kRuC * 128 +
         kRuHBytes + kRuEpiWarps * ru_stage_bytes_per_warp(p.act_out);
}

__global__ void __launch_bounds__(kRuThreads, 1)
conv_ru2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW7,
                const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmR,
                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmX,
                const __grid_constant__ RuParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* a_empty = a_full + 8;
  uint64_t* b_full = a_full + 16;
  uint64_t* b_empty = a_full + 32;
  uint64_t* d1_full = a_full + 48;     // [2] GEMM1 into buffer j has retired
  uint64_t* buf_empty = a_full + 50;   // [2] EPI2 has drained buffer j (16 arrivals)
  uint64_t* h_full = a_full + 52;
  uint64_t* h_empty = a_full + 53;
  uint64_t* d2h_full = a_full + 54;    // GEMM2 of half 0 has retired: rows 0..127 of D2 are final
  uint64_t* d2_full = a_full + 55;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_full + 56);
  uint64_t* res_full = a_full + 58;    // [16 epilogue warps][2 slots]
  uint8_t* a_ring = smem + 1024;
  const uint32_t a_bytes = static_cast<uint32_t>(p.nbox) * p.RB * 128;
  constexpr uint32_t b_bytes = kRuC * 128;
  uint8_t* b_ring = a_ring + static_cast<size_t>(p.SA) * a_bytes;
  uint8_t* h_buf = b_ring + static_cast<size_t>(p.SB) * b_bytes;
  uint8_t* stage_base = h_buf + kRuHBytes;

  const int warp = ptx::warp_idx();
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW7);
    ptx::prefetch_tmap(&tmW1);
    ptx::prefetch_tmap(&tmX);
    if (p.raw_out) ptx::prefetch_tmap(&tmR);
    if (p.act_out) ptx::prefetch_tmap(&tmO);
    for (int i = 0; i < p.SA; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < p.SB; ++i) { ptx::mbar_init(&b_full[i], 1); ptx::mbar_init(&b_empty[i], 1); }
    for (int j = 0; j < 2; ++j) { ptx::mbar_init(&d1_full[j], 1); ptx::mbar_init(&buf_empty[j], kRuEpiWarps); }
    ptx::mbar_init(h_full, kRuEpiWarps);
    ptx::mbar_init(h_empty, 1);
    ptx::mbar_init(d2h_full, 1);
    ptx::mbar_init(d2_full, 1);
    for (int i = 0; i < 2 * kRuEpiWarps; ++i) ptx::mbar_init(&res_full[i], 1);
    ptx::fence_mbar_init();
  }
  ptx::pdl_launch_dependents();
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  ptx::pdl_wait();
  const uint32_t tmem_base = *tmem_slot;
  constexpr int k0 = kRuK0, k1 = kRuK1;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer: ring entries in MMA issue order
    {   // warp-uniform loop, one elected lane issues
      int bs = 0;
      uint32_t bph = 0;
      auto load_w = [&](const CUtensorMap* tm, int c0, int c2) {
        ptx::mbar_wait(&b_empty[bs], bph ^ 1u);
        if (ptx::elect_one()) {
          ptx::mbar_expect_tx(&b_full[bs], b_bytes);
          ptx::tma_load_3d(b_ring + static_cast<size_t>(bs) * b_bytes, tm, &b_full[bs], c0, 0, c2);
        }
        __syncwarp();
        if (++bs == p.SB) { bs = 0; bph ^= 1u; }
      };
      for (int i = -1, nxt = blockIdx.x;; ++i, nxt += gridDim.x) {
        const bool has_cur = i >= 0, has_next = nxt < p.total_tiles;
        for (int s = 0; s < 14; ++s) {
          if (has_cur && (s == k0 || s == k1)) {
            load_w(&tmW1, 0, 0);
            load_w(&tmW1, 64, 0);
          }
          if (has_next) load_w(&tmW7, (s / 7) * 64, s % 7);
        }
        if (!has_next) break;
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------ TMA producer for the activation slabs, on its own
    // thread: in one FIFO with the weights a slab was requested only SB weight stages (~1 us) before its first MMA,
    // less than an HBM round trip, although its ring stage had been free for half a tile (profiles/r01_ru_ablation.txt:
    // removing these 67 KB per tile saved 23 % of the launch).  Here a slab is requested the moment its stage is free.
    {   // warp-uniform loop, one elected lane issues
      int as = 0;
      uint32_t aph = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int b = tile / p.q_tiles;
        const int q0 = (tile % p.q_tiles) * 256;
        for (int ch = 0; ch < 2; ++ch) {
          ptx::mbar_wait(&a_empty[as], aph ^ 1u);
          if (ptx::elect_one()) {
            ptx::mbar_expect_tx(&a_full[as], a_bytes);
            for (int bx = 0; bx < p.nbox; ++bx)
              ptx::tma_load_4d(a_ring + static_cast<size_t>(as) * a_bytes + bx * p.RB * 128, &tmA, &a_full[as], ch * 64, 0,
                               q0 + p.slab_row0 + bx * p.RB, b);
          }
          __syncwarp();
          if (++as == p.SA) { as = 0; aph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ UMMA issuer
    {   // the whole warp walks the schedule and the barriers, one elected lane issues (see conv_umma2.cuh)
      const uint32_t idesc1 = ptx::idesc_bf16_f32(128, 256);
      const uint32_t idesc2 = ptx::idesc_bf16_f32(128, 128);
      const uint64_t desc_hi = (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      const uint32_t a_lo0 = ((ptx::smem_u32(a_ring) & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t b_lo0 = ((ptx::smem_u32(b_ring) & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t h_lo0 = ((ptx::smem_u32(h_buf) & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t a_stage16 = a_bytes >> 4, b_stage16 = b_bytes >> 4;
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0, hf_ph = 0;
      int cur_a = 0;
      uint32_t cur_lo = 0;
      for (int i = -1, nxt = blockIdx.x;; ++i, nxt += gridDim.x) {
        const bool has_cur = i >= 0, has_next = nxt < p.total_tiles;
        const uint32_t dcur = tmem_base + static_cast<uint32_t>(i & 1) * 256;        // D1 / D2 of tile i
        const uint32_t dnext = tmem_base + static_cast<uint32_t>((i + 1) & 1) * 256;  // D1 of tile i + 1
#pragma unroll 1
        for (int s = 0; s < 14; ++s) {
          if (has_cur && (s == k0 || s == k1)) {
            // ---- GEMM2 of one 128-row half of tile i, in place over the D1 columns EPI1 has consumed
            const int half = (s == k0) ? 0 : 1;
            const int s0 = bs;
            const uint32_t ph0 = bph;
            if (++bs == p.SB) { bs = 0; bph ^= 1u; }
            const int s1 = bs;
            const uint32_t ph1 = bph;
            if (++bs == p.SB) { bs = 0; bph ^= 1u; }
            ptx::mbar_wait(&b_full[s0], ph0);
            ptx::mbar_wait(&b_full[s1], ph1);
            ptx::mbar_wait(h_full, hf_ph);
            hf_ph ^= 1u;
            ptx::tc_fence_after();
            const uint32_t dd = dcur + half * 128;
            const uint32_t w_lo[2] = {b_lo0 + s0 * b_stage16, b_lo0 + s1 * b_stage16};
            if (ptx::elect_one()) {
#pragma unroll
              for (int kc = 0; kc < 2; ++kc) {
                const uint32_t hl = h_lo0 + kc * (16384 >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  ptx::umma_f16(dd, desc_hi | (w_lo[kc] + 2 * k), desc_hi | (hl + 2 * k), idesc2, (kc | k) ? 1u : 0u);
              }
              ptx::umma_commit(h_empty);
              ptx::umma_commit(&b_empty[s0]);
              ptx::umma_commit(&b_empty[s1]);
              ptx::umma_commit(half == 0 ? d2h_full : d2_full);
            }
            __syncwarp();
          }
          if (has_next) {
            // ---- slab s of GEMM1 of tile i + 1: chunk s / 7, tap s % 7
            if (s == 0) {
              const int j = i + 1;                                   // this CTA's j-th tile
              ptx::mbar_wait(&buf_empty[j & 1], ((j >> 1) & 1u) ^ 1u);
              ptx::tc_fence_after();
            }
            if (s == 0 || s == 7) {
              ptx::mbar_wait(&a_full[as], aph);
              cur_a = as;
              cur_lo = a_lo0 + as * a_stage16;
              if (++as == p.SA) { as = 0; aph ^= 1u; }
            }
            ptx::mbar_wait(&b_full[bs], bph);
            ptx::tc_fence_after();
            const int t = s >= 7 ? s - 7 : s;
            const uint32_t al = cur_lo + p.tap_shift16[t];
            const uint32_t bl = b_lo0 + bs * b_stage16;
            const int cbs = bs;
            if (++bs == p.SB) { bs = 0; bph ^= 1u; }
            if (ptx::elect_one()) {
              ptx::umma_f16(dnext, desc_hi | bl, desc_hi | al, idesc1, s ? 1u : 0u);
              ptx::umma_f16(dnext, desc_hi | (bl + 2), desc_hi | (al + 2), idesc1, 1u);
              ptx::umma_f16(dnext, desc_hi | (bl + 4), desc_hi | (al + 4), idesc1, 1u);
              ptx::umma_f16(dnext, desc_hi | (bl + 6), desc_hi | (al + 6), idesc1, 1u);
              ptx::umma_commit(&b_empty[cbs]);
              if (s == 6 || s == 13) ptx::umma_commit(&a_empty[cur_a]);
              if (s == 13) ptx::umma_commit(&d1_full[(i + 1) & 1]);
            }
            __syncwarp();
          }
        }
        if (!has_next) break;
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue warps (fragment mapping)
    const int e = warp - 4;                            // 0..15
    const int quad = warp & 3;                         // TMEM lane quadrant = channels quad*32 .. +31
    const int sub = e >> 2;                            // 0..3
    const int g = lane >> 2;                           // fragment row: channel within a group of 8
    const int rr = lane & 7, mj = lane >> 3;           // ldmatrix/stmatrix: this lane addresses row rr of matrix mj
    const int cbase = quad * 32;
    auto dup = [](float f) { return ptx::f2_pack(f, f); };
    // EPI1 share of a 128-column half: 16 channels (lane half hl) x 64 time columns (block cb)
    const int hl = sub & 1, cb = sub >> 1;
    const int c1 = cbase + hl * 16 + g;                // this thread's EPI1 channels: c1 and c1 + 8
    const uint32_t d1_lane = tmem_base + (static_cast<uint32_t>(cbase + hl * 16) << 16) + cb * 64;
    const int hch = cbase + hl * 16 + (mj & 1) * 8;    // first channel of the 8-channel group of matrix mj
    const uint32_t h_lane = ptx::smem_u32(h_buf) + (hch >> 6) * 16384 + (cb * 64 + (mj >> 1) * 8 + rr) * 128 +
                            ((((hch & 63) >> 3) ^ rr) << 4);
    // EPI2 staging: fp16 stream blocks [16 rows x 64 B] and the bf16 operand block, SWIZZLE_64B; lane half 1 = ^ 32
    uint8_t* ring = stage_base + e * ru_stage_bytes_per_warp(p.act_out);
    const int brow = (mj >> 1) * 8 + rr;
    const uint32_t blk_lane = brow * 64 + (((mj & 1) ^ ((brow >> 1) & 3)) << 4);
    const uint32_t ring_lane = ptx::smem_u32(ring) + blk_lane;
    const uint32_t ablk_lane = ring_lane + 2 * kRuActBlk;
    uint8_t* ablk = ring + 2 * kRuActBlk;
    uint64_t* my_res_full = res_full + e * 2;
    const bool has_snake = p.sn_a != nullptr;
    auto issue_skip = [&](int tb, int tq0, int item, int slot) {   // lane 0 only; (tb, tq0) = clip, first row of the tile
      ptx::mbar_expect_tx(&my_res_full[slot], kRuActBlk);
      ptx::tma_load_4d(ring + slot * kRuActBlk, &tmX, &my_res_full[slot], cbase, 0, tq0 + item * 16, tb);
    };
    if (static_cast<int>(blockIdx.x) < p.total_tiles && ptx::elect_one())
      issue_skip(blockIdx.x / p.q_tiles, (blockIdx.x % p.q_tiles) * 256, sub, 0);
    int slot = 0;
    uint32_t he_ph = 0, d2f_ph = 0, res_ph = 0;
    int it = 0;                                          // this CTA's it-th tile: accumulator buffer it & 1
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      // (quotients come out of the vector ALU; the lane-0 broadcast tells ptxas they are warp-uniform, so the TMA
      // coordinates built from them sit in uniform registers instead of going through an R2UR waterfall loop per issue)
      const int b = __shfl_sync(0xffffffffu, tile / p.q_tiles, 0);
      const int q0 = __shfl_sync(0xffffffffu, (tile % p.q_tiles) * 256, 0);
      const int ntile = tile + gridDim.x;                // this CTA's next tile (its first skip block is prefetched below)
      const int nb = __shfl_sync(0xffffffffu, ntile / p.q_tiles, 0), nq0 = __shfl_sync(0xffffffffu, (ntile % p.q_tiles) * 256, 0);
      const uint32_t boff = static_cast<uint32_t>(it & 1) * 256;
      // ---- EPI1 share: D1 -> bias, SnakeBeta -> h
      {
        const uint64_t kb[2] = {dup(__ldg(p.bias7 + c1)), dup(__ldg(p.bias7 + c1 + 8))};
        const uint64_t ka[2] = {dup(__ldg(p.s2_a + c1)), dup(__ldg(p.s2_a + c1 + 8))};
        const uint64_t kib[2] = {dup(__ldg(p.s2_inv_b + c1)), dup(__ldg(p.s2_inv_b + c1 + 8))};
        ptx::mbar_wait_parked(&d1_full[it & 1], (it >> 1) & 1u);
        ptx::tc_fence_after();
        for (int half = 0; half < 2; ++half) {
          uint32_t r[32], pk[16];
          __syncwarp();
          ptx::tmem_ld_16x256b_x8(d1_lane + boff + half * 128, r);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 16; ++q) {                 // q = 2n + hi: column group n, channel c1 + 8 hi
            const uint64_t v = ptx::f2_add(ptx::f2_pack_u(r[2 * q], r[2 * q + 1]), kb[q & 1]);
            float t0, t1, y0, y1;
            ptx::f2_unpack(ptx::f2_mul(v, ka[q & 1]), t0, t1);
            const uint64_t sn = ptx::f2_pack(sin_fast(t0), sin_fast(t1));
            ptx::f2_unpack(ptx::f2_fma(ptx::f2_mul(kib[q & 1], sn), sn, v), y0, y1);
            const __nv_bfloat162 hb2 = __floats2bfloat162_rn(y0, y1);
            pk[q] = *reinterpret_cast<const uint32_t*>(&hb2);
          }
          ptx::mbar_wait_parked(h_empty, he_ph ^ 1u);      // GEMM2 of the previous half has consumed h
          he_ph ^= 1u;
#pragma unroll
          for (int m = 0; m < 4; ++m)
            ptx::stmatrix_x4_trans(h_lane + m * 2048, pk[4 * m], pk[4 * m + 1], pk[4 * m + 2], pk[4 * m + 3]);
          ptx::fence_proxy_async();
          ptx::tc_fence_before();                        // this half of D1 has been read: GEMM2 may overwrite it
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(h_full);
        }
      }
      // ---- EPI2 share: D2 -> bias, + skip -> stream / operand out
      uint64_t kb[4], ka[4], kib[4];                     // index 2 * lane half + hi: channel cbase + 16 L + 8 hi + g
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ch = cbase + (i >> 1) * 16 + (i & 1) * 8 + g;
        kb[i] = dup(__ldg(p.bias1 + ch));
        ka[i] = has_snake ? dup(__ldg(p.sn_a + ch)) : 0ull;
        kib[i] = has_snake ? dup(__ldg(p.sn_inv_b + ch)) : 0ull;
      }
      ptx::mbar_wait_parked(d2h_full, d2f_ph);           // rows 0..127 first: GEMM2 of half 1 is issued later
      ptx::tc_fence_after();
#pragma unroll 1
      for (int item = sub; item < 16; item += 4) {
        const int r0 = q0 + item * 16;
        if (item == sub + 8) {                             // rows 128..255
          ptx::mbar_wait_parked(d2_full, d2f_ph);
          ptx::tc_fence_after();
        }
        if (ptx::elect_one()) {
          // every store issued so far has read its shared-memory source: the other stream slot and the operand
          // block are free again; fetch the NEXT item's skip block into the other slot
          ptx::bulk_wait_read<0>();
          if (item + 4 < 16) issue_skip(b, q0, item + 4, slot ^ 1);
          else if (ntile < p.total_tiles) issue_skip(nb, nq0, sub, slot ^ 1);
        }
        uint32_t r[16], sk[8];
        __syncwarp();
        const uint32_t t2 = tmem_base + boff + (static_cast<uint32_t>(cbase) << 16) + item * 16;
        ptx::tmem_ld_16x256b_x2(t2, r);
        ptx::tmem_ld_16x256b_x2(t2 + (16u << 16), r + 8);
        const uint32_t rb = ring_lane + slot * kRuActBlk;
        ptx::mbar_wait_parked(&my_res_full[slot], (res_ph >> slot) & 1u);
        ptx::ldmatrix_x4_trans(rb, sk[0], sk[1], sk[2], sk[3]);
        ptx::ldmatrix_x4_trans(rb ^ 32u, sk[4], sk[5], sk[6], sk[7]);
        res_ph ^= (1u << slot);
        ptx::tmem_ld_wait();
        uint64_t v[8];                                     // q = 4 L + 2 n + hi
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float2 sf = __half22float2(*reinterpret_cast<const __half2*>(&sk[q]));
          v[q] = ptx::f2_add(ptx::f2_add(ptx::f2_pack_u(r[2 * q], r[2 * q + 1]), kb[(q >> 2) * 2 + (q & 1)]),
                             ptx::f2_pack(sf.x, sf.y));
        }
        if (p.raw_out) {
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
        if (p.act_out) {
          uint32_t w[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float y0, y1;
            if (has_snake) {
              const int ci = (q >> 2) * 2 + (q & 1);
              float t0, t1;
              ptx::f2_unpack(ptx::f2_mul(v[q], ka[ci]), t0, t1);
              const uint64_t sn = ptx::f2_pack(sin_fast(t0), sin_fast(t1));
              ptx::f2_unpack(ptx::f2_fma(ptx::f2_mul(kib[ci], sn), sn, v[q]), y0, y1);
            } else {
              ptx::f2_unpack(v[q], y0, y1);
            }
            if (p.act_f16) {
              w[q] = ptx::f2h2_sat(y0, y1);
            } else {
              const __nv_bfloat162 h2 = __floats2bfloat162_rn(y0, y1);
              w[q] = *reinterpret_cast<const uint32_t*>(&h2);
            }
          }
          ptx::stmatrix_x4_trans(ablk_lane, w[0], w[1], w[2], w[3]);
          ptx::stmatrix_x4_trans(ablk_lane ^ 32u, w[4], w[5], w[6], w[7]);
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (ptx::elect_one()) {
          uint8_t* const rblk = ring + slot * kRuActBlk;
          if (p.raw_out) ptx::tma_store_4d(&tmR, rblk, cbase, 0, r0, b);
          if (p.act_out) ptx::tma_store_4d(&tmO, ablk, cbase, 0, r0, b);
          ptx::bulk_commit();
        }
        slot ^= 1;
      }
      d2f_ph ^= 1u;
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&buf_empty[it & 1]);   // GEMM1 of tile it + 2 may reuse this accumulator
    }
    if (lane == 0) ptx::bulk_wait<0>();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}

}  // namespace kvae
