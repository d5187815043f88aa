// The two thin convolutions at the waveform boundary of the Oobleck stack.  They hold < 0.3 % of the
// FLOPs but touch the longest tensors, and their channel counts (io_channels = 1 or 2) do not fit a
// tensor-core tile, so they get HBM-streaming CUDA-core kernels of their own:
//   conv_wave_out_kernel  decoder tail: SnakeBeta -> Conv1d(C -> io, k7, pad 3, bias=False) [-> tanh]
//                         (autoencoders.py:183-185); reads the fp32 residual stream [B, T, C], applies
//                         SnakeBeta once per staged element in fp32, accumulates in fp32 and writes the
//                         waveform directly in the API layout [B, io, T].  Keeping this layer in fp32
//                         removes what SURVEY.md (H1) measured as half of the bf16 error budget.
//   conv_wave_in_kernel   encoder head: Conv1d(io -> C, k7, pad 3) (autoencoders.py:133); reads the waveform
//                         in the API layout and writes the fp32 residual stream plus the SnakeBeta-activated
//                         bf16 operand of the first ResidualUnit, both channels-last.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "conv_common.cuh"  // snake_beta
#include "elementwise.cuh"  // ld_elem / st_elem
#include "ptx.cuh"

namespace kvae {

struct WaveOutParams {
  const float* x;         // [B, T, Cin] fp32 residual stream
  const float* pro_a;     // SnakeBeta exp(alpha) [Cin]
  const float* pro_inv_b;
  const float* w;         // [7][Cin][COUT] fp32
  void* y;                // [B, COUT, T]
  int y_f32;
  int T, Cin, tanh_out;
  int B, tiles_per_clip, total_tiles;
  int precise;            // fp32 mode: range-reduced sine (<= 1e-5 budget) instead of the plain MUFU approximation
  // input geometry (a whole clip: T_in = T, in_row0 = -3, x_pitch = T; the streaming decoder passes a window buffer):
  // output t reads input rows t + in_row0 .. t + in_row0 + 6, rows outside [0, T_in) are the conv's zero padding
  int T_in, in_row0;
  long long x_pitch;      // rows between clips in x
};

constexpr int kWaveOutTile = 128;              // outputs per tile
constexpr int kWaveOutRows = kWaveOutTile + 6; // staged input rows per tile
constexpr int kWaveOutBufs = 3;

inline size_t wave_out_smem(int Cin) {
  return 1024 + static_cast<size_t>(kWaveOutBufs) * kWaveOutRows * Cin * sizeof(float);
}

// Persistent HBM-streaming kernel: one CTA per SM walks over 128-sample output tiles.  The 134 input rows a
// tile needs are CONTIGUOUS in the channels-last stream, so a producer thread fetches them with bulk async
// copies into a 3-deep shared-memory ring (mbarrier full/empty), keeping ~130 KB per SM in flight; 8 compute
// warps each own 16 outputs: lane l holds channels 4l..4l+3 (one conflict-free 16-byte shared load per row),
// keeps a 7-row register window with SnakeBeta applied once per loaded element, keeps its 7x4xCOUT weights in
// registers, and the 32 lanes' partial sums are combined by a transposing butterfly (31 shuffles per 32 sums).
// Requires Cin == 128.  grid = min(tiles, #SM), block = 288 (8 compute warps + 1 producer warp).
template <int COUT>
__global__ void __launch_bounds__(288, 1) conv_wave_out_kernel(const WaveOutParams p) {
  constexpr int TT = kWaveOutTile, RS = kWaveOutRows, NB = kWaveOutBufs, CIN = 128;
  extern __shared__ uint8_t sm_wo_raw[];
  const uint32_t raw_addr = ptx::smem_u32(sm_wo_raw);
  uint8_t* smem = sm_wo_raw + (((raw_addr + 127u) & ~127u) - raw_addr);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  uint64_t* empty = full + NB;
  float* ring = reinterpret_cast<float*>(smem + 128);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < NB; ++i) { ptx::mbar_init(&full[i], 1); ptx::mbar_init(&empty[i], 8); }
    ptx::fence_mbar_init();
  }
  __syncthreads();

  if (warp == 8) {
    // ---------------------------------------------------------- producer
    if (lane == 0) {
      int buf = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int b = tile / p.tiles_per_clip;
        const int t0 = (tile % p.tiles_per_clip) * TT;
        const int r_lo = max(0, -(t0 + p.in_row0));             // first staged row that exists
        const int r_hi = max(r_lo, min(RS, p.T_in - (t0 + p.in_row0)));   // one past the last
        ptx::mbar_wait(&empty[buf], ph ^ 1u);
        if (r_hi == r_lo) {                                    // nothing to fetch (cannot happen for a tile with outputs)
          ptx::mbar_arrive(&full[buf]);
          if (++buf == NB) { buf = 0; ph ^= 1u; }
          continue;
        }
        ptx::mbar_expect_tx(&full[buf], static_cast<uint32_t>(r_hi - r_lo) * CIN * 4);
        const float* src = p.x + (static_cast<size_t>(b) * p.x_pitch + (t0 + p.in_row0 + r_lo)) * CIN;
        float* dst = ring + static_cast<size_t>(buf) * RS * CIN + r_lo * CIN;
        for (int r = r_lo; r < r_hi; r += 32) {
          const int n = min(32, r_hi - r);
          ptx::bulk_load_1d(dst, src, static_cast<uint32_t>(n) * CIN * 4, &full[buf]);
          dst += 32 * CIN;
          src += 32 * CIN;
        }
        if (++buf == NB) { buf = 0; ph ^= 1u; }
      }
    }
    return;
  }

  // ------------------------------------------------------------ compute warps
  float w[7][4][COUT];
#pragma unroll
  for (int k = 0; k < 7; ++k)
#pragma unroll
    for (int e = 0; e < 4; ++e)
#pragma unroll
      for (int c = 0; c < COUT; ++c) w[k][e][c] = __ldg(p.w + (static_cast<size_t>(k) * CIN + 4 * lane + e) * COUT + c);
  const float4 sa = __ldg(reinterpret_cast<const float4*>(p.pro_a + 4 * lane));
  const float4 sib = __ldg(reinterpret_cast<const float4*>(p.pro_inv_b + 4 * lane));
  int buf = 0;
  uint32_t ph = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const int b = tile / p.tiles_per_clip;
    const int t0 = (tile % p.tiles_per_clip) * TT;
    ptx::mbar_wait(&full[buf], ph);
    const float* tile_s = ring + static_cast<size_t>(buf) * RS * CIN + 4 * lane;
    auto load_row = [&](int r) -> float4 {   // staged row r <-> input row t0 + in_row0 + r; zero outside (conv padding)
      const int t = t0 + p.in_row0 + r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t >= 0 && t < p.T_in) {
        v = *reinterpret_cast<const float4*>(tile_s + r * CIN);
        if (p.precise) {
          v.x = snake_beta_rr(v.x, sa.x, sib.x); v.y = snake_beta_rr(v.y, sa.y, sib.y);
          v.z = snake_beta_rr(v.z, sa.z, sib.z); v.w = snake_beta_rr(v.w, sa.w, sib.w);
        } else {
          v.x = snake_beta<true>(v.x, sa.x, sib.x); v.y = snake_beta<true>(v.y, sa.y, sib.y);
          v.z = snake_beta<true>(v.z, sa.z, sib.z); v.w = snake_beta<true>(v.w, sa.w, sib.w);
        }
      }
      return v;
    };
    const int o0 = warp * 16;                 // this warp's first output inside the tile
    // Row-major accumulation: each staged row (SnakeBeta applied once) feeds the 7 outputs whose windows
    // contain it, so the 56 FMAs per row go to 14 independent accumulators -- no long dependent chains.
    float acc[16 * COUT];
#pragma unroll
    for (int i = 0; i < 16 * COUT; ++i) acc[i] = 0.f;
#pragma unroll
    for (int r = 0; r < 22; ++r) {
      const float4 x = load_row(o0 + r);
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        const int o = r - k;                  // output (inside this warp's 16) whose tap k reads row r
        if (o >= 0 && o < 16) {
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            float a = acc[c * 16 + o];
            a = fmaf(x.x, w[k][0][c], a);
            a = fmaf(x.y, w[k][1][c], a);
            a = fmaf(x.z, w[k][2][c], a);
            a = fmaf(x.w, w[k][3][c], a);
            acc[c * 16 + o] = a;
          }
        }
      }
    }
    // this warp no longer reads the staged tile
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&empty[buf]);
    if (++buf == NB) { buf = 0; ph ^= 1u; }
    // transposing butterfly: afterwards lane L holds the sum over all lanes of acc[L % (16*COUT)]
    constexpr int NV = 16 * COUT;             // 16 or 32 values
#pragma unroll
    for (int s = NV / 2; s >= 1; s >>= 1) {
#pragma unroll
      for (int i = 0; i < s; ++i) {
        const bool up = (lane & s) != 0;
        const float send = up ? acc[i] : acc[i + s];
        const float keep = up ? acc[i + s] : acc[i];
        acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
      }
    }
    float total = acc[0];
    if (COUT == 1) total += __shfl_xor_sync(0xffffffffu, total, 16);   // 16 values: the two half-warps hold halves
    const int idx = lane & (NV - 1);
    const int c = idx / 16, o = idx % 16;
    const int t = t0 + o0 + o;
    if (t < p.T && (COUT == 2 || lane < 16)) {
      if (p.tanh_out) total = tanhf(total);
      st_elem(p.y, (static_cast<size_t>(b) * COUT + c) * p.T + t, p.y_f32, total);
    }
  }
}

// ---------------------------------------------------------------- decoder tail on the tensor cores (TF32)
// Same layer as conv_wave_out_kernel.  On the CUDA cores it needs 1792 FMAs per output sample and ran at ~30 % of
// HBM speed.  Here the channel contraction is ONE small tcgen05 kind::tf32 GEMM per tile and the 7 taps are summed
// afterwards:   P[t, (k, co)] = sum_ci SnakeBeta(x)[t, ci] * w[k][ci][co]      (M = 128 rows, N = 16 >= 7*io, K = 128)
//               y[t, co]      = sum_k P[t + k - 3, (k, co)]
// so every staged element is read by the tensor core exactly once (a first version that used row-shifted
// descriptors per tap re-read the tile 7 times and was bound by the shared-memory port).
//   * warp 0 (TMA) streams the fp32 residual stream tile [128 rows x 128 ch] as four 32-channel boxes
//     (SWIZZLE_128B: one 128-byte line = 32 floats = one K-major tf32 operand row) into a 3-slot ring;
//   * warps 4-19 apply SnakeBeta IN PLACE on the staged tile (element-wise, so the swizzle is irrelevant; the
//     channel of a 16-byte unit is recovered from its position), round to tf32 (cvt.rna) and hand the slot to the
//     MMA warp through fence.proxy.async + mbarrier;
//   * warp 1 issues 4 chunks x 4 K-steps MMAs of 128 x 16 x 8; the weights [4][16 x 32] stay in shared memory;
//   * warps 20-23 move P (TMEM lane = row) to shared memory, sum the taps of the 122 outputs whose windows lie
//     inside the tile and write [B, io, T] directly, coalesced.
// The stream stays fp32 in HBM and the accumulation fp32; only the operands are rounded to tf32 (11 significant
// bits), ~4x finer than the bf16 operands of every other conv in the stack.
struct WaveOutTcParams {
  const float* pro_a;       // SnakeBeta exp(alpha) [128]
  const float* pro_inv_b;
  const float* w;           // [7][128][COUT] fp32
  void* y;                  // [B, COUT, T]
  int y_f32;
  int T, B, COUT, tanh_out;
  int tiles_per_clip, total_tiles;
  int in_row0;              // output t reads input rows t + in_row0 .. +6 of tmX (-3 for a whole clip)
  int preact;               // kF16 only: tmX maps SnakeBeta(x) already in fp16 (written by the last ResidualUnit's epilogue):
                            // no transform stage, the MMAs read the tile as it lands
  unsigned int* peak_bits;  // nullptr, or: atomicMax of the bit pattern of |y| over everything written (phase 1 of the
                            // peak-normalised int16 conversion, infer_0828_sigma.py:298) -- one atomic per warp and tile
};

// kF16 = true: the residual stream is fp16 in HBM (inference plans).  The tile is then two 64-channel chunks of
// 128-byte rows, SnakeBeta is applied in fp32 and written back as fp16, and the GEMM is kind::f16 (fp16 x fp16 ->
// fp32; 11 significant bits like tf32) with K = 16 per instruction.
constexpr int kWoTcRows = 128;                       // staged rows per tile
constexpr int kWoTcTile = kWoTcRows - 6;             // outputs per tile (k7: 3 halo rows each side)
constexpr int kWoTcChunk = kWoTcRows * 128;          // bytes of one chunk (32 fp32 or 64 fp16 channels)
constexpr int kWoTcSlots = 3;
constexpr int kWoTcPStride = 17;                     // floats per P row in shared memory (conflict-free)
constexpr int kWoTcThreads = 768;                   // warps 0-2 control, 4-19 SnakeBeta transform, 20-23 epilogue
template <bool kF16> struct WoTc {
  static constexpr int kChunks = kF16 ? 2 : 4;
  static constexpr int kSlab = kChunks * kWoTcChunk;             // 32768 / 65536 B
  static constexpr int kWBytes = kChunks * 16 * 128;             // weights [chunk][16 rows x 128 B]
};

template <bool kF16>
inline size_t wave_out_tc_smem() {
  return 1024 + 1024 + kWoTcSlots * WoTc<kF16>::kSlab + WoTc<kF16>::kWBytes + 1024 + 2 * kWoTcRows * kWoTcPStride * 4;
}

template <bool kF16>
__global__ void __launch_bounds__(kWoTcThreads, 1)
conv_wave_out_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ WaveOutTcParams p) {
  constexpr int kWoTcSlab = WoTc<kF16>::kSlab, kWoTcWBytes = WoTc<kF16>::kWBytes, kChunks = WoTc<kF16>::kChunks;
  extern __shared__ uint8_t sm_wotc_raw[];
  const uint32_t raw_addr = ptx::smem_u32(sm_wotc_raw);
  uint8_t* smem = sm_wotc_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);      // [3] TMA landed
  uint64_t* ready = full + 4;                               // [3] SnakeBeta applied (8 warps)
  uint64_t* empty = full + 8;                               // [3] MMAs done reading the slot
  uint64_t* acc_full = full + 12;                           // [2]
  uint64_t* acc_empty = full + 14;                          // [2] (4 epilogue warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full + 16);
  uint8_t* ring = smem + 1024;
  uint8_t* wsm = ring + kWoTcSlots * kWoTcSlab;
  float* tab = reinterpret_cast<float*>(wsm + kWoTcWBytes);   // [128] a, [128] inv_b
  float* pbuf = tab + 256;                                    // [2][128][17]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmX);
    for (int i = 0; i < kWoTcSlots; ++i) { ptx::mbar_init(&full[i], 1); ptx::mbar_init(&ready[i], 16); ptx::mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 4); }
    ptx::fence_mbar_init();
  }
  ptx::pdl_launch_dependents();
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 32);
    ptx::tmem_relinquish();
  }
  // weights -> K-major SWIZZLE_128B tiles [chunk][16 rows n = k*COUT + co (zero-padded)][32 floats | 64 halves]
  for (int i = threadIdx.x; i < 16 * 128; i += kWoTcThreads) {
    const int ci = i & 127, n = i >> 7;               // input channel, GEMM column
    float v = 0.f;
    if (n < 7 * p.COUT) {
      const int k = n / p.COUT, co = n % p.COUT;
      v = __ldg(p.w + (static_cast<size_t>(k) * 128 + ci) * p.COUT + co);
    }
    if (kF16) {
      const int c = ci >> 6, cc = ci & 63;
      *reinterpret_cast<__half*>(wsm + c * 2048 + n * 128 + (((cc >> 3) ^ (n & 7)) << 4) + (cc & 7) * 2) = __float2half_rn(v);
    } else {
      const int c = ci >> 5, cc = ci & 31;
      *reinterpret_cast<float*>(wsm + c * 2048 + n * 128 + (((cc >> 2) ^ (n & 7)) << 4) + (cc & 3) * 4) = ptx::round_tf32(v);
    }
  }
  if (threadIdx.x < 128) {
    tab[threadIdx.x] = __ldg(p.pro_a + threadIdx.x);
    tab[128 + threadIdx.x] = __ldg(p.pro_inv_b + threadIdx.x);
  }
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  ptx::pdl_wait();                 // the weight / table staging above reads constants only
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (ptx::elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        const int b = tile / p.tiles_per_clip;
        const int t0 = (tile % p.tiles_per_clip) * kWoTcTile;
        ptx::mbar_wait(&empty[s], ph ^ 1u);
        ptx::mbar_expect_tx(&full[s], kWoTcSlab);
        for (int c = 0; c < kChunks; ++c)
          ptx::tma_load_4d(ring + s * kWoTcSlab + c * kWoTcChunk, &tmX, &full[s], c * (kF16 ? 64 : 32), 0, t0 + p.in_row0, b);
        if (++s == kWoTcSlots) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      const uint32_t idesc = kF16 ? ptx::idesc_f16_f32(128, 16) : ptx::idesc_tf32_f32(128, 16);
      const uint64_t desc_hi = (static_cast<uint64_t>(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      const uint32_t ring_lo = ((ptx::smem_u32(ring) & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t w_lo = ((ptx::smem_u32(wsm) & 0x3FFFFu) >> 4) | (1u << 16);
      int s = 0, a = 0;
      uint32_t ph = 0, aph = 0;
      for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
        ptx::mbar_wait(p.preact ? &full[s] : &ready[s], ph);
        ptx::mbar_wait(&acc_empty[a], aph ^ 1u);
        ptx::tc_fence_after();
        const uint32_t d = tmem_base + a * 16;
#pragma unroll
        for (int c = 0; c < kChunks; ++c) {
          const uint32_t al = ring_lo + ((s * kWoTcSlab + c * kWoTcChunk) >> 4);
          const uint32_t bl = w_lo + ((c * 2048) >> 4);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {                       // 8 tf32 / 16 fp16 = 32 B per K-step
            if (kF16) ptx::umma_f16(d, desc_hi | (al + 2 * ks), desc_hi | (bl + 2 * ks), idesc, (c | ks) ? 1u : 0u);
            else ptx::umma_tf32(d, desc_hi | (al + 2 * ks), desc_hi | (bl + 2 * ks), idesc, (c | ks) ? 1u : 0u);
          }
        }
        ptx::umma_commit(&empty[s]);
        ptx::umma_commit(&acc_full[a]);
        if (++s == kWoTcSlots) { s = 0; ph ^= 1u; }
        if (++a == 2) { a = 0; aph ^= 1u; }
      }
    }
  } else if (warp >= 4 && warp < 20 && !p.preact) {
    // ------------------------------------------------------------ SnakeBeta in place on the staged tile
    const int tid = threadIdx.x - 128;                    // 0..511
    // A thread's 16-byte units are tid + 512*i: the same position inside a row and the same row phase (row & 7)
    // for every i, so the channels it touches are fixed -- chunk i/2, group g -- and their SnakeBeta constants
    // live in registers (a table lookup per element made this stage issue-bound).
    constexpr int kPer = kF16 ? 8 : 4;                    // channels per 16-byte unit
    constexpr int kChunkCh = kF16 ? 64 : 32;
    const int g = (tid & 7) ^ ((tid >> 3) & 7);
    float ca[kChunks][kPer], cb[kChunks][kPer];
#pragma unroll
    for (int c = 0; c < kChunks; ++c)
#pragma unroll
      for (int e = 0; e < kPer; ++e) {
        ca[c][e] = tab[c * kChunkCh + g * kPer + e];
        cb[c][e] = tab[128 + c * kChunkCh + g * kPer + e];
      }
    int s = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      ptx::mbar_wait(&full[s], ph);
      float4* slab = reinterpret_cast<float4*>(ring + s * kWoTcSlab);
#pragma unroll
      for (int i = 0; i < 2 * kChunks; ++i) {              // kChunks * 128 rows * 8 units / 512 threads
        const int u = tid + 512 * i;
        const int c = i >> 1;
        float4 q = slab[u];
        if (kF16) {
          __half2* h2 = reinterpret_cast<__half2*>(&q);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float2 f = __half22float2(h2[e]);
            f.x = snake_beta<true>(f.x, ca[c][2 * e], cb[c][2 * e]);
            f.y = snake_beta<true>(f.y, ca[c][2 * e + 1], cb[c][2 * e + 1]);
            reinterpret_cast<uint32_t*>(h2)[e] = ptx::f2h2_sat(f.x, f.y);
          }
        } else {
          q.x = ptx::round_tf32(snake_beta<true>(q.x, ca[c][0], cb[c][0]));
          q.y = ptx::round_tf32(snake_beta<true>(q.y, ca[c][1], cb[c][1]));
          q.z = ptx::round_tf32(snake_beta<true>(q.z, ca[c][2], cb[c][2]));
          q.w = ptx::round_tf32(snake_beta<true>(q.w, ca[c][3], cb[c][3]));
        }
        slab[u] = q;
      }
      ptx::fence_proxy_async();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&ready[s]);
      if (++s == kWoTcSlots) { s = 0; ph ^= 1u; }
    }
  } else if (warp >= 20) {
    // ------------------------------------------------------------ P -> shared memory -> tap sum -> [B, io, T]
    const int quad = warp & 3;
    const int i = quad * 32 + lane;                      // row of the tile / output index
    int a = 0;
    uint32_t aph = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const int b = tile / p.tiles_per_clip;
      const int t = (tile % p.tiles_per_clip) * kWoTcTile + i;
      ptx::mbar_wait(&acc_full[a], aph);
      ptx::tc_fence_after();
      uint32_t r[16];
      ptx::tmem_ld_32x16(tmem_base + a * 16 + (static_cast<uint32_t>(quad * 32) << 16), r);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      float* pb = pbuf + a * kWoTcRows * kWoTcPStride;
#pragma unroll
      for (int j = 0; j < 16; ++j) pb[i * kWoTcPStride + j] = __uint_as_float(r[j]);
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[a]);
      ptx::named_bar_sync(1, 128);                       // all 128 rows of P are in shared memory
      float peak = 0.f;
      if (i < kWoTcTile && t < p.T) {
        for (int co = 0; co < p.COUT; ++co) {
          float v = 0.f;
#pragma unroll
          for (int k = 0; k < 7; ++k) v += pb[(i + k) * kWoTcPStride + k * p.COUT + co];
          if (p.tanh_out) v = tanhf(v);
          st_elem(p.y, (static_cast<size_t>(b) * p.COUT + co) * p.T + t, p.y_f32, v);
          // the peak of what a reader of y sees: the value rounded to the output dtype
          peak = fmaxf(peak, fabsf(p.y_f32 ? v : __bfloat162float(__float2bfloat16(v))));
        }
      }
      if (p.peak_bits) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) peak = fmaxf(peak, __shfl_xor_sync(0xffffffffu, peak, o));
        if (lane == 0 && peak > 0.f) atomicMax(p.peak_bits, __float_as_uint(peak));
      }
      if (++a == 2) { a = 0; aph ^= 1u; }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 32);
}

struct WaveInParams {
  const void* x;          // [B, CIN, T]
  int x_f32;
  const float* w;         // [7][CIN][Cout] fp32
  const float* bias;      // [Cout]
  void* out_raw;          // [B, T, Cout] fp32 (or fp16 when raw_f16) or nullptr
  int raw_f16;
  int precise;            // fp32 mode: range-reduced sine
  int act_split;          // fp32 mode: out_act is [B, T, 2*Cout], bf16 (hi | lo) halves for the tensor-core consumer
  __nv_bfloat16* out_act; // [B, T, Cout] bf16 or nullptr
  const float* snake_a;   // epilogue SnakeBeta of the first ResidualUnit (or nullptr: plain cast)
  const float* snake_inv_b;
  int T, Cout;            // T: output rows
  // input geometry as in WaveOutParams (a whole clip: T_in = T, in_row0 = -3, x_pitch = T; the streaming encoder passes
  // its sample window): output t reads samples t + in_row0 .. t + in_row0 + 6, those outside [0, T_in) are zero padding
  int T_in, in_row0;
  long long x_pitch;      // samples between channel rows of x
  long long out_pitch;    // rows between clips in out_raw / out_act
};

constexpr int kWaveInTile = 64;

// grid (ceil(T/64), Cout/128, B), block 128: warp w handles rows w, w+4, ...; lane handles 4 out-channels.
template <int CIN>
__global__ void __launch_bounds__(128) conv_wave_in_kernel(const WaveInParams p) {
  constexpr int TT = kWaveInTile, RS = TT + 6;
  __shared__ float xs[CIN][RS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.z;
  const int t0 = blockIdx.x * TT;
  const int co = blockIdx.y * 128 + lane * 4;
  for (int i = threadIdx.x; i < CIN * RS; i += 128) {
    const int c = i / RS, r = i % RS;
    const int t = t0 + p.in_row0 + r;
    xs[c][r] = (t >= 0 && t < p.T_in) ? ld_elem(p.x, (static_cast<size_t>(b) * CIN + c) * p.x_pitch + t, p.x_f32) : 0.f;
  }
  float w[7][CIN][4];
#pragma unroll
  for (int k = 0; k < 7; ++k)
#pragma unroll
    for (int c = 0; c < CIN; ++c) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(p.w + (static_cast<size_t>(k) * CIN + c) * p.Cout + co));
      w[k][c][0] = v.x; w[k][c][1] = v.y; w[k][c][2] = v.z; w[k][c][3] = v.w;
    }
  const float4 bias = __ldg(reinterpret_cast<const float4*>(p.bias + co));
  float4 sa = make_float4(0.f, 0.f, 0.f, 0.f), sib = sa;
  if (p.snake_a) {
    sa = __ldg(reinterpret_cast<const float4*>(p.snake_a + co));
    sib = __ldg(reinterpret_cast<const float4*>(p.snake_inv_b + co));
  }
  __syncthreads();
  for (int r = warp; r < TT; r += 4) {
    const int t = t0 + r;
    if (t >= p.T) break;
    float v0 = bias.x, v1 = bias.y, v2 = bias.z, v3 = bias.w;
#pragma unroll
    for (int k = 0; k < 7; ++k)
#pragma unroll
      for (int c = 0; c < CIN; ++c) {
        const float xv = xs[c][r + k];
        v0 = fmaf(xv, w[k][c][0], v0); v1 = fmaf(xv, w[k][c][1], v1);
        v2 = fmaf(xv, w[k][c][2], v2); v3 = fmaf(xv, w[k][c][3], v3);
      }
    const size_t o = (static_cast<size_t>(b) * p.out_pitch + t) * p.Cout + co;
    if (p.out_raw) {
      if (p.raw_f16) {
        *reinterpret_cast<uint2*>(static_cast<__half*>(p.out_raw) + o) =
            make_uint2(ptx::f2h2_sat(v0, v1), ptx::f2h2_sat(v2, v3));
      } else {
        *reinterpret_cast<float4*>(static_cast<float*>(p.out_raw) + o) = make_float4(v0, v1, v2, v3);
      }
    }
    if (p.out_act) {
      if (p.snake_a) {
        if (p.precise) {
          v0 = snake_beta_rr(v0, sa.x, sib.x); v1 = snake_beta_rr(v1, sa.y, sib.y);
          v2 = snake_beta_rr(v2, sa.z, sib.z); v3 = snake_beta_rr(v3, sa.w, sib.w);
        } else {
          v0 = snake_beta<true>(v0, sa.x, sib.x); v1 = snake_beta<true>(v1, sa.y, sib.y);
          v2 = snake_beta<true>(v2, sa.z, sib.z); v3 = snake_beta<true>(v3, sa.w, sib.w);
        }
      }
      __nv_bfloat162 h0 = __floats2bfloat162_rn(v0, v1), h1 = __floats2bfloat162_rn(v2, v3);
      if (p.act_split) {
        const size_t o2 = (static_cast<size_t>(b) * p.out_pitch + t) * 2 * p.Cout + co;
        const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
        __nv_bfloat162 l0 = __floats2bfloat162_rn(v0 - f0.x, v1 - f0.y), l1 = __floats2bfloat162_rn(v2 - f1.x, v3 - f1.y);
        *reinterpret_cast<uint2*>(p.out_act + o2) =
            make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
        *reinterpret_cast<uint2*>(p.out_act + o2 + p.Cout) =
            make_uint2(*reinterpret_cast<uint32_t*>(&l0), *reinterpret_cast<uint32_t*>(&l1));
      } else {
        *reinterpret_cast<uint2*>(p.out_act + o) =
            make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
      }
    }
  }
}

// ---- encoder head on the tensor cores (bf16 mode, inference).  conv_wave_in_kernel issues 14 * CIN FMAs + SnakeBeta
// per output element on the CUDA cores and ran at 36 % of its HBM floor (1.55 ms per 16 x 442 368 rows).  The k = 7
// conv over CIN <= 2 channels is a K = 7 CIN <= 14 dot product per output, i.e. ONE tcgen05 K-chunk: this kernel writes
// the im2col rows as a channels-last bf16 operand [B, T, 64] and conv_umma2_kernel<1> runs the layer as a k = 1 conv
// with its usual epilogue (bias, fp16 stream, SnakeBeta -> bf16 operand).  Four 16-column blocks, column
// jj = tap * CIN + channel inside a block (jj >= 7 CIN: zero):
//   block 0  hi(x) x hi(w)      block 1  lo(x) x hi(w)      block 2  hi(x) x lo(w)      block 3  zero
// with hi = bf16 rounding and lo = bf16(v - hi): the product is exact to 2^-16 relative (the lo x lo term), far
// inside the bf16 rounding of the operand the layer writes.  Blocks past the im2col rows pack the weights
// [Cout][64] in the same column order, so the pair stays one launch ahead of the conv.
struct WaveInColParams {
  const void* x;          // [B, CIN, T]
  int x_f32;
  __nv_bfloat16* col;     // [B, T, 64]
  const float* w;         // [7][CIN][Cout] fp32 (folded weight-norm weights)
  __nv_bfloat16* wp;      // [Cout][64]
  int T, B, Cout, CIN;    // T: output rows
  int row_blocks;         // blocks that write im2col rows (kColRows rows each); the rest pack weights
  int T_in, in_row0;      // input geometry, as in WaveInParams
  long long x_pitch;
};

constexpr int kColRows = 512;   // im2col rows per block

__global__ void __launch_bounds__(256) wave_in_im2col_kernel(const WaveInColParams p) {
  const int n = 7 * p.CIN;
  if (static_cast<int>(blockIdx.x) >= p.row_blocks) {
    // weight pack: one thread per (out-channel, column)
    const int i = (blockIdx.x - p.row_blocks) * 256 + threadIdx.x;
    if (i < p.Cout * 64) {
      const int co = i >> 6, blk = (i >> 4) & 3, jj = i & 15;
      float v = 0.f;
      if (blk < 3 && jj < n) {
        const float wv = __ldg(p.w + static_cast<size_t>(jj) * p.Cout + co);
        const float hi = __bfloat162float(__float2bfloat16(wv));
        v = (blk < 2) ? hi : wv - hi;
      }
      p.wp[i] = __float2bfloat16(v);
    }
    return;
  }
  constexpr int RS = kColRows + 6;
  __shared__ float xs[3 * RS];     // channels 0 .. CIN-1, then a row of zeros for the padding columns
  const int tiles_per_clip = (p.T + kColRows - 1) / kColRows;
  const int b = blockIdx.x / tiles_per_clip, t0 = (blockIdx.x % tiles_per_clip) * kColRows;
  for (int i = threadIdx.x; i < (p.CIN + 1) * RS; i += 256) {
    const int c = i / RS, r = i - c * RS;
    const int t = t0 + p.in_row0 + r;
    xs[i] = (c < p.CIN && t >= 0 && t < p.T_in) ? ld_elem(p.x, (static_cast<size_t>(b) * p.CIN + c) * p.x_pitch + t, p.x_f32) : 0.f;
  }
  // two threads per row: thread h owns columns 8h .. 8h+7 of every block, i.e. 16 bytes of the hi block (written
  // twice), 16 bytes of the lo block and 16 bytes of zeros -- a lane pair writes 32 contiguous bytes per store
  const int h = threadIdx.x & 1;
  int off[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int jj = 8 * h + q, k = jj / p.CIN, c = jj - k * p.CIN;
    off[q] = jj < n ? c * RS + k : p.CIN * RS;
  }
  __syncthreads();
#pragma unroll
  for (int r = threadIdx.x >> 1; r < kColRows; r += 128) {
    const int t = t0 + r;
    if (t >= p.T) continue;
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float x0 = xs[off[2 * q] + r], x1 = xs[off[2 * q + 1] + r];
      const __nv_bfloat162 h2 = __floats2bfloat162_rn(x0, x1);
      const float2 hf = __bfloat1622float2(h2);
      const __nv_bfloat162 l2 = __floats2bfloat162_rn(x0 - hf.x, x1 - hf.y);
      hi[q] = *reinterpret_cast<const uint32_t*>(&h2);
      lo[q] = *reinterpret_cast<const uint32_t*>(&l2);
    }
    uint4* row = reinterpret_cast<uint4*>(p.col + (static_cast<size_t>(b) * p.T + t) * 64) + h;
    const uint4 hv = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    row[0] = hv;
    row[2] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    row[4] = hv;
    row[6] = make_uint4(0u, 0u, 0u, 0u);
  }
}

}  // namespace kvae
