// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (TMEM alloc / UMMA / commit / ld).  Nothing here is generic CUDA; this header only
// compiles with -gencode arch=compute_100a,code=sm_100a.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace kvae {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Warp index broadcast from lane 0: ptxas then treats it (and everything derived from it -- staging addresses, TMA
// coordinates, loop counters) as warp-uniform and keeps it in uniform registers.  With a plain threadIdx.x >> 5 every
// TMA issue under `lane == 0` is wrapped in a per-operand R2UR waterfall loop (~25 instructions per issue).
__device__ __forceinline__ int warp_idx() {
  return __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .b32 rx;\n\t"
      ".reg .pred px;\n\t"
      "elect.sync rx|px, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, px;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- programmatic dependent launch
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start while its predecessor in the
// stream is still running: its CTAs are scheduled as soon as every CTA of the predecessor has executed
// pdl_launch_dependents() (or exited) and SMs are free, run their prologue (barrier init, TMEM allocation,
// tensor-map prefetch) and then block in pdl_wait() until the predecessor has completed and its writes are visible.
// With small batches (streaming decode: ~30 launches of 5-30 us per hop) the prologues and the launch latency of
// kernel N+1 disappear under the tail of kernel N.  Both are no-ops in a kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a protocol bug traps (-> cudaErrorLaunchFailure) instead of hanging the GPU box.
#ifndef KVAE_SPIN_LIMIT
#define KVAE_SPIN_LIMIT (1u << 26)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > KVAE_SPIN_LIMIT) {
      printf("kvae: mbarrier timeout block(%d,%d,%d) thread %d bar %p parity %u\n", blockIdx.x,
             blockIdx.y, blockIdx.z, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// Wait with a hardware suspend-time hint: the warp is parked by the barrier unit until the phase completes (or the
// hint, in ns, expires) instead of re-issuing try_wait + loop overhead -- with 16 epilogue warps per CTA the plain
// spin loops were a quarter of all issued instructions (profiles/r01_conv_ru_unified_epilogue_B16.ncu-rep).
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(20000u)
        : "memory");
    if (ok) return;
    if (++spins > (KVAE_SPIN_LIMIT >> 6)) {
      printf("kvae: mbarrier timeout (parked) block(%d,%d,%d) thread %d bar %p parity %u\n", blockIdx.x, blockIdx.y,
             blockIdx.z, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// Same, for warps that are not on the critical path (epilogues): back off between polls so that a dozen
// waiting warps do not eat the issue slots of the one thread that feeds the tensor core.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(40);
    if (++spins > (KVAE_SPIN_LIMIT >> 4)) {
      printf("kvae: mbarrier timeout (relaxed) block(%d,%d,%d) thread %d bar %p parity %u\n", blockIdx.x,
             blockIdx.y, blockIdx.z, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0,
                                            int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// L2 prefetch of a tensor-map box (no shared-memory destination): a later TMA load of the same box hits L2.
__device__ __forceinline__ void tma_prefetch_l2_4d(const CUtensorMap* m, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global [%0, {%1, %2, %3, %4}];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

// L2 prefetch of a contiguous global range (no shared-memory destination); address and size multiples of 16 B.
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<uint64_t>(src)), "r"(bytes) : "memory");
}

// 1-D bulk copy global -> shared (no tensor map): size and both addresses multiples of 16 B.
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// TMA store (shared -> global, bulk-group completion).  Rows/columns outside the tensor are clipped.
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2,
                                             int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T ; kind::f16 covers bf16/fp16 operands, fp32 accum.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same for fp32 operands read as TF32 (kind::tf32, K = 8 per instruction).
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// fp32 -> fp16 for the residual stream: round to nearest, SATURATING at +-65504 instead of overflowing to inf
// (a checkpoint with unusually large activations degrades gracefully instead of producing NaNs downstream)
__device__ __forceinline__ uint16_t f2h_sat(float x) {
  uint16_t r;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ uint32_t f2h2_sat(float lo, float hi) {   // {hi, lo} packed, lo in bits 0-15
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// round-to-nearest fp32 -> tf32 (the tensor core itself truncates)
__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
// Arrives (count 1) on `bar` once every tcgen05.mma issued so far by this thread has retired.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i <-> lane base+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 16 lanes x 256 bits, mma-accumulator-style fragments (PTX ISA "tcgen05 matrix fragments", .16x256b): for column
// group n (8 fp32 columns each), thread t holds  r[4n+0], r[4n+1] = lane base + t/4,     columns 8n + 2(t%4), +1
//                                                r[4n+2], r[4n+3] = lane base + t/4 + 8, same columns.
// A (column, column+1) pair converted to 16-bit and packed is exactly the ldmatrix/stmatrix .trans fragment, so a
// [lane = channel][column = time] accumulator goes to a [time][channel] shared-memory tile with 16-byte row stores.
__device__ __forceinline__ void tmem_ld_16x256b_x8(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x8.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t* r) {   // 32 columns -> 16 registers
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, uint32_t* r) {   // 16 columns -> 8 registers
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// Four 8x8 b16 matrices, transposed on the way: lane i supplies the address of (16-byte) row i%8 of matrix i/8;
// register j of thread t carries matrix j's elements (row 2(t%4), column t/4) in bits 0-15 and (row 2(t%4)+1,
// column t/4) in bits 16-31.
__device__ __forceinline__ void stmatrix_x4_trans(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(a), "r"(b),
               "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t saddr, uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(a), "=r"(b), "=r"(c), "=r"(d)
               : "r"(saddr)
               : "memory");
}
// Packed fp32 pairs (sm_100 FADD2 / FMUL2 / FFMA2): IEEE round-to-nearest per element, i.e. bit-identical to the
// scalar instructions at half the issue slots.
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ uint64_t f2_pack_u(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, K-major operand stored as rows of 128 B with the
// 128-byte swizzle (what a TMA box {64 bf16, R rows} with CU_TENSOR_MAP_SWIZZLE_128B writes):
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4 (unused here)
//   bits [32,46) stride byte offset >> 4 = 1024 B between 8-row groups
//   bits [46,48) version = 1 (sm_100)      bits [49,52) base offset
//   bits [61,64) layout type = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr, uint32_t base_offset) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(base_offset & 7u) << 49;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16: bf16 x bf16 -> fp32, both operands K-major.
//   [4,6) D format 1=f32   [7,10) A format 1=bf16   [10,13) B format 1=bf16
//   [15] A major 0=K  [16] B major 0=K   [17,23) N>>3   [24,29) M>>4
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// kind::f16 with fp16 (not bf16) operands, both K-major.
__host__ __device__ constexpr uint32_t idesc_f16_f32(int M, int N) {
  return (1u << 4) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}
// kind::tf32: tf32 x tf32 -> fp32, both operands K-major (rows of 32 floats = 128 B).
__host__ __device__ constexpr uint32_t idesc_tf32_f32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// Same with both operands MN-major (bits 15 / 16): the contraction dimension is the slow one in shared memory.
__host__ __device__ constexpr uint32_t idesc_bf16_f32_mn(int M, int N) {
  return idesc_bf16_f32(M, N) | (1u << 15) | (1u << 16);
}

// 16-byte vector reduction to global memory (fp32 x 4), address 16-byte aligned.
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

}  // namespace ptx
}  // namespace kvae
