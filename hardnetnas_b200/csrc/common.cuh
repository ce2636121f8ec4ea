// Thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM).
// Everything here is device-side plumbing shared by the conv / head / distance kernels.
#pragma once

#include <cuda.h>          // CUtensorMap (types only; the driver entry point is resolved at run time)
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace hn {

// ------------------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a fully converged warp (warp-uniform callers only).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// {a, b, c, d} -> four e4m3 bytes (a lowest), round to nearest even like torch's .to(torch.float8_e4m3fn), two
// F2FP.SATFINITE.E4M3 instructions. Unit descriptors never reach the saturation bound (448).
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
  return static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16);
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug must surface as a trapped launch (error code on the host), never as a
// hung GPU. 4 s is far beyond any legitimate wait in these kernels.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023u) == 0 && globaltimer_ns() - t0 > 4000000000ull) {
      printf("hardnet_b200: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n",
             blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ------------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                            int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                            int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(bar), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}

// Tensor-map shared -> global store (bulk group completion): the box at `src` (laid out in the map's swizzle) is written
// to coordinates (c0, c1); parts outside the tensor are clipped.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}

// Bulk (non-tensor) shared -> global store through the async proxy: one thread moves a contiguous block.
__device__ __forceinline__ void bulk_store(void* gdst, uint32_t smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_src), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// Wait until all but the newest `N` committed bulk groups have finished READING their shared-memory source.
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation, UMMA issue/commit, TMEM loads
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
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

// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (fp16 or bf16 operands, fp32 accumulate).
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                         uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same instruction with the two 64-bit shared-memory descriptors given as (lo, hi) words. The issue loops keep the
// hi words (SBO, version, layout) as compile-time constants and advance only the lo word (start address >> 4, plus the
// constant LBO field), so stepping to the next operand tile is ONE 32-bit add instead of rebuilding a descriptor.
__device__ __forceinline__ void umma_f16_w(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f8f6f4 twin of umma_f16_w (UTCQMMA): one MMA takes K = 32 one-byte elements, i.e. the same 32 bytes of a K-major row
// as a K = 16 fp16 MMA, so the descriptors advance exactly as in the fp16 loops. The A / B format fields of the instruction
// descriptor are 0 for E4M3, so make_idesc_f16(m, n, 0) is also the E4M3 x E4M3 -> fp32 descriptor.
__device__ __forceinline__ void umma_f8_w(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// lo / hi words of the two descriptor flavours (see make_kmajor_desc below and make_noswizzle_desc in tc_conv.cuh)
__host__ __device__ constexpr uint32_t kmajor_desc_hi(uint32_t row_bytes) {
  return ((8u * row_bytes) >> 4) | (1u << 14) | ((row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u)) << 29);
}
__device__ __forceinline__ uint32_t kmajor_desc_lo(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }
__host__ __device__ constexpr uint32_t noswizzle_desc_hi(uint32_t sbo_bytes) { return (sbo_bytes >> 4) | (1u << 14); }
__device__ __forceinline__ uint32_t noswizzle_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16);
}

// Arrives (count 1) on the mbarrier once every previously issued tcgen05.mma of this thread retired.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}

// TMEM -> registers: lane (= accumulator row) per thread, `n` consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// UMMA descriptors (bit layouts as in the PTX ISA "matrix descriptor" / "instruction descriptor")
// ------------------------------------------------------------------------------------------------
// K-major operand tile in shared memory whose rows are `row_bytes` (64 or 128) wide and hardware-
// swizzled with the matching TMA mode; 8-row groups are packed back to back (SBO = 8 * row_bytes).
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4 (unused, =1)
//   bits [32,46) stride byte offset >> 4   bits [46,48) descriptor version (1 on sm_100)
//   bits [61,64) layout: 2 = 128B swizzle, 4 = 64B swizzle, 6 = 32B swizzle
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, uint32_t row_bytes) {
  const uint64_t layout = row_bytes == 128 ? 2ull : (row_bytes == 64 ? 4ull : 6ull);
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= 1ull << 16;
  d |= static_cast<uint64_t>((8u * row_bytes) >> 4) << 32;
  d |= 1ull << 46;
  d |= layout << 61;
  return d;
}

// kind::f16 instruction descriptor: fp32 accumulate, K-major A and B.
//   [4,6) D format (1 = f32)  [7,10) A format  [10,13) B format (0 = f16, 1 = bf16)
//   [15] A major  [16] B major (0 = K)  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(int m, int n, int fmt /*0 f16, 1 bf16*/) {
  return (1u << 4) | (static_cast<uint32_t>(fmt) << 7) | (static_cast<uint32_t>(fmt) << 10) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}

}  // namespace hn
