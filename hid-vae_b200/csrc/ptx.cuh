// Thin inline-PTX wrappers for the sm_100a features the RQ kernels use: mbarrier, bulk TMA copies
// (cp.async.bulk), tcgen05 (TMEM alloc / mma / commit / ld) and the proxy fences between them.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace hv {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// The warp's index inside the CTA as a value the compiler KNOWS to be warp-uniform (a broadcast from lane 0).  With the plain
// threadIdx.x >> 5, every branch or loop bound derived from the warp index counts as divergent, and each warp-collective
// instruction below it (shfl.sync, vote, bar, tcgen05 .sync.aligned) gets a WARPSYNC.COLLECTIVE / ENDCOLLECTIVE pair, register
// moves and sometimes a duplicated code path (the row loop of the backward kernel shrank from 1376 to 872 instructions).
__device__ __forceinline__ int warp_index() { return __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0); }
__device__ __forceinline__ int uniform(int v) { return __shfl_sync(0xffffffffu, v, 0); }

// One lane of the (converged) warp: ptxas knows that a region guarded by elect.sync has a single active thread, so
// operands that must live in uniform registers (tcgen05.mma descriptors) need no per-value "waterfall" loop --
// unlike a region guarded by `lane == 0`.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier --------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Same probe with a suspend-time hint (ns): the warp stays parked until the phase completes or the time is up, instead
// of coming back after the short default interval and burning issue slots and load/store-pipe probes in a spin.
__device__ __forceinline__ bool mbar_try_wait_parked(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (mbarrier.try_wait may suspend the thread for a hardware-defined time before it answers; a
// scheduler that polls several barriers must not sleep on the first one that is not ready).
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// ---- shared-memory progress counters (cheap to poll: one LDS instead of a ~150-cycle mbarrier probe) -----------
__device__ __forceinline__ void counter_add_release(uint32_t addr, uint32_t v) {
  asm volatile("red.release.cta.shared::cta.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t counter_ld_acquire(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
// bounded spin until the counter reaches `need` (wrap-safe comparison)
__device__ __forceinline__ void counter_wait(uint32_t addr, uint32_t need) {
  if (static_cast<int32_t>(counter_ld_acquire(addr) - need) >= 0) return;
  const long long t0 = clock64();
  while (static_cast<int32_t>(counter_ld_acquire(addr) - need) < 0) {
    if (clock64() - t0 > 4000000000LL) {
      printf("hidvae_b200: counter wait timed out (block %d thread %d addr 0x%x need %u)\n", blockIdx.x, threadIdx.x, addr, need);
      __trap();
    }
  }
}

// Bounded wait: a protocol bug must end the kernel with an error, never hang the GPU (a hung box is a lost box).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_parked(bar, parity, 1000000u)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      printf("hidvae_b200: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", blockIdx.x,
             threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// ---- async-proxy fences and bulk TMA -----------------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (tcgen05.mma / TMA reading shared memory)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src_gmem), "r"(bytes), "r"(bar)
               : "memory");
}

// ---- Ampere-style asynchronous 16-byte copies global -> shared (generic proxy, L2 only), per-thread completion ----
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src_gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// ---- named barriers among a subset of the CTA's warps (id 1..15; id 0 is __syncthreads) ---------------------------
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// ask L2 to fetch `bytes` (multiple of 16) starting at the 16-byte aligned global address (SASS: UBLKPF)
__device__ __forceinline__ void bulk_prefetch_l2(const void* src_gmem, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}

// ---- register reallocation between warpgroups (all warps of a warpgroup execute it) ------------------------------
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, issued by ONE thread for the CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every tcgen05.mma previously issued by this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Same wait, but the 32 destination registers of the load are tied to the asm as in/out operands, so the compiler
// cannot schedule any use of them above the wait (a plain "memory" clobber orders memory, not registers).
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                 "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]),
                 "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]),
                 "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
               :
               : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives row (lane_base + i), columns [col, col+32)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                 "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}
// 32 lanes x 8 consecutive fp32 columns (the small shape lets a thread keep two loads in flight in 16 registers)
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
// wait for every outstanding tcgen05.ld of the thread; the registers of the load(s) that must be complete are tied to the
// asm so that no use of them is scheduled above the wait
__device__ __forceinline__ void tmem_wait_ld8(uint32_t (&v)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld8(uint32_t (&v)[8], uint32_t (&w)[8]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(w[0]),
                 "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7])
               :
               : "memory");
}
// registers -> tensor memory: 8 consecutive 32-bit columns of the thread's own lane
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
// registers -> tensor memory: thread i of the warp writes row (lane_base + i), 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
// registers -> tensor memory, 32 columns of the thread's own lane
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
      "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
      "r"(v[31])
      : "memory");
}
// 16 lanes x 32 columns in the mma-accumulator fragment layout (16x256b, four 8-column repeats): thread t receives, for
// repeat i, columns 8i + 2(t % 4) + {0, 1} of lane t / 4 in v[4i], v[4i + 1] and of lane t / 4 + 8 in v[4i + 2], v[4i + 3]
__device__ __forceinline__ void tmem_ld_16x256_x4(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]^T: the A operand (M rows = TMEM lanes, two bf16 per 32-bit column) in tensor memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// Shared-memory matrix descriptor, K-major, no swizzle ("interleave"): core matrix = 8 rows x 16 bytes stored
// as 128 contiguous bytes; LBO = byte distance between core matrices adjacent in K, SBO = byte distance between
// 8-row groups adjacent in M/N.  Bits: [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version = 1
// (sm_100), [61,64) layout type 0 = no swizzle.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;
  return d;
}
// The same descriptor split in its two 32-bit words, so that the issuing thread only adds to the low word:
//   lo = (addr >> 4) | (LBO >> 4) << 16,  hi = (SBO >> 4) | version 1 at bit 46 (bit 14 of the high word)
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr, uint32_t lbo_bytes) {
  return ((smem_addr >> 4) & 0x3FFFu) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__device__ __forceinline__ uint32_t umma_desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14); }
__device__ __forceinline__ uint64_t umma_desc(uint32_t lo, uint32_t hi) {
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
// Instruction descriptor for kind::f16: fp32 accumulate (bits [4,6) = 1), A/B = bf16 (bits [7,10), [10,13) = 1),
// both K-major (bits 15, 16 = 0), N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t m, uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

}  // namespace ptx
}  // namespace hv
