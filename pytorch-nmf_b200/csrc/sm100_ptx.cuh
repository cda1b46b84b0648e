// Thin inline-PTX wrappers for the sm_100a features the fused kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05.{alloc,mma,commit,ld,st,fence}, UMMA descriptors; and the host helpers
// that tc_nmf.cu and tc_nmfd.cu share (tensor maps, the wait-abort record).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace nmfb200 {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking probe of a phase (try_wait may suspend the thread until the phase completes or a time limit expires)
__device__ __forceinline__ bool mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes or the hint expires instead of
// returning after a few tens of cycles (CUTLASS passes the same 0x989680).  Unparked poll loops executed ~4 M try_wait per
// launch (ncu source page), a quarter of the SM's issue slots and avoidable power on a power-capped part.
__device__ __forceinline__ bool mbar_try_wait_parked(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(0x989680u)
      : "memory");
  return ok != 0;
}
// Bounded wait: on a protocol bug (no progress for ~1 s) the first waiter records (block, thread, barrier, parity)
// in g_wait_abort and every wait in the grid then falls through, so the kernel terminates instead of hanging
// the GPU box; the host checks the record after the launch (check_wait_abort below).
static __device__ unsigned int g_wait_abort[8];      // one record per translation unit (tc_nmf.cu, tc_nmfd.cu)
// Slow path of mbar_wait, out of line on purpose: the warp-specialised loops are latency-bound serial instruction
// streams (one MMA-issuing warp feeds the whole SM), so every wait site inlines only try_wait + a predicated call.
// The poll loop touches nothing but the barrier; the watchdog (clock, abort flag in global memory) is looked at once
// per 1024 failed polls -- a global load per poll costs an L2 round trip under a saturated memory system and shows up
// as microseconds of wake-up latency at every hand-off.
static __device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  uint32_t polls = 0;
  long long t0 = 0;
  while (!mbar_try_wait_parked(bar, parity)) {      // parked polls: +1 % sustained at cfg2 (power-capped part), nothing in a burst
    if ((++polls & 1023u) != 0u) continue;
    if (*reinterpret_cast<volatile unsigned int*>(&g_wait_abort[0]) != 0u) return;
    const long long now = clock64();
    if (t0 == 0) { t0 = now; continue; }
    if (now - t0 > 20000000000LL) {      // ~10 s of SM clocks: far beyond any time-slice or profiler replay (ADVICE r1)
      if (atomicCAS(&g_wait_abort[0], 0u, 1u) == 0u) {
        g_wait_abort[1] = blockIdx.x; g_wait_abort[2] = threadIdx.x; g_wait_abort[3] = bar; g_wait_abort[4] = parity;
        __threadfence();
      }
      return;
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity);
}

// ---- TMA ----------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint32_t bar, uint32_t dst, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(x), "r"(y)
      : "memory");
}

// ---- tcgen05 ------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// all previously issued tcgen05 async ops of this thread -> one arrive on `bar` when they complete
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets lane (base_lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// ---- UMMA descriptors (cute/arch/mma_sm100_desc.hpp bit layout) -----------------------------------
// shared-memory matrix descriptor, SWIZZLE_128B: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout_type=2 [61,64)
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// instruction descriptor for kind::f16: fp16 A/B, fp32 accumulate
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4)                       // c_format = F32
         | (0u << 7) | (0u << 10)        // a_format = b_format = F16
         | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16)
         | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// descriptor split into a loop-invariant high word and a low word that only carries the start address, so the
// issue loop advances operands with one 32-bit add (saddr < 256 KB: (saddr >> 4) never carries into the LBO field)
__device__ __forceinline__ constexpr uint32_t smem_desc_hi_sw128(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);
}
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16);
}
__device__ __forceinline__ uint64_t make_desc(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }

// one lane of a fully converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---- small math helpers ----------------------------------------------------------------------------
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// ---- packed fp32 pairs (sm_100: FFMA2 / FMUL2, two fp32 lanes per 64-bit register pair and per issue slot) ---------
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
  return d;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// {lo, hi} fp32 -> packed f16x2 (lo in bits 0-15), round-to-nearest, saturating to the largest finite half
__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

// ---- host side ------------------------------------------------------------------------------------------
// After a stream synchronise: report (to stderr, after `label`) and clear the wait-abort record of the translation unit this
// is compiled into.  1: one of its kernels aborted a wait since the last check; 0: none did; -1: the record is unreadable.
static inline int check_wait_abort(const char* label) {
  unsigned int h[8] = {0};
  if (cudaMemcpyFromSymbol(h, g_wait_abort, sizeof(h)) != cudaSuccess) return -1;
  if (!h[0]) return 0;
  fprintf(stderr, "nmf_b200: %smbarrier wait aborted: block %u thread %u (warp %u) bar_addr %u parity %u\n", label, h[1], h[2],
          h[2] / 32, h[3], h[4]);
  const unsigned int z[8] = {0};
  cudaMemcpyToSymbol(g_wait_abort, z, sizeof(z));
  return 1;
}

}  // namespace ptx

// 2-D fp16 row-major tensor map (rows x cols, row pitch ld elements), box 64 cols x box_rows rows, SWIZZLE_128B (tc_nmf.cu)
int make_tmap(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows);

}  // namespace nmfb200
