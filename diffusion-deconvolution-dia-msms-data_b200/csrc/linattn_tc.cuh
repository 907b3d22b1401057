// tcgen05 / TMEM building blocks of the LinearAttention kernels (linattn_tc.cu), sm_100a only.
//
// Operand conventions (every one of them verified on a B200 by tools/tc_probe/tc_probe.cu, profiles/r2_tc_probe.log):
//   * shared-memory operands use the NO-SWIZZLE canonical layouts: core matrix = 8 rows x 16 bytes, stored contiguously
//     (128 B); descriptor LBO = byte distance between core matrices adjacent in K, SBO = between core matrices adjacent
//     in M / N.  K-major tf32 element (r, k):  (r % 8) * 16 + (r / 8) * SBO + (k / 4) * LBO + (k % 4) * 4
//                K-major bf16 element (r, k):  (r % 8) * 16 + (r / 8) * SBO + (k / 8) * LBO + (k % 8) * 2
//                MN-major bf16 element (m, k): (m % 8) * 2 + (k % 8) * 16 + (k / 8) * LBO + (m / 8) * SBO
//   * an A operand in TMEM (kind::tf32) is lane = row, column = k (one 32-bit column per element)
//   * accumulators: lane = row (M = 128), column = n
//   * an MMA that overwrites TMEM columns a previously issued MMA reads as its A operand must wait for that MMA
//     (tcgen05.commit -> mbarrier): the tensor pipe does NOT order that write-after-read (probe T4).
#pragma once
#include "common.cuh"

namespace dq {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
// Bounded wait: a protocol mistake must fail loudly instead of hanging the GPU.  The first waiter that times out
// (~0.15 s) records (code, block, thread, barrier address) in g_tc_err and every wait of the grid then falls through,
// so the kernel drains quickly; the host reads the record with dq_la_tc_last_error() and raises.
__device__ unsigned int g_tc_err[8];
__device__ unsigned int g_tc_dbg[32];   // per-warp (wait code << 24 | step) of the CTA that timed out first
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t code = 0, volatile uint32_t* dbg = nullptr,
                                          uint32_t step = 0) {
  if (mbar_try_wait(bar, parity)) return;
  if (dbg) dbg[threadIdx.x >> 5] = (code << 24) | (step & 0xFFFFFFu);
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (*reinterpret_cast<volatile unsigned int*>(&g_tc_err[0]) != 0) return;
    if (clock64() - t0 > 300000000LL) {
      if (atomicCAS(&g_tc_err[0], 0u, 0x80000000u | code) == 0u) {
        g_tc_err[1] = blockIdx.x; g_tc_err[2] = blockIdx.y; g_tc_err[3] = threadIdx.x; g_tc_err[4] = bar; g_tc_err[5] = parity;
        if (dbg) for (int i = 0; i < 32; ++i) g_tc_dbg[i] = dbg[i];
        __threadfence();
      }
      return;
    }
  }
  if (dbg) dbg[threadIdx.x >> 5] = 0;
}

// low / high words of a no-swizzle descriptor (LBO = 128 B everywhere in these kernels); advancing the start address by
// b bytes adds b >> 4 to the low word
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFF) | ((128u >> 4) << 16); }
__device__ __forceinline__ uint64_t mk_desc(uint32_t lo, uint32_t hi) { return ((uint64_t)hi << 32) | lo; }
// exactly one lane of a converged warp: lets ptxas issue the uniform-datapath tcgen05 instructions without a lane loop
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
constexpr uint32_t kFmtBF16 = 1, kFmtTF32 = 2;
// instruction descriptor: fp32 accumulate, A / B format, A / B major (0 = K, 1 = MN), N >> 3, M >> 4
__host__ __device__ constexpr uint32_t make_idesc(uint32_t fmt, int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_ss_tf32(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_ts_tf32(uint32_t d, uint32_t a_tmem, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d), "r"(a_tmem), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_ss_f16(uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem, uint32_t cols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {      // the allocating warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 32 lanes x 32-bit, N consecutive columns per thread (thread = TMEM lane of the warp's quadrant).  No wait inside:
// issue several, then tmem_ld_wait() once.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- packed fp32 pairs (Blackwell f32x2 arithmetic: one issue slot per two elements)
__device__ __forceinline__ unsigned long long pk2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void upk2(unsigned long long v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ float max3(float a, float b, float c) {   // FMNMX3
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float ex2f(float x) {   // one MUFU.EX2
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// bf16x2 {lo, hi} with round-to-nearest-even (lo in the low half = lower element index)
__device__ __forceinline__ uint32_t bf16x2_rn(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// The TF32 MMA truncates the low 13 mantissa bits of an fp32 operand; adding half an ulp first makes it round to nearest.
__device__ __forceinline__ float rtf32(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }

}  // namespace tc
}  // namespace dq
