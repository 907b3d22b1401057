// LinearAttention on tcgen05 / TMEM (reference /root/reference/dquartic/model/unet1d.py:473-496; the algebra - rank-C
// restructuring, saved statistics, partial buffers - is the one described at the top of linattn.cu).
//
// Why this shape.  Per position and head the kernels evaluate 32 exponentials; everything else is products of a
// [positions x 128 (head, d)] matrix with C <= 16 channel matrices.  With mma.sync those products live in register
// fragments and every softmax reduction / transposed product costs shuffles and shared-memory transposes (ncu r1d: LSU
// 64 %, 41-169 M bank conflicts, issue 60 %).  Here:
//   * TMEM lane = position: a thread owns one position and reads the 32 (q, dq) values of a head as 32 consecutive TMEM
//     columns - softmax over d and its backward are thread-local loops (no shuffles);
//   * the products with contraction over (head, d) take their A operand straight from TMEM (tcgen05.mma .ts form);
//   * the products with contraction over positions (Gq, dWq) read ONE bf16 [d][pos] tile through an MN-major
//     shared-memory descriptor - nobody transposes anything;
//   * warp-specialised roles decoupled by mbarriers: compute warps (per-element math), staging / draining warps
//     (global memory <-> operand tiles / accumulators), MMA-issuing warps.
// Measured bounds (profiles/r2_tc_probe.log, profiles/r2_la_bwd_q_tc_*): MUFU.EX2 delivers 15 results / clk / SM = 2.55 ms
// per 128 x L x R pass at level 0 with 64 samples; ex2.approx.f16x2 is two MUFU ops (no gain), a MUFU + FMA-polynomial mix
// reaches 19 / clk.  What bounds THIS kernel, though, is the tensor pipe: a tcgen05.mma costs 76 (SS tf32) / 103 (TS) /
// 119 (SS bf16 MN-major) cycles whatever N <= 128 is, and a 128-position tile needs 40 of them (8 score, 16 dXn_q, 16
// Gq / dWq) - about 2500 cycles per tile against 1100 for the exponentials.  The kernel is 1.3-1.45x faster than the
// mma.sync one (level 0: 0.9 vs 1.32 ms per 8 samples); moving the small-N products to ldmatrix + mma.sync on the
// staging warps and keeping tcgen05 for the N = 256 score product only is the next step (DESIGN.md).
#include <stdio.h>
#include <stdlib.h>
#include "linattn_args.cuh"
#include "linattn_tc.cuh"

#ifndef LA_AUX_SETS
#define LA_AUX_SETS 1
#endif
#ifndef LA_AUX_SETS8
#define LA_AUX_SETS8 2
#endif
namespace dq {
namespace tc {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kTfBiasMul = 1.00048828125f;   // (1 + 2^-11): un-biases the MMA's truncation of fp32 A operands in TMEM

__device__ __forceinline__ uint32_t f2tf(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

// =====================================================================================================================
// backward, q path.  Per row r and chunk of positions:
//   dy = RMSNorm_out backward(dres);  Q' = log2e Xn Wq^T;  dQs = dY G;  qs = softmax_d(Q) scale;
//   dQr = qs (dQs - sum_d qs dQs / scale);  dXn_q = dQr Wq;  Gq = Qs^T dY (partial);  dWq += dQr^T Xn.
// One CTA per SM, 24 warps: 16 compute warps = 4 groups (group g owns head g of every position tile; warp = TMEM lane
// quadrant), 4 staging / draining warps (thread = position), 4 MMA-issuing warps (score MMAs of the even / odd steps,
// dXn_q MMAs, Gq / dWq MMAs).  A "step" s = 4 t + h is (tile t, head h).
// TMEM (512 columns): score rings of 5 slots (slot = s % 5): Q' [32 i, +32), dQs [160 + 32 i, +32) - a slot is free again as
// soon as its group has LOADED it, so the scores of the next tile are computed while this one is processed; dQr of head h
// [320 + 32 h, +32); dXn_q accumulators of two tiles [448 + 16 p, +16); Gq [480, +16); dWq [496, +16).
template <int C>
struct BQ {
  static constexpr int CP = (C + 7) / 8 * 8;     // K of the position x channel products (tf32, k = 8 per MMA)
  static constexpr int KS = CP / 8;
  static constexpr int NC = 16;                  // N of the (.., channel) products
  static constexpr uint32_t A_SBO = 128 * (CP / 4);
  static constexpr int A_BYTES = 128 * CP * 4;   // one [128 x CP] tf32 tile
  static constexpr int T_BYTES = NC * 128 * 2;   // one [NC x 128 positions] bf16 tile
  static constexpr int TILE = 128 * 128 * 2;     // one [16 d-groups][128 pos][8] bf16 tile
  static constexpr int oBQ = 0;                          // 4 heads x [32 x CP] tf32: log2e Wq
  static constexpr int oBG = oBQ + A_BYTES;              // 4 heads x [32 x CP] tf32: G^T
  static constexpr int oBW = oBG + A_BYTES;              // 4 heads x [NC x 32] tf32: Wq^T (1 + 2^-11)
  static constexpr int NSTG = (CP == 8) ? 4 : 2;       // stage buffers: xn | dy [128 x CP] tf32, xn^T | dy^T [NC x 128] bf16
  static constexpr int oAX = oBW + 4 * NC * 32 * 4;
  static constexpr int oAD = oAX + NSTG * A_BYTES;
  static constexpr int oXT = oAD + NSTG * A_BYTES;
  static constexpr int oDT = oXT + NSTG * T_BYTES;
  static constexpr int oQS = oDT + NSTG * T_BYTES;       // 2 x qs tile
  static constexpr int oDR = oQS + 2 * TILE;             // 2 x dQr tile
  static constexpr int oBAR = oDR + 2 * TILE;
  static constexpr int NBAR = 48;
  static constexpr int SMEM = oBAR + NBAR * 8 + 16 + 128;   // barriers, TMEM address slot, per-warp wait record
  // staging / draining warp sets (tile t belongs to set t % AUX).  Measured (level shapes, 16 samples, whole backward):
  // C = 4: 1 set (24 warps, 80 registers) 3.57 ms vs 2 sets (28 warps, 72 registers, spills) 3.77 ms; C = 8, where a
  // set stages twice the channels per tile and was the pipeline's critical path: 1.57 -> 1.43 ms (L = 10000),
  // 0.85 -> 0.80 ms (L = 5000) with 2 sets; C = 12: no difference.
  static constexpr int AUX = (C == 8) ? LA_AUX_SETS8 : LA_AUX_SETS;
  static constexpr int MMAW0 = 16 + 4 * AUX;             // first MMA-issuing warp
  static constexpr int THREADS = (MMAW0 + 4) * 32;       // 16 compute + 4 AUX staging / draining + 4 MMA warps
};
constexpr int NREG = 5;       // slots of the TMEM score rings
// mbarrier indices
// The score-ring barriers are indexed by s % (2 NREG): the compute groups (and the two score-issuing warps) are NOT
// ordered among each other, so with one barrier per slot a waiter could be two phases ahead of the barrier and its
// parity test would alias (seen on the GPU: scores of step s + 5 issued before step s was consumed).  With 2 NREG
// barriers a waiter would have to be 2 NREG steps = 2.5 tiles ahead, which the tile-buffer hand-shake (bG) excludes.
constexpr int bS = 0, bLD = 10, bDONE = 20, bA = 24, bDXN = 28, bDXNFREE = 30, bFULL = 32, bG = 36, bTILE = 38, bSFREE = 40;
constexpr uint32_t cQ = 0, cDQ = 160, cDR = 320, cDXN = 448, cGQ = 480, cDWQ = 496;

template <int C>
__global__ void __launch_bounds__(BQ<C>::THREADS, 1) la_bwd_q_tc_kernel(LAArgs a) {
  using K = BQ<C>;
  extern __shared__ __align__(16) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = blockIdx.y, ch = blockIdx.x;
  const int n_begin = ch * a.chunk, n_end = min(a.L, n_begin + a.chunk);
  const int NT = (n_end - n_begin + 127) >> 7, S = 4 * NT;
  const uint32_t sb = smem_u32(smem);
  const uint32_t bar0 = sb + K::oBAR;
#define BAR(i) (bar0 + 8u * (uint32_t)(i))
  volatile uint32_t* tslot = reinterpret_cast<volatile uint32_t*>(smem + K::oBAR + K::NBAR * 8);
  volatile uint32_t* wdbg = reinterpret_cast<volatile uint32_t*>(smem + K::oBAR + K::NBAR * 8 + 16);
  if (tid < 32) wdbg[tid] = 0;

  if (tid == 0) {
    for (int i = 0; i < 2 * NREG; ++i) { mbar_init(BAR(bS + i), 1); mbar_init(BAR(bLD + i), 4); }
    for (int i = 0; i < 4; ++i) { mbar_init(BAR(bDONE + i), 4); mbar_init(BAR(bA + i), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(BAR(bDXN + i), 1); mbar_init(BAR(bDXNFREE + i), 4); mbar_init(BAR(bG + i), 1); mbar_init(BAR(bTILE + i), 16); }
    for (int i = 0; i < K::NSTG; ++i) { mbar_init(BAR(bFULL + i), 4); mbar_init(BAR(bSFREE + i), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == K::MMAW0) tmem_alloc(smem_u32(const_cast<const uint32_t*>(tslot)), 512);
  // operand staging buffers start as zeros (padding channels stay zero for the CTA's lifetime)
  for (int i = tid; i < (K::oQS - K::oAX) / 16; i += K::THREADS) reinterpret_cast<uint4*>(smem + K::oAX)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < 128 * K::CP; i += K::THREADS) {
    const int hd = i / K::CP, c = i % K::CP, h = hd >> 5, d = hd & 31;
    const uint32_t off = h * (32 * K::CP * 4) + (d & 7) * 16 + (d >> 3) * K::A_SBO + (c >> 2) * 128 + (c & 3) * 4;
    const float wq = c < C ? a.wqkv[(size_t)hd * C + c] * kLog2e : 0.f;
    const float gg = c < C ? a.gmat[((size_t)r * C + c) * kHD + hd] : 0.f;
    *reinterpret_cast<uint32_t*>(smem + K::oBQ + off) = f2tf(wq);
    *reinterpret_cast<uint32_t*>(smem + K::oBG + off) = f2tf(gg);
  }
  for (int i = tid; i < 4 * K::NC * 32; i += K::THREADS) {
    const int h = i / (K::NC * 32), rem = i % (K::NC * 32), c = rem >> 5, d = rem & 31;
    const float w = c < C ? a.wqkv[(size_t)(h * 32 + d) * C + c] * kTfBiasMul : 0.f;
    *reinterpret_cast<uint32_t*>(smem + K::oBW + h * (K::NC * 128) + (c & 7) * 16 + (c >> 3) * 1024 + (d >> 2) * 128 + (d & 3) * 4) = f2tf(w);
  }
  proxy_fence();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = *tslot;
  if (warp >= 16 && warp < 20) {   // (one staging set) every accumulating MMA is issued with accumulate = 1 (four issuing warps, no order)
    uint32_t z[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) z[i] = 0u;
    tmem_st32(tm + ((uint32_t)((warp - 16) * 32) << 16) + cDXN, z);
    tmem_st32(tm + ((uint32_t)((warp - 16) * 32) << 16) + cDXN + 32, z);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // Two staging sets = 28 warps compiled for 72 registers (pool 28 x 72 = 2016 per lane): the roles are re-balanced with
  // setmaxnreg - compute warps 80, staging / draining warps 64, MMA-issuing warps 40 (16 x 80 + 8 x 64 + 4 x 40 = 1952 <=
  // 2016; a request beyond the pool would block forever).  Measured at C = 8, L = 10000: backward 1.436 -> 1.395 ms;
  // 88 / 56 / 40 is slower (the staging warps spill at 56)
  if constexpr (K::AUX == 2) {
    if (warp < 16) asm volatile("setmaxnreg.inc.sync.aligned.u32 80;");
    else if (warp < K::MMAW0) asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
  }
  if (warp < 16) {
    // ------------------------------------------------------------------------------------------ per-element math
    const int h = warp >> 2, quad = warp & 3;
    const uint32_t lane_addr = tm + ((uint32_t)(quad * 32) << 16);
    const int pos = quad * 32 + lane;
    const float scale = rsqrtf((float)kDimHead), inv_scale = sqrtf((float)kDimHead);
    for (int t = 0; t < NT; ++t) {
      const int s = 4 * t + h, reg = s % NREG;
      mbar_wait(BAR(bS + s % (2 * NREG)), (uint32_t)((s / (2 * NREG)) & 1), 10, wdbg, (uint32_t)(s));
      tc_fence_after();
      uint32_t qv[32], dv[32];
      tmem_ld32(lane_addr + cQ + reg * 32, qv);
      tmem_ld32(lane_addr + cDQ + reg * 32, dv);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(bLD + s % (2 * NREG)));   // the slot may take the scores of step s + 5
      float* q = reinterpret_cast<float*>(qv);
      float* dq = reinterpret_cast<float*>(dv);
      float m0 = max3(q[0], q[1], q[2]), m1 = max3(q[3], q[4], q[5]);
#pragma unroll
      for (int i = 6; i < 30; i += 4) { m0 = max3(m0, q[i], q[i + 1]); m1 = max3(m1, q[i + 2], q[i + 3]); }
      const float m = max3(fmaxf(m0, m1), q[30], q[31]);
      const unsigned long long nm2 = pk2(-m, -m);
      unsigned long long sa = pk2(0.f, 0.f), sb2 = pk2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        float a0, a1, a2, a3;
        upk2(add2(pk2(q[i], q[i + 1]), nm2), a0, a1);
        upk2(add2(pk2(q[i + 2], q[i + 3]), nm2), a2, a3);
        q[i] = ex2f(a0); q[i + 1] = ex2f(a1); q[i + 2] = ex2f(a2); q[i + 3] = ex2f(a3);
        sa = add2(sa, pk2(q[i], q[i + 1]));
        sb2 = add2(sb2, pk2(q[i + 2], q[i + 3]));
      }
      float s0, s1;
      upk2(add2(sa, sb2), s0, s1);
      const float f = __fdividef(scale, s0 + s1);
      const unsigned long long f2 = pk2(f, f);
      unsigned long long ta = pk2(0.f, 0.f), tb = pk2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 32; i += 4) {   // qs = e f;  t = qs dQs
        const unsigned long long q01 = mul2(pk2(q[i], q[i + 1]), f2), q23 = mul2(pk2(q[i + 2], q[i + 3]), f2);
        const unsigned long long t01 = mul2(q01, pk2(dq[i], dq[i + 1])), t23 = mul2(q23, pk2(dq[i + 2], dq[i + 3]));
        upk2(q01, q[i], q[i + 1]); upk2(q23, q[i + 2], q[i + 3]);
        upk2(t01, dq[i], dq[i + 1]); upk2(t23, dq[i + 2], dq[i + 3]);
        ta = add2(ta, t01);
        tb = add2(tb, t23);
      }
      float t0, t1;
      upk2(add2(ta, tb), t0, t1);
      const float nts = -(t0 + t1) * inv_scale;
      const unsigned long long nts2 = pk2(nts, nts);
#pragma unroll
      for (int i = 0; i < 32; i += 2)   // dQr = t - ts qs
        upk2(fma2(nts2, pk2(q[i], q[i + 1]), pk2(dq[i], dq[i + 1])), dq[i], dq[i + 1]);
      if (t >= 1) mbar_wait(BAR(bA + h), (uint32_t)((t - 1) & 1), 12, wdbg, (uint32_t)(t));   // dQr of the previous tile consumed
      tmem_st32(lane_addr + cDR + h * 32, dv);
      // the bf16 tile buffers of tile t - 2 must have been consumed by its Gq / dWq MMAs
      if (t >= 2) mbar_wait(BAR(bG + (t & 1)), (uint32_t)(((t >> 1) - 1) & 1), 11, wdbg, (uint32_t)(t));
      uint8_t* tq = smem + K::oQS + (t & 1) * K::TILE;
      uint8_t* tr = smem + K::oDR + (t & 1) * K::TILE;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const uint32_t off = (uint32_t)(((4 * h + g) * 128 + pos) * 16);
        *reinterpret_cast<uint4*>(tq + off) =
            make_uint4(bf16x2_rn(q[8 * g], q[8 * g + 1]), bf16x2_rn(q[8 * g + 2], q[8 * g + 3]),
                       bf16x2_rn(q[8 * g + 4], q[8 * g + 5]), bf16x2_rn(q[8 * g + 6], q[8 * g + 7]));
        *reinterpret_cast<uint4*>(tr + off) =
            make_uint4(bf16x2_rn(dq[8 * g], dq[8 * g + 1]), bf16x2_rn(dq[8 * g + 2], dq[8 * g + 3]),
                       bf16x2_rn(dq[8 * g + 4], dq[8 * g + 5]), bf16x2_rn(dq[8 * g + 6], dq[8 * g + 7]));
      }
      tmem_st_wait();
      proxy_fence();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(BAR(bDONE + h)); mbar_arrive(BAR(bTILE + (t & 1))); }
    }
  } else if (warp >= K::MMAW0) {
    // ------------------------------------------------------------------------------------------ MMA issue
    // Four issuing warps (a single thread cannot issue ~40 small MMAs per tile fast enough, and the score MMAs must
    // run ahead of the compute warps, never behind a wait for them): warps 20 / 21 the score MMAs of the even / odd
    // steps, warp 22 the dXn_q MMAs, warp 23 the Gq / dWq MMAs.  All lanes run the control flow, one elected lane
    // issues.  Accumulators start as zeros (see above), every accumulating MMA has accumulate = 1.
    constexpr uint32_t id_s = make_idesc(kFmtTF32, 128, 32, 0, 0);
    constexpr uint32_t id_x = make_idesc(kFmtTF32, 128, K::NC, 0, 0);
    constexpr uint32_t id_g = make_idesc(kFmtBF16, 128, K::NC, 1, 0);
    constexpr uint32_t hiA = (K::A_SBO >> 4) | (1u << 14), hiW = (1024u >> 4) | (1u << 14), hiT = (2048u >> 4) | (1u << 14);
    if (warp <= K::MMAW0 + 1) {
      for (int s = warp - K::MMAW0; s < S; s += 2) {   // Q' and dQs of step s into ring slot s % NREG
        const int t = s >> 2, h = s & 3, reg = s % NREG, st = t % K::NSTG;
        mbar_wait(BAR(bFULL + st), (uint32_t)((t / K::NSTG) & 1), 20, wdbg, (uint32_t)(s));
        if (s >= NREG) mbar_wait(BAR(bLD + (s - NREG) % (2 * NREG)), (uint32_t)(((s - NREG) / (2 * NREG)) & 1), 21, wdbg, (uint32_t)(s));   // slot loaded by step s - 5
        tc_fence_after();
        if (elect_one()) {
          const uint32_t ax = desc_lo(sb + K::oAX + st * K::A_BYTES), ad = desc_lo(sb + K::oAD + st * K::A_BYTES);
          const uint32_t bq = desc_lo(sb + K::oBQ + h * (32 * K::CP * 4)), bg = desc_lo(sb + K::oBG + h * (32 * K::CP * 4));
#pragma unroll
          for (int ks = 0; ks < K::KS; ++ks) mma_ss_tf32(tm + cQ + reg * 32, mk_desc(ax + ks * 16, hiA), mk_desc(bq + ks * 16, hiA), id_s, ks > 0);
#pragma unroll
          for (int ks = 0; ks < K::KS; ++ks) mma_ss_tf32(tm + cDQ + reg * 32, mk_desc(ad + ks * 16, hiA), mk_desc(bg + ks * 16, hiA), id_s, ks > 0);
          umma_commit(BAR(bS + s % (2 * NREG)));
        }
        __syncwarp();
      }
    } else if (warp == K::MMAW0 + 2) {
      for (int t = 0; t < NT; ++t) {
        const int p = t & 1;
        if (t >= 2) mbar_wait(BAR(bDXNFREE + p), (uint32_t)(((t >> 1) - 1) & 1), 23, wdbg, (uint32_t)(t));   // accumulator of tile t - 2 drained
        for (int h = 0; h < 4; ++h) {
          mbar_wait(BAR(bDONE + h), (uint32_t)(t & 1), 22, wdbg, (uint32_t)(4 * t + h));
          tc_fence_after();
          if (elect_one()) {
            const uint32_t bw = desc_lo(sb + K::oBW + h * (K::NC * 128));
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)   // dXn_q[p] += dQr_h Wq_h
              mma_ts_tf32(tm + cDXN + 16 * p, tm + cDR + h * 32 + ks * 8, mk_desc(bw + ks * 16, hiW), id_x, 1u);
            umma_commit(BAR(bA + h));
            if (h == 3) umma_commit(BAR(bDXN + p));
          }
          __syncwarp();
        }
      }
    } else {
      for (int t = 0; t < NT; ++t) {   // Gq += Qs^T dY, dWq += dQr^T Xn over the 128 positions of tile t
        const int p = t & 1, st = t % K::NSTG;
        mbar_wait(BAR(bTILE + p), (uint32_t)((t >> 1) & 1), 24, wdbg, (uint32_t)(t));
        tc_fence_after();
        if (elect_one()) {
          const uint32_t aq = desc_lo(sb + K::oQS + p * K::TILE), ar = desc_lo(sb + K::oDR + p * K::TILE);
          const uint32_t bd = desc_lo(sb + K::oDT + st * K::T_BYTES), bx = desc_lo(sb + K::oXT + st * K::T_BYTES);
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            mma_ss_f16(tm + cGQ, mk_desc(aq + ks * 16, hiT), mk_desc(bd + ks * 16, hiT), id_g, 1u);
            mma_ss_f16(tm + cDWQ, mk_desc(ar + ks * 16, hiT), mk_desc(bx + ks * 16, hiT), id_g, 1u);
          }
          umma_commit(BAR(bG + p));
          umma_commit(BAR(bSFREE + st));
        }
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------------------------------------ staging / draining
    const int w = (warp - 16) & 3, j = w * 32 + lane, set = (warp - 16) >> 2;   // warps 16..23: set 0 even tiles, set 1 odd
    const uint32_t lane_addr = tm + ((uint32_t)(w * 32) << 16);
    const float sqrtC = sqrtf((float)C);
    float gp[C], go[C], dgo[C], dbo[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { gp[c] = __ldg(a.g_pre + c); go[c] = __ldg(a.g_out + c); dgo[c] = 0.f; dbo[c] = 0.f; }
    float xv[C], yv[C], rv[C];
    auto load_tile = [&](int t) {
      const int n = n_begin + t * 128 + j;
      const bool ok = n < n_end;
      const size_t base = (size_t)r * C * a.L + (ok ? n : n_end - 1);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        xv[c] = ok ? __ldg(a.x + base + (size_t)c * a.L) : 0.f;
        yv[c] = ok ? __ldg(a.ypre + base + (size_t)c * a.L) : 0.f;
        rv[c] = ok ? __ldg(a.dres + base + (size_t)c * a.L) : 0.f;
      }
    };
    auto stage = [&](int t) {
      const int st = t % K::NSTG;
      const bool ok = n_begin + t * 128 + j < n_end;
      float xn[K::CP], dy[K::CP];
      {
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) s2 = fmaf(xv[c], xv[c], s2);
        const float sc = sqrtC * rsqrtf(fmaxf(s2, 1e-24f));   // = sqrt(C) / max(|x|, 1e-12)
#pragma unroll
        for (int c = 0; c < K::CP; ++c) xn[c] = c < C ? xv[c < C ? c : 0] * sc * gp[c < C ? c : 0] : 0.f;
      }
      {  // RMSNorm_out backward
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) s2 = fmaf(yv[c], yv[c], s2);
        const float inv = rsqrtf(fmaxf(s2, 1e-24f));         // = 1 / max(|y|, 1e-12)
        const bool big = s2 > 1e-24f;
        float uh[C], duh[C], dot = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          uh[c] = yv[c] * inv;
          dgo[c] = fmaf(rv[c] * uh[c], sqrtC, dgo[c]);
          duh[c] = rv[c] * go[c] * sqrtC;
          dot = fmaf(duh[c], uh[c], dot);
        }
#pragma unroll
        for (int c = 0; c < K::CP; ++c) {
          float d = 0.f;
          if (c < C) {
            const int cc = c < C ? c : 0;
            d = big ? (duh[cc] - uh[cc] * dot) * inv : duh[cc] * inv;
            d = ok ? d : 0.f;
            dbo[cc] += d;
          }
          dy[c] = d;
        }
      }
      const uint32_t arow = (uint32_t)((j & 7) * 16 + (j >> 3) * K::A_SBO);
#pragma unroll
      for (int c4 = 0; c4 < K::CP / 4; ++c4) {
        *reinterpret_cast<float4*>(smem + K::oAX + st * K::A_BYTES + arow + c4 * 128) =
            make_float4(rtf32(xn[4 * c4]), rtf32(xn[4 * c4 + 1]), rtf32(xn[4 * c4 + 2]), rtf32(xn[4 * c4 + 3]));
        *reinterpret_cast<float4*>(smem + K::oAD + st * K::A_BYTES + arow + c4 * 128) =
            make_float4(rtf32(dy[4 * c4]), rtf32(dy[4 * c4 + 1]), rtf32(dy[4 * c4 + 2]), rtf32(dy[4 * c4 + 3]));
      }
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const uint32_t off = (uint32_t)(st * K::T_BYTES + (c & 7) * 16 + (c >> 3) * 2048 + (j >> 3) * 128 + (j & 7) * 2);
        *reinterpret_cast<__nv_bfloat16*>(smem + K::oXT + off) = __float2bfloat16_rn(xn[c]);
        *reinterpret_cast<__nv_bfloat16*>(smem + K::oDT + off) = __float2bfloat16_rn(dy[c]);
      }
      proxy_fence();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(bFULL + st));
    };
    auto drain = [&](int t) {   // dXn_q of tile t -> global
      const int p = t & 1;
      mbar_wait(BAR(bDXN + p), (uint32_t)((t >> 1) & 1), 30, wdbg, (uint32_t)(t));
      tc_fence_after();
      uint32_t d[16];
      tmem_ld16(lane_addr + cDXN + 16 * p, d);
      tmem_ld_wait();
      {
        uint32_t z[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) z[i] = 0u;
        tmem_st16(lane_addr + cDXN + 16 * p, z);
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(bDXNFREE + p));
      const int n = n_begin + t * 128 + j;
      if (n < n_end) {
#pragma unroll
        for (int c = 0; c < C; ++c) a.dxnq[((size_t)r * C + c) * a.L + n] = __uint_as_float(d[c]);
      }
    };
    for (int t = set; t < K::NSTG && t < NT; t += K::AUX) { load_tile(t); stage(t); }
    if (K::NSTG + set < NT) load_tile(K::NSTG + set);
    for (int t = set; t < NT; t += K::AUX) {
      if (t + K::NSTG < NT) {
        // stage buffer t % NSTG has been consumed (a barrier per buffer: its next phase needs this very staging, so a
        // slow staging warp can never miss a phase)
        mbar_wait(BAR(bSFREE + t % K::NSTG), (uint32_t)((t / K::NSTG) & 1), 31, wdbg, (uint32_t)(t));
        stage(t + K::NSTG);
        if (t + K::NSTG + K::AUX < NT) load_tile(t + K::NSTG + K::AUX);     // in flight while this tile drains
      }
      drain(t);
    }
    if (set != 0) {   // the chunk totals are read by set 0
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float s1 = warp_sum(dgo[c]), s2 = warp_sum(dbo[c]);
        if (lane == 0) { atomicAdd(a.dg_out + c, s1); atomicAdd(a.dbout + c, s2); }
      }
    } else {
    // chunk totals: Gq partial (rows = (head, d), this thread's TMEM lane) and dWq
    mbar_wait(BAR(bG + ((NT - 1) & 1)), (uint32_t)(((NT - 1) >> 1) & 1), 32, wdbg, (uint32_t)(NT));
    tc_fence_after();
    uint32_t gq[16], dw[16];
    tmem_ld16(lane_addr + cGQ, gq);
    tmem_ld16(lane_addr + cDWQ, dw);
    tmem_ld_wait();
    float* dp = a.dpart + (((size_t)r * a.nchunk + ch) * kHD + j) * K::CP;
#pragma unroll
    for (int c4 = 0; c4 < K::CP / 4; ++c4)
      *reinterpret_cast<float4*>(dp + 4 * c4) = make_float4(__uint_as_float(gq[4 * c4]), __uint_as_float(gq[4 * c4 + 1]),
                                                            __uint_as_float(gq[4 * c4 + 2]), __uint_as_float(gq[4 * c4 + 3]));
#pragma unroll
    for (int c = 0; c < C; ++c) atomicAdd(a.dwqkv + (size_t)j * C + c, __uint_as_float(dw[c]));
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float s1 = warp_sum(dgo[c]), s2 = warp_sum(dbo[c]);
      if (lane == 0) { atomicAdd(a.dg_out + c, s1); atomicAdd(a.dbout + c, s2); }
    }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == K::MMAW0) tmem_dealloc(tm, 512);
#undef BAR
}

template <int C>
static int launch_bwd_q(const LAArgs& a, cudaStream_t st) {
  using K = BQ<C>;
  auto kern = la_bwd_q_tc_kernel<C>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, K::SMEM);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((unsigned)a.nchunk, (unsigned)a.R);
  kern<<<grid, K::THREADS, K::SMEM, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

}  // namespace tc

}  // namespace dq
// pipeline-timeout record of the tcgen05 LinearAttention kernels: out[0] = 0 when clean, else 0x80000000 | wait code,
// out[1..5] = blockIdx.x, blockIdx.y, threadIdx.x, barrier address, parity.  Reading clears it.
DQ_API int dq_la_tc_last_error(unsigned int* out6) {
  unsigned int v[8] = {0};
  if (cudaMemcpyFromSymbol(v, dq::tc::g_tc_err, sizeof(v)) != cudaSuccess) return -1;
  for (int i = 0; i < 6; ++i) out6[i] = v[i];
  if (v[0] && getenv("DQ_LA_TC_DEBUG")) {
    unsigned int d[32];
    if (cudaMemcpyFromSymbol(d, dq::tc::g_tc_dbg, sizeof(d)) == cudaSuccess)
      for (int i = 0; i < 32; ++i) fprintf(stderr, "  warp %2d: wait code %u step %u\n", i, d[i] >> 24, d[i] & 0xFFFFFFu);
  }
  if (v[0]) { unsigned int z[8] = {0}; cudaMemcpyToSymbol(dq::tc::g_tc_err, z, sizeof(z)); }
  return v[0] ? 1 : 0;
}
namespace dq {

int la_bwd_q_tc(const LAArgs& a, int C, cudaStream_t st) {
  switch (C) {
    case 4: return tc::launch_bwd_q<4>(a, st);
    case 8: return tc::launch_bwd_q<8>(a, st);
    case 12: return tc::launch_bwd_q<12>(a, st);
    default: return -3;
  }
}

}  // namespace dq
