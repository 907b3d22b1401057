// Fused LinearAttention (reference /root/reference/dquartic/model/unet1d.py:473-496, wrapped as
// Residual(PreNorm(.)) at 1017/1068): out = x + RMSNorm_out(W_out . attn(RMSNorm_pre(x)) + b_out).
//
// Rank-C restructuring.  q, k, v are 1x1 projections of the C-channel (C <= 32) normalised input xn, so every
// per-head 32 x 32 contraction of the reference factors through C:
//     ctx[d][e]  = sum_n ks[d][n] v[e][n]           = sum_c Ms[d][c] Wv[e][c],     Ms[d][c] = sum_n ks[d][n] xn[c][n]
//     y[c'][n]   = sum_e Wout[c'][e] sum_d ctx[d][e] q[d][n] = sum_d G[c'][d] q[d][n],  G = Wout_h ctx_h^T   (C x 32)
// and likewise in the backward pass (Gq[d][c'] = sum_n q[d][n] dy[c'][n], H[d][c] = sum_e dctx[d][e] Wv[e][c]).
// Per position and head the work is a handful of 32 x C products instead of 32 x 32 ones, nothing of size
// 128 x L (let alone 384 x L) is ever materialised, and the v projection disappears from the per-position loops.
//
//   forward : la_stats  (per chunk: online softmax_L(k) partials  m, s, M[d][c] = sum_n exp(k-m) xn)
//             la_combine (per row: m, s, Ms = M/s, G)
//             la_out    (q = softmax_d(Wq xn) * scale, y = sum_h G_h q_h + b, RMSNorm_out, + x)
//   backward: la_bwd_q  (dy = RMSNorm_out backward; dq = G^T dy; softmax backward; d xn_q; partial Gq, dWq)
//             la_bwd_combine (per row: ctx, dctx, sd, H; dWout, dWv)
//             la_bwd_kv (ks, dks = H xn, d k_raw, d xn = Wk^T dk + H^T ks + d xn_q, RMSNorm_pre backward, + dres; dWk)
//
// Tensor cores: mma.sync m16n8k8 TF32 (fp32 accumulate), one warp = one head, all per-position intermediates in
// MMA register fragments; the accumulator fragment of one MMA is re-used directly as the A operand of the next.
// (tcgen05 does not fit: the contraction dims are C = 4..16 and the products are block-diagonal per (row, head) —
// a 128 x N x 16 tcgen05 tile would be >= 75 % padding and its TMEM round trip costs more than the math.)
//
// Fragment conventions (PTX m16n8k8 .tf32, g = lane/4, t = lane%4):
//   C/D: c0 (g, 2t) c1 (g, 2t+1) c2 (g+8, 2t) c3 (g+8, 2t+1)
//   A  : a0 (g, k=t) a1 (g+8, t) a2 (g, t+4) a3 (g+8, t+4)        B: b0 (k=t, n=g) b1 (k=t+4, n=g)
// We use a fixed permutation of the k index inside every k8 block: slot t <-> actual k = 2t, slot t+4 <-> 2t+1.
// Then (c0, c2, c1, c3) of an accumulator tile IS an A fragment and operands that come from memory are loaded
// with the same permutation (one 64-bit load).
#include <stdlib.h>
#include "common.cuh"
#include "linattn_args.cuh"

namespace dq {


template <int C>
struct TC {
  static constexpr int KC = (C + 7) / 8;                              // k8 steps over the C input channels
  static constexpr int CP = KC * 8;                                   // padded channel count
  static constexpr int XS = (CP == 8) ? 8 : (CP <= 24 ? 24 : 40);     // [pos][c] row stride: = 8 or 24 (mod 32)
  static constexpr int CT = KC;                                       // n8 tiles over C output channels
  static constexpr int PS = 2 + CP;                                   // partial record: m, s, M[CP]
  static constexpr int YS = C;                                        // row stride of per-head [pos][c] partial tiles (only c < C stored)
};
#ifndef LA_KV_ASYNC_MAXC
#define LA_KV_ASYNC_MAXC 4  // k / v backward: epilogue inputs and the next x tile prefetched by cp.async up to this C
#endif
#ifndef LA_OCCBIG
#define LA_OCCBIG 1  // the same for C = 12 / 16 (0 = no request)
#endif
#ifndef LA_OCC8
#define LA_OCC8 4  // resident CTAs per SM asked of the C = 8 backward kernels
#endif
#ifndef LA_OCC4
#define LA_OCC4 5  // resident CTAs per SM asked of the C = 4 backward kernels
#endif
constexpr int SP = 128;  // positions per staged sub-tile (= threads per CTA)
constexpr int XT = 136;  // row stride of the transposed [c][pos] tiles (= 8 mod 32: 64-bit fragment loads conflict-free)
constexpr int RS = 40;   // row stride of the warp-private 16 x 32 transpose tiles (= 8 mod 32, rows permuted: see store_tile16x32)
constexpr float kLazy = 8.f;  // online-softmax rescale threshold (numerators stay <= e^8)

__device__ __forceinline__ uint32_t f2tf(float x) {  // exact round-to-nearest TF32 (used outside the hot loops)
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// The TF32 MMA ignores the low 13 mantissa bits of its operands (truncation).  Adding half an ulp first makes that
// truncation a round-to-nearest (ties away) in ONE integer instruction; cvt.rna.tf32 compiles to two plus a NaN test.
__device__ __forceinline__ uint32_t rtf(float x) { return __float_as_uint(x) + 0x1000u; }
__device__ __forceinline__ float fexp2(float x) {  // single MUFU.EX2 (no denormal fix-up code)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kTfBias = 7.0444e-4f;           // log2(1 + 2^-11): pre-scaling a value by (1 + 2^-11) un-biases the
constexpr float kTfBiasMul = 1.00048828125f;    // MMA's operand truncation when it can be folded into an existing op
__device__ __forceinline__ void mma8(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                     uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// d = a b (zero accumulator input: no register zeroing)
__device__ __forceinline__ void mma8_z(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                       uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.f));
}
// A operand of the next MMA from an accumulator tile whose elements already carry TF32-ready bit patterns
// (rows g / g+8, cols 2t / 2t+1; k = its columns)
__device__ __forceinline__ void mma8_acc(float (&d)[4], const uint32_t (&v)[4], uint32_t b0, uint32_t b1) {
  mma8(d, v[0], v[2], v[1], v[3], b0, b1);
}
__device__ __forceinline__ void mma8_acc_z(float (&d)[4], const uint32_t (&v)[4], uint32_t b0, uint32_t b1) {
  mma8_z(d, v[0], v[2], v[1], v[3], b0, b1);
}
// d (+)= A[ks] B[ks] over the KC k8 steps of the C input channels, starting from zero
template <int KC>
__device__ __forceinline__ void mma_kc(float (&d)[4], const uint32_t (&a)[KC][4], const uint32_t (&b)[KC][2]) {
  mma8_z(d, a[0][0], a[0][1], a[0][2], a[0][3], b[0][0], b[0][1]);
#pragma unroll
  for (int ks = 1; ks < KC; ++ks) mma8(d, a[ks][0], a[ks][1], a[ks][2], a[ks][3], b[ks][0], b[ks][1]);
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// Software pipeline over the 128-position sub-tiles: the C raw inputs of the NEXT sub-tile are fetched into registers
// (load_x) before the slab loop of the current one, so their HBM latency hides behind the MMA / softmax work.
template <int C>
__device__ __forceinline__ void load_x(const float* __restrict__ x, int r, int L, int n0, int n_end, float (&v)[C]) {
  const int n = n0 + threadIdx.x;
  const bool ok = n < n_end;
#pragma unroll
  for (int c = 0; c < C; ++c) v[c] = ok ? __ldg(x + ((size_t)r * C + c) * L + n) : 0.f;
}
// The same prefetch without registers: 4-byte cp.async into a [C][SP] shared tile (slot [c][thread]); each thread reads
// back only what it copied itself, so cp.async.wait_group is the only synchronisation.  Used where the register
// prefetch would be spilled (ptxas stores a just-loaded register to local memory and stalls on the load).
__device__ __forceinline__ void cp_async4(float* dst_smem, const float* src, bool ok) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
  const int sz = ok ? 4 : 0;   // src-size 0: zero fill
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int C>
__device__ __forceinline__ void prefetch_x(const float* __restrict__ x, int r, int L, int n0, int n_end, float* dst) {
  const int n = n0 + threadIdx.x;
  const bool ok = n < n_end;
  const float* p = x + (size_t)r * C * L + (ok ? n : n_end - 1);
#pragma unroll
  for (int c = 0; c < C; ++c) cp_async4(dst + c * SP + threadIdx.x, p + (size_t)c * L, ok);
}
template <int C>
__device__ __forceinline__ void take_x(const float* src, float (&v)[C]) {
#pragma unroll
  for (int c = 0; c < C; ++c) v[c] = src[c * SP + threadIdx.x];
}
// Thread j normalises its position (RMSNorm over C with gain g) and writes the TF32-rounded row xn_s[j][0..CP)
// and column xnT_s[0..CP)[j]; invalid positions (all-zero inputs) give zeros.
// TROWS = rows of the transposed tile that are written: CP, or C when the caller lets the (never consumed) padding
// columns of the B operand alias whatever follows the tile in shared memory.
// ONES (C = 4 only): columns 4 and 5 of the [pos][8] row hold 1.0, so that per-channel constants ride in the spare
// k-slots of the position x channel MMAs (constant = hi + lo split over the two slots).
// NAT: xn_s is in the natural A-operand layout (TA<C>, see below) instead of [pos][XS] rows.
template <int C, int TROWS = TC<C>::CP, bool ONES = false, bool NAT = false>
__device__ __forceinline__ void stage_xn(const float (&xin)[C], const float* __restrict__ g, float* xn_s, float* xnT_s,
                                         float* inv_s) {
  using T = TC<C>;
  const int j = threadIdx.x;
  float v[T::CP];
  float s2 = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) s2 = fmaf(xin[c], xin[c], s2);
  const float inv = 1.f / fmaxf(sqrtf(s2), 1e-12f);
  const float sc = inv * sqrtf((float)C);
#pragma unroll
  for (int c = 0; c < T::CP; ++c)
    v[c] = (c < C) ? __uint_as_float(rtf(xin[c < C ? c : 0] * sc * __ldg(g + (c < C ? c : 0)))) : ((ONES && c < C + 2) ? 1.f : 0.f);
  if (xn_s) {
    if (NAT) {
      float* col = xn_s + (j >> 4) * (T::CP * 20) + 2 * (j & 7) + ((j >> 3) & 1);
#pragma unroll
      for (int c = 0; c < T::CP; ++c) col[c * 20] = v[c];
    } else {
      float4* row = reinterpret_cast<float4*>(xn_s + j * T::XS);
#pragma unroll
      for (int c4 = 0; c4 < T::CP / 4; ++c4) row[c4] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
    }
  }
  if (xnT_s) {
#pragma unroll
    for (int c = 0; c < TROWS; ++c) xnT_s[c * XT + j] = v[c];
  }
  if (inv_s) inv_s[j] = inv;
}

// B fragments of X^T (k = channel, n = position) for the two n8 tiles of slab s:  bx[j][ks] = {xn[pos][8ks+2t], [..+1]}
template <int C>
__device__ __forceinline__ void load_bx(const float* xn_s, int s, int g, int t, uint32_t (&bx)[2][TC<C>::KC][2]) {
  using T = TC<C>;
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int ks = 0; ks < T::KC; ++ks) {
      float2 v = *reinterpret_cast<const float2*>(xn_s + (16 * s + 8 * j + g) * T::XS + 8 * ks + 2 * t);
      bx[j][ks][0] = __float_as_uint(v.x);
      bx[j][ks][1] = __float_as_uint(v.y);
    }
}
// A fragments of X (rows = positions g, g+8 of slab s; k = channel)
template <int C>
__device__ __forceinline__ void load_ax(const float* xn_s, int s, int g, int t, uint32_t (&ax)[TC<C>::KC][4]) {
  using T = TC<C>;
#pragma unroll
  for (int ks = 0; ks < T::KC; ++ks) {
    float2 lo = *reinterpret_cast<const float2*>(xn_s + (16 * s + g) * T::XS + 8 * ks + 2 * t);
    float2 hi = *reinterpret_cast<const float2*>(xn_s + (16 * s + 8 + g) * T::XS + 8 * ks + 2 * t);
    ax[ks][0] = __float_as_uint(lo.x); ax[ks][2] = __float_as_uint(lo.y);
    ax[ks][1] = __float_as_uint(hi.x); ax[ks][3] = __float_as_uint(hi.y);
  }
}
// B fragments of X (k = position inside k8 block j of slab s, n = channel) from the transposed tile
template <int C>
__device__ __forceinline__ void load_bT(const float* xT_s, int s, int j, int g, int t, uint32_t (&b)[TC<C>::CT][2]) {
  using T = TC<C>;
#pragma unroll
  for (int ct = 0; ct < T::CT; ++ct) {
    float2 v = *reinterpret_cast<const float2*>(xT_s + (8 * ct + g) * XT + 16 * s + 8 * j + 2 * t);
    b[ct][0] = __float_as_uint(v.x);
    b[ct][1] = __float_as_uint(v.y);
  }
}
// store a tile set v[4][4] (rows = positions g / g+8 of the slab, cols = channel 8*tile + 2t, +1).
// Position p lives in row p ^ ((p >> 2) & 1): with RS = 8 (mod 32) the 64-bit stores of a half-warp (4 positions x
// 8 words) and the 32-bit transposed loads of a warp (positions 2t (+1) x 8 channels) both cover all 32 banks once.
__device__ __forceinline__ void store_tile16x32(float* scr, const uint32_t (&v)[4][4], int g, int t) {
  float* p = scr + (g ^ (g >> 2)) * RS + 2 * t;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    *reinterpret_cast<uint2*>(p + 8 * dt) = make_uint2(v[dt][0], v[dt][1]);
    *reinterpret_cast<uint2*>(p + 8 * RS + 8 * dt) = make_uint2(v[dt][2], v[dt][3]);
  }
}
// A fragment of the TRANSPOSED tile: rows = channels 16*mt + g (+8), k = positions 8*j + 2t (+1)
__device__ __forceinline__ void load_At(const float* scr, int mt, int j, int g, int t, uint32_t (&A)[4]) {
  const int r0 = (2 * t) ^ (t >> 1);                                  // row of position 2t; position 2t+1 is in row r0 ^ 1
  const uint32_t* p0 = reinterpret_cast<const uint32_t*>(scr) + (8 * j + r0) * RS + 16 * mt + g;
  const uint32_t* p1 = p0 + ((t >> 1) ? -RS : RS);
  A[0] = p0[0]; A[1] = p0[8]; A[2] = p1[0]; A[3] = p1[8];
}
// softmax over the 32 columns (4 n8 tiles) of rows g and g+8, times `scale`, in place
// packed 2 x fp32 arithmetic (Blackwell fma/mul/add.rn.f32x2): one issue slot per two elements.  The element pairs are
// the adjacent accumulator registers (c0, c1) / (c2, c3) of the MMA fragments, so packing is a register alias.
__device__ __forceinline__ unsigned long long pk2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void upk2(unsigned long long v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
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
// softmax over the 32 columns (4 n8 tiles) of rows g and g+8, times `scale`, in place
__device__ __forceinline__ void softmax_rows(float (&q)[4][4], float scale) {
  const unsigned long long l2e = pk2(kLog2e, kLog2e);
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    float mx = -INFINITY;
#pragma unroll
    for (int dt = 0; dt < 4; ++dt) mx = fmaxf(mx, fmaxf(q[dt][2 * hf], q[dt][2 * hf + 1]));
    const float nm = -quad_max(mx) * kLog2e;
    const unsigned long long nm2 = pk2(nm, nm);
    unsigned long long sm2 = pk2(0.f, 0.f);
#pragma unroll
    for (int dt = 0; dt < 4; ++dt) {
      float a0, a1;
      upk2(fma2(pk2(q[dt][2 * hf], q[dt][2 * hf + 1]), l2e, nm2), a0, a1);
      q[dt][2 * hf] = fexp2(a0);
      q[dt][2 * hf + 1] = fexp2(a1);
      sm2 = add2(sm2, pk2(q[dt][2 * hf], q[dt][2 * hf + 1]));
    }
    float s0, s1;
    upk2(sm2, s0, s1);
    const float f = __fdividef(scale, quad_sum(s0 + s1));
    const unsigned long long f2 = pk2(f, f);
#pragma unroll
    for (int dt = 0; dt < 4; ++dt) upk2(mul2(pk2(q[dt][2 * hf], q[dt][2 * hf + 1]), f2), q[dt][2 * hf], q[dt][2 * hf + 1]);
  }
}
__device__ __forceinline__ void round_tile(const float (&v)[4][4], uint32_t (&o)[4][4]) {
#pragma unroll
  for (int dt = 0; dt < 4; ++dt)
#pragma unroll
    for (int i = 0; i < 4; ++i) o[dt][i] = rtf(v[dt][i]);
}

// "Natural" A-operand layout of a normalised input sub-tile: per slab of 16 positions a block of CP channel rows of
// AROW floats, position p of the slab at column 2 (p & 7) + (p >> 3).  The fragment registers (a0, a1) = rows g / g+8 of
// k-slot t and (a2, a3) of k-slot t+4 are then two 64-bit loads that land in HMMA operand order (the [pos][c] layout
// needs a 4-register permutation per fragment, which ptxas materialises as ~14 moves per slab); k-slot t <-> channel
// 2t, t+4 <-> 2t+1 as everywhere; AROW = 20 keeps the fragment loads conflict-free (the staging stores, once per
// sub-tile, are 2-way conflicted).
constexpr int AROW = 20;   // (stage_xn's NAT branch spells the same numbers out: it is defined before this point)
template <int C>
struct TA {
  static constexpr int SLAB = TC<C>::CP * AROW;         // floats per slab block
  static constexpr int SIZE = (SP / 16) * SLAB;
};
template <int C>
__device__ __forceinline__ void stage_xn_nat(const float (&xin)[C], const float* __restrict__ g, float* xa_s) {
  using T = TC<C>;
  const int j = threadIdx.x;
  float s2 = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) s2 = fmaf(xin[c], xin[c], s2);
  const float sc = sqrtf((float)C) / fmaxf(sqrtf(s2), 1e-12f);
  float* col = xa_s + (j >> 4) * TA<C>::SLAB + 2 * (j & 7) + ((j >> 3) & 1);
#pragma unroll
  for (int c = 0; c < T::CP; ++c)
    col[c * AROW] = (c < C) ? __uint_as_float(rtf(xin[c < C ? c : 0] * sc * __ldg(g + (c < C ? c : 0)))) : 0.f;
}
template <int C>
__device__ __forceinline__ void load_ax_nat(const float* xa_s, int s, int g, int t, uint32_t (&ax)[TC<C>::KC][4]) {
#pragma unroll
  for (int ks = 0; ks < TC<C>::KC; ++ks) {
    const float* p = xa_s + s * TA<C>::SLAB + (8 * ks + 2 * t) * AROW + 2 * g;
    const float2 v01 = *reinterpret_cast<const float2*>(p), v23 = *reinterpret_cast<const float2*>(p + AROW);
    ax[ks][0] = __float_as_uint(v01.x); ax[ks][1] = __float_as_uint(v01.y);
    ax[ks][2] = __float_as_uint(v23.x); ax[ks][3] = __float_as_uint(v23.y);
  }
}
// softmax over the 32 columns of rows g and g+8 times `scale`, delivered as the A operand of the next MMA:
// A[dt] = (q[dt][0], q[dt][2], q[dt][1], q[dt][3]).  After the exponentials the packed arithmetic pairs the two ROWS
// (c0, c2) / (c1, c3), so the results are born in operand order and the row sums come out packed.
__device__ __forceinline__ void softmax_rows_A(const float (&q)[4][4], float scale, uint32_t (&A)[4][4]) {
  const unsigned long long l2e = pk2(kLog2e, kLog2e);
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    mx0 = fmaxf(mx0, fmaxf(q[dt][0], q[dt][1]));
    mx1 = fmaxf(mx1, fmaxf(q[dt][2], q[dt][3]));
  }
  const float nm0 = -quad_max(mx0) * kLog2e, nm1 = -quad_max(mx1) * kLog2e;
  const unsigned long long n0 = pk2(nm0, nm0), n1 = pk2(nm1, nm1);
  unsigned long long e02[4], e13[4], sm = pk2(0.f, 0.f);
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    float a0, a1, a2, a3;
    upk2(fma2(pk2(q[dt][0], q[dt][1]), l2e, n0), a0, a1);
    upk2(fma2(pk2(q[dt][2], q[dt][3]), l2e, n1), a2, a3);
    e02[dt] = pk2(fexp2(a0), fexp2(a2));
    e13[dt] = pk2(fexp2(a1), fexp2(a3));
    sm = add2(add2(sm, e02[dt]), e13[dt]);
  }
  float s0, s1;
  upk2(sm, s0, s1);
  const unsigned long long f = pk2(__fdividef(scale, quad_sum(s0)), __fdividef(scale, quad_sum(s1)));
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
    float x0, x1;
    upk2(mul2(e02[dt], f), x0, x1);
    A[dt][0] = __float_as_uint(x0); A[dt][1] = __float_as_uint(x1);
    upk2(mul2(e13[dt], f), x0, x1);
    A[dt][2] = __float_as_uint(x0); A[dt][3] = __float_as_uint(x1);
  }
}

// ------------------------------------------------------------------------------------------- forward: stats
// K^T = Wk_h X^T as (32 channels x 16 positions) accumulator tiles; softmax over positions is a row-wise online
// softmax with a lazy rescale; M[d][c] += P[d][n] Xn[n][c] re-uses the K^T accumulators as the A operand.
// The numerators carry a (1 + 2^-11) factor (folded into the exponent) so that the MMA's operand truncation is
// unbiased; the same factor is in s, so it cancels in Ms = M / s up to the rounding of the individual terms.
template <int C, bool FULL>
__device__ __forceinline__ void stats_slab(const float* xn_s, const float* xnT_s, int s, int g, int t, int n_left,
                                           const uint32_t (&wk)[2][TC<C>::KC][4], float (&m_run)[2][2],
                                           float (&nm2)[2][2], float (&s_run)[2][2], float (&Macc)[2][TC<C>::CT][4]) {
  using T = TC<C>;
  uint32_t bx[2][T::KC][2];
  load_bx<C>(xn_s, s, g, t, bx);
  float kacc[2][2][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int j = 0; j < 2; ++j) mma_kc<T::KC>(kacc[mt][j], wk[mt], bx[j]);
  if (!FULL) {  // positions >= n_left (relative to the slab) do not exist: push them to -inf (exp -> 0)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int i = 0; i < 2; ++i)
        if (8 * j + 2 * t + i >= n_left) {
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) { kacc[mt][j][i] = -INFINITY; kacc[mt][j][2 + i] = -INFINITY; }
        }
  }
  // lazy online softmax: rescale only when some row's slab maximum exceeds the running reference by > kLazy
  float lm[2][2];
  bool need = false;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      lm[mt][hf] = fmaxf(fmaxf(kacc[mt][0][2 * hf], kacc[mt][0][2 * hf + 1]), fmaxf(kacc[mt][1][2 * hf], kacc[mt][1][2 * hf + 1]));
      need |= lm[mt][hf] > m_run[mt][hf] + kLazy;
    }
  if (__any_sync(0xffffffffu, need)) {
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const float m_new = fmaxf(m_run[mt][hf], quad_max(lm[mt][hf]));
        const float f = fexp2((m_run[mt][hf] - m_new) * kLog2e);  // exp(-inf) = 0 on the first slab
        s_run[mt][hf] *= f;
#pragma unroll
        for (int ct = 0; ct < T::CT; ++ct) { Macc[mt][ct][2 * hf] *= f; Macc[mt][ct][2 * hf + 1] *= f; }
        m_run[mt][hf] = m_new;
        nm2[mt][hf] = fmaf(-m_new, kLog2e, kTfBias);
      }
  }
  uint32_t pk[2][2][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float p = fexp2(fmaf(kacc[mt][j][i], kLog2e, nm2[mt][i >> 1]));
        s_run[mt][i >> 1] += p;
        pk[mt][j][i] = __float_as_uint(p);
      }
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    uint32_t bt[T::CT][2];
    load_bT<C>(xnT_s, s, j, g, t, bt);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int ct = 0; ct < T::CT; ++ct) mma8_acc(Macc[mt][ct], pk[mt][j], bt[ct][0], bt[ct][1]);
  }
}

template <int C>
__global__ void __launch_bounds__(128) la_stats_kernel(LAArgs a) {
  using T = TC<C>;
  __shared__ __align__(16) float xn_s[SP * T::XS];
  __shared__ __align__(16) float xnT_s[T::CP * XT];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int r = blockIdx.y, ch = blockIdx.x;
  const int n_begin = ch * a.chunk, n_end = min(a.L, n_begin + a.chunk);

  uint32_t wk[2][T::KC][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int ks = 0; ks < T::KC; ++ks)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int d = h * 32 + 16 * mt + g + 8 * (i & 1), c = 8 * ks + 2 * t + (i >> 1);
        wk[mt][ks][i] = f2tf(c < C ? a.wqkv[(size_t)(kHD + d) * C + c] : 0.f);
      }
  float m_run[2][2], nm2[2][2], s_run[2][2], Macc[2][T::CT][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    m_run[mt][0] = m_run[mt][1] = -INFINITY;
    nm2[mt][0] = nm2[mt][1] = 0.f;
    s_run[mt][0] = s_run[mt][1] = 0.f;
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 4; ++i) Macc[mt][ct][i] = 0.f;
  }

  float xv[C];
  load_x<C>(a.x, r, a.L, n_begin, n_end, xv);
  for (int n0 = n_begin; n0 < n_end; n0 += SP) {
    stage_xn<C>(xv, a.g_pre, xn_s, xnT_s, nullptr);
    __syncthreads();
    if (n0 + SP < n_end) load_x<C>(a.x, r, a.L, n0 + SP, n_end, xv);
    const int nfull = min(SP, n_end - n0) / 16, nslab = min(SP / 16, (n_end - n0 + 15) / 16);
    for (int s = 0; s < nfull; ++s) stats_slab<C, true>(xn_s, xnT_s, s, g, t, 16, wk, m_run, nm2, s_run, Macc);
    if (nslab > nfull) stats_slab<C, false>(xn_s, xnT_s, nfull, g, t, n_end - n0 - 16 * nfull, wk, m_run, nm2, s_run, Macc);
    __syncthreads();
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const float s = quad_sum(s_run[mt][hf]);
      const int d = h * 32 + 16 * mt + 8 * hf + g;
      float* po = a.part + (((size_t)r * a.nchunk + ch) * kHD + d) * T::PS;
      if (t == 0) { po[0] = m_run[mt][hf]; po[1] = s; }
#pragma unroll
      for (int ct = 0; ct < T::CT; ++ct)
        *reinterpret_cast<float2*>(po + 2 + 8 * ct + 2 * t) = make_float2(Macc[mt][ct][2 * hf], Macc[mt][ct][2 * hf + 1]);
    }
}

// per row: m, s, Ms = M / s, ctx (registers only), G[c'][h*32+d] = sum_e Wout[c'][h*32+e] ctx[d][e]
template <int C>
__global__ void __launch_bounds__(128) la_combine_kernel(LAArgs a) {
  using T = TC<C>;
  const int j = threadIdx.x, h = j >> 5, r = blockIdx.x;
  const float* p = a.part + ((size_t)r * a.nchunk * kHD + j) * T::PS;
  float M = -INFINITY;
  for (int ch = 0; ch < a.nchunk; ++ch) M = fmaxf(M, p[(size_t)ch * kHD * T::PS]);
  float S = 0.f, ms[C];
#pragma unroll
  for (int c = 0; c < C; ++c) ms[c] = 0.f;
  for (int ch = 0; ch < a.nchunk; ++ch) {
    const float* q = p + (size_t)ch * kHD * T::PS;
    const float f = fexp2((q[0] - M) * kLog2e);
    S = fmaf(q[1], f, S);
#pragma unroll
    for (int c = 0; c < C; ++c) ms[c] = fmaf(q[2 + c], f, ms[c]);
  }
  const float inv = 1.f / S;
  float* mo = a.msm + ((size_t)r * kHD + j) * T::PS;
  mo[0] = M;
  mo[1] = S;
#pragma unroll
  for (int c = 0; c < T::CP; ++c) {
    if (c < C) ms[c < C ? c : 0] *= inv;
    mo[2 + c] = (c < C) ? ms[c < C ? c : 0] : 0.f;
  }
  float gacc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) gacc[c] = 0.f;
  for (int e = 0; e < 32; ++e) {
    const float* wv = a.wqkv + (size_t)(2 * kHD + h * 32 + e) * C;
    float cx = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) cx = fmaf(ms[c], __ldg(wv + c), cx);
#pragma unroll
    for (int c = 0; c < C; ++c) gacc[c] = fmaf(__ldg(a.wout + (size_t)c * kHD + h * 32 + e), cx, gacc[c]);
  }
#pragma unroll
  for (int c = 0; c < C; ++c) a.gmat[((size_t)r * C + c) * kHD + j] = gacc[c];
}

// ------------------------------------------------------------------------------------------- forward: output
// Per 16-position slab and head: Q = X Wq^T (positions x d) -> softmax over d (quad shuffles) -> Y_h = Qs G_h^T,
// all in fragments; the four heads' Y_h meet in shared memory for bias + RMSNorm + residual.
template <int C>
__global__ void __launch_bounds__(128) la_out_kernel(LAArgs a) {
  using T = TC<C>;
  extern __shared__ float4 dyn_smem4[];
  float* xn_s = reinterpret_cast<float*>(dyn_smem4);  // TA<C>::SIZE: natural A-operand layout
  float* yp_s = xn_s + TA<C>::SIZE;                   // 4 * SP * YS
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int r = blockIdx.y;
  const int n_begin = blockIdx.x * a.chunk, n_end = min(a.L, n_begin + a.chunk);
  const float scale = rsqrtf((float)kDimHead);

  uint32_t bq[4][T::KC][2], bg[4][T::CT][2];
#pragma unroll
  for (int dt = 0; dt < 4; ++dt)
#pragma unroll
    for (int ks = 0; ks < T::KC; ++ks)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int d = h * 32 + 8 * dt + g, c = 8 * ks + 2 * t + i;
        bq[dt][ks][i] = f2tf(c < C ? a.wqkv[(size_t)d * C + c] : 0.f);
      }
#pragma unroll
  for (int kd = 0; kd < 4; ++kd)
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = 8 * ct + g;
        bg[kd][ct][i] = f2tf(c < C ? a.gmat[((size_t)r * C + c) * kHD + h * 32 + 8 * kd + 2 * t + i] : 0.f);
      }

  float xv[C], xcur[C];
  load_x<C>(a.x, r, a.L, n_begin, n_end, xv);
  for (int n0 = n_begin; n0 < n_end; n0 += SP) {
    stage_xn_nat<C>(xv, a.g_pre, xn_s);
#pragma unroll
    for (int c = 0; c < C; ++c) xcur[c] = xv[c];   // residual input of this sub-tile's epilogue
    __syncthreads();
    if (n0 + SP < n_end) load_x<C>(a.x, r, a.L, n0 + SP, n_end, xv);
    const int nslab = min(SP / 16, (n_end - n0 + 15) / 16);
    for (int s = 0; s < nslab; ++s) {
      uint32_t ax[T::KC][4];
      load_ax_nat<C>(xn_s, s, g, t, ax);
      float q[4][4];
#pragma unroll
      for (int dt = 0; dt < 4; ++dt) mma_kc<T::KC>(q[dt], ax, bq[dt]);
      uint32_t qa[4][4];
      softmax_rows_A(q, scale * kTfBiasMul, qa);   // q is only an MMA operand here: pre-bias against the truncation
      float y[T::CT][4];
#pragma unroll
      for (int ct = 0; ct < T::CT; ++ct) {
        mma8_z(y[ct], qa[0][0], qa[0][1], qa[0][2], qa[0][3], bg[0][ct][0], bg[0][ct][1]);
#pragma unroll
        for (int kd = 1; kd < 4; ++kd) mma8(y[ct], qa[kd][0], qa[kd][1], qa[kd][2], qa[kd][3], bg[kd][ct][0], bg[kd][ct][1]);
      }
#pragma unroll
      for (int ct = 0; ct < T::CT; ++ct)
        if (8 * ct + 2 * t < C) {
          float* p0 = yp_s + ((size_t)h * SP + 16 * s + g) * T::YS + 8 * ct + 2 * t;
          *reinterpret_cast<float2*>(p0) = make_float2(y[ct][0], y[ct][1]);
          *reinterpret_cast<float2*>(p0 + 8 * T::YS) = make_float2(y[ct][2], y[ct][3]);
        }
    }
    __syncthreads();
    {
      const int j = threadIdx.x, n = n0 + j;
      if (n < n_end) {
        float y[C];
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          y[c] = a.bout[c] + yp_s[(0 * SP + j) * T::YS + c] + yp_s[(1 * SP + j) * T::YS + c] +
                 yp_s[(2 * SP + j) * T::YS + c] + yp_s[(3 * SP + j) * T::YS + c];
          s2 = fmaf(y[c], y[c], s2);
        }
        const float sc = sqrtf((float)C) / fmaxf(sqrtf(s2), 1e-12f);
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const size_t idx = ((size_t)r * C + c) * a.L + n;
          if (a.ypre) a.ypre[idx] = y[c];
          a.out[idx] = fmaf(y[c] * sc, a.g_out[c], xcur[c]);
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------- backward: q path
// Per slab and head (fragments): Q -> Qs, dQs = dY G_h, dQr (softmax backward), dXn_q = dQr Wq_h.
// Reductions over positions (Gq = Qs^T dY, dWq = dQr^T Xn) read Qs / dQr back from warp-private shared tiles in
// the transposed role.
template <int C>
__global__ void __launch_bounds__(128, (C <= 4 ? LA_OCC4 : (C <= 8 ? LA_OCC8 : LA_OCCBIG))) la_bwd_q_kernel(LAArgs a) {
  using T = TC<C>;
  extern __shared__ float4 dyn_smem4[];
  // C = 4: ONE [pos][8] tile with xn and dy interleaved (xn0, dy0, xn1, dy1, ..): a single A fragment then carries xn
  // in k = 0..3 and dy in k = 4..7, and the two B operands (Wq^T | 0) and (0 | G) need one register each
  constexpr bool kMerged = (C == 4);
  float* xn_s = reinterpret_cast<float*>(dyn_smem4);   // TA<C>::SIZE (natural A-operand layout)
  float* dy_s = xn_s + (kMerged ? 0 : TA<C>::SIZE);    // TA<C>::SIZE (merged: same tile)
  // transposed tiles hold only the C real channel rows: rows C..CP-1 of a B fragment (n = channel) alias the next
  // array; those accumulator columns are never stored
  float* xnT_s = dy_s + TA<C>::SIZE;                   // C * XT
  float* dyT_s = xnT_s + C * XT;                       // C * XT
  float* yp_s = dyT_s + C * XT;                        // 4 * SP * YS   per-head d xn_q
  float* scr = yp_s + 4 * SP * T::YS;                  // 4 warps * 2 tiles * 16 * RS
  float* acc_s = scr + 4 * 2 * 16 * RS;                // 2 * C  (d g_out, d b_out)
  constexpr bool kAsync = (C == 4);                    // prefetch through shared memory (registers would spill)
  float* pf_s = acc_s + 2 * C;                         // kAsync: 3 * C * SP (x, ypre, dres of the next sub-tile)
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int r = blockIdx.y, ch = blockIdx.x;
  const int n_begin = ch * a.chunk, n_end = min(a.L, n_begin + a.chunk);
  const float scale = rsqrtf((float)kDimHead), inv_scale = sqrtf((float)kDimHead);
  const float sqrtC = sqrtf((float)C);
  float* scrQ = scr + (h * 2 + 0) * 16 * RS;
  float* scrR = scr + (h * 2 + 1) * 16 * RS;

  uint32_t bq[4][T::KC][2], bgA[4][T::KC][2], bqT[4][T::CT][2];
#pragma unroll
  for (int dt = 0; dt < 4; ++dt)
#pragma unroll
    for (int ks = 0; ks < T::KC; ++ks)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = 8 * ks + 2 * t + i, d = h * 32 + 8 * dt + g;
        if (kMerged) {  // k = t: xn channel t, k = t + 4: dy channel t; only element [0] of each is used
          bq[dt][ks][i] = f2tf(a.wqkv[(size_t)d * C + t]);
          bgA[dt][ks][i] = f2tf(a.gmat[((size_t)r * C + t) * kHD + d]);
        } else {
          bq[dt][ks][i] = f2tf(c < C ? a.wqkv[(size_t)d * C + c] : 0.f);
          bgA[dt][ks][i] = f2tf(c < C ? a.gmat[((size_t)r * C + c) * kHD + d] : 0.f);   // B[k = c'][n = d] = G[c'][d]
        }
      }
#pragma unroll
  for (int kd = 0; kd < 4; ++kd)
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = 8 * ct + g;
        bqT[kd][ct][i] = f2tf(c < C ? a.wqkv[(size_t)(h * 32 + 8 * kd + 2 * t + i) * C + c] : 0.f);
      }
  float gq[2][T::CT][4], dwq[2][T::CT][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 4; ++i) { gq[mt][ct][i] = 0.f; dwq[mt][ct][i] = 0.f; }
  if (threadIdx.x < 2 * C) acc_s[threadIdx.x] = 0.f;
  __syncthreads();

  float xv[C], yv[C], drv[C];
  if (kAsync) {
    prefetch_x<C>(a.x, r, a.L, n_begin, n_end, pf_s);
    prefetch_x<C>(a.ypre, r, a.L, n_begin, n_end, pf_s + C * SP);
    prefetch_x<C>(a.dres, r, a.L, n_begin, n_end, pf_s + 2 * C * SP);
    cp_async_commit();
  } else {
    load_x<C>(a.x, r, a.L, n_begin, n_end, xv);
    load_x<C>(a.ypre, r, a.L, n_begin, n_end, yv);
    load_x<C>(a.dres, r, a.L, n_begin, n_end, drv);
  }
  for (int n0 = n_begin; n0 < n_end; n0 += SP) {
    if (kAsync) {
      cp_async_wait0();
      take_x<C>(pf_s, xv);
      take_x<C>(pf_s + C * SP, yv);
      take_x<C>(pf_s + 2 * C * SP, drv);
    }
    stage_xn<C, C, false, true>(xv, a.g_pre, kMerged ? nullptr : xn_s, xnT_s, nullptr);
    {  // d y = RMSNorm_out backward of d res, thread j = position
      const int j = threadIdx.x, n = n0 + j;
      const bool ok = n < n_end;
      float y[C], dr[C];
      float s2 = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        y[c] = yv[c];
        dr[c] = drv[c];
        s2 = fmaf(y[c], y[c], s2);
      }
      const float nrm = sqrtf(s2), inv = 1.f / fmaxf(nrm, 1e-12f);
      float dot = 0.f, dgl[C];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float uh = y[c] * inv;
        dgl[c] = dr[c] * uh * sqrtC;
        const float duh = dr[c] * a.g_out[c] * sqrtC;
        dot = fmaf(duh, uh, dot);
        y[c] = uh; dr[c] = duh;
      }
      float dv[T::CP];
#pragma unroll
      for (int c = 0; c < T::CP; ++c) {
        float d = 0.f;
        if (c < C) {
          d = (nrm > 1e-12f) ? (dr[c < C ? c : 0] - y[c < C ? c : 0] * dot) * inv : dr[c < C ? c : 0] * inv;
          d = ok ? d : 0.f;
          const float s1 = warp_sum(dgl[c < C ? c : 0]), s2b = warp_sum(d);
          if (lane == 0) { atomicAdd(acc_s + c, s1); atomicAdd(acc_s + C + c, s2b); }
        }
        dv[c] = __uint_as_float(rtf(d));
        if (c < C) dyT_s[c * XT + j] = dv[c];
      }
      float* col = dy_s + (j >> 4) * TA<C>::SLAB + 2 * (j & 7) + ((j >> 3) & 1);
      if (kMerged) {  // rows (xn0, dy0, xn1, dy1, ..); xn comes back from its own column of the transposed tile
#pragma unroll
        for (int c = 0; c < C; ++c) {
          col[(2 * c) * AROW] = xnT_s[c * XT + j];
          col[(2 * c + 1) * AROW] = dv[c];
        }
      } else {
#pragma unroll
        for (int c = 0; c < T::CP; ++c) col[c * AROW] = dv[c];
      }
    }
    __syncthreads();
    if (n0 + SP < n_end) {
      if (kAsync) {
        prefetch_x<C>(a.x, r, a.L, n0 + SP, n_end, pf_s);
        prefetch_x<C>(a.ypre, r, a.L, n0 + SP, n_end, pf_s + C * SP);
        prefetch_x<C>(a.dres, r, a.L, n0 + SP, n_end, pf_s + 2 * C * SP);
        cp_async_commit();
      } else {
        load_x<C>(a.x, r, a.L, n0 + SP, n_end, xv);
        load_x<C>(a.ypre, r, a.L, n0 + SP, n_end, yv);
        load_x<C>(a.dres, r, a.L, n0 + SP, n_end, drv);
      }
    }
    const int nslab = min(SP / 16, (n_end - n0 + 15) / 16);
    for (int s = 0; s < nslab; ++s) {
      float qs[4][4], dqs[4][4];
      {
        uint32_t ax[T::KC][4];
        load_ax_nat<C>(xn_s, s, g, t, ax);
        if (kMerged) {
#pragma unroll
          for (int dt = 0; dt < 4; ++dt) {
            mma8_z(qs[dt], ax[0][0], ax[0][1], ax[0][2], ax[0][3], bq[dt][0][0], 0u);
            mma8_z(dqs[dt], ax[0][0], ax[0][1], ax[0][2], ax[0][3], 0u, bgA[dt][0][0]);
          }
        } else {
#pragma unroll
          for (int dt = 0; dt < 4; ++dt) mma_kc<T::KC>(qs[dt], ax, bq[dt]);
          load_ax_nat<C>(dy_s, s, g, t, ax);
#pragma unroll
          for (int dt = 0; dt < 4; ++dt) mma_kc<T::KC>(dqs[dt], ax, bgA[dt]);
        }
      }
      // q carries a (1 + 2^-11) factor: the MMA's operand truncation of q (in Gq) and of dQr = q (dQs - ts) (in dWq,
      // d xn_q) is then unbiased without any explicit rounding instruction
      softmax_rows(qs, scale * kTfBiasMul);
      store_tile16x32(scrQ, reinterpret_cast<const uint32_t(&)[4][4]>(qs), g, t);
      // softmax backward: dQr = Qs * (dQs - sum_d Qs dQs / scale)
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        float ts = 0.f;
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) ts += qs[dt][2 * hf] * dqs[dt][2 * hf] + qs[dt][2 * hf + 1] * dqs[dt][2 * hf + 1];
        ts = quad_sum(ts) * inv_scale;
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) {
          dqs[dt][2 * hf] = qs[dt][2 * hf] * (dqs[dt][2 * hf] - ts);
          dqs[dt][2 * hf + 1] = qs[dt][2 * hf + 1] * (dqs[dt][2 * hf + 1] - ts);
        }
      }
      const uint32_t (&rq)[4][4] = reinterpret_cast<const uint32_t(&)[4][4]>(dqs);
      store_tile16x32(scrR, rq, g, t);
      {  // d xn_q (this head) = dQr Wq_h
        float dxn[T::CT][4];
#pragma unroll
        for (int ct = 0; ct < T::CT; ++ct) {
          mma8_acc_z(dxn[ct], rq[0], bqT[0][ct][0], bqT[0][ct][1]);
#pragma unroll
          for (int kd = 1; kd < 4; ++kd) mma8_acc(dxn[ct], rq[kd], bqT[kd][ct][0], bqT[kd][ct][1]);
        }
#pragma unroll
        for (int ct = 0; ct < T::CT; ++ct)
          if (8 * ct + 2 * t < C) {
            float* p0 = yp_s + ((size_t)h * SP + 16 * s + g) * T::YS + 8 * ct + 2 * t;
            *reinterpret_cast<float2*>(p0) = make_float2(dxn[ct][0], dxn[ct][1]);
            *reinterpret_cast<float2*>(p0 + 8 * T::YS) = make_float2(dxn[ct][2], dxn[ct][3]);
          }
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        uint32_t Bdy[T::CT][2], Bxn[T::CT][2];
        load_bT<C>(dyT_s, s, j, g, t, Bdy);
        load_bT<C>(xnT_s, s, j, g, t, Bxn);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          uint32_t Aq[4], Ar[4];
          load_At(scrQ, mt, j, g, t, Aq);
          load_At(scrR, mt, j, g, t, Ar);
#pragma unroll
          for (int ct = 0; ct < T::CT; ++ct) {
            mma8(gq[mt][ct], Aq[0], Aq[1], Aq[2], Aq[3], Bdy[ct][0], Bdy[ct][1]);
            mma8(dwq[mt][ct], Ar[0], Ar[1], Ar[2], Ar[3], Bxn[ct][0], Bxn[ct][1]);
          }
        }
      }
      __syncwarp();
    }
    __syncthreads();
    {
      const int j = threadIdx.x, n = n0 + j;
      if (n < n_end) {
#pragma unroll
        for (int c = 0; c < C; ++c)
          a.dxnq[((size_t)r * C + c) * a.L + n] = yp_s[(0 * SP + j) * T::YS + c] + yp_s[(1 * SP + j) * T::YS + c] +
                                                  yp_s[(2 * SP + j) * T::YS + c] + yp_s[(3 * SP + j) * T::YS + c];
      }
    }
    __syncthreads();
  }
  // Gq partial of this chunk: rows d, cols c'
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      float* dp = a.dpart + (((size_t)r * a.nchunk + ch) * kHD + h * 32 + 16 * mt + 8 * hf + g) * T::CP;
#pragma unroll
      for (int ct = 0; ct < T::CT; ++ct)
        *reinterpret_cast<float2*>(dp + 8 * ct + 2 * t) = make_float2(gq[mt][ct][2 * hf], gq[mt][ct][2 * hf + 1]);
    }
  // d Wq (rows d, cols c)
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int d = h * 32 + 16 * mt + g + 8 * (i >> 1), c = 8 * ct + 2 * t + (i & 1);
        if (c < C) atomicAdd(a.dwqkv + (size_t)d * C + c, dwq[mt][ct][i]);
      }
  __syncthreads();
  if (threadIdx.x < C) atomicAdd(a.dg_out + threadIdx.x, acc_s[threadIdx.x]);
  else if (threadIdx.x < 2 * C) atomicAdd(a.dbout + threadIdx.x - C, acc_s[threadIdx.x]);
}

// per row: Gq, ctx, dctx, sd, H; dWout and dWv (their reductions over positions collapsed to reductions over d)
template <int C>
__global__ void __launch_bounds__(128) la_bwd_combine_kernel(LAArgs a, int rows_per_block) {
  using T = TC<C>;
  extern __shared__ float4 dyn_smem4[];
  float* ctx_s = reinterpret_cast<float*>(dyn_smem4);  // 128 * 33
  float* dctx_s = ctx_s + kHD * 33;                    // 128 * 33
  float* gq_s = dctx_s + kHD * 33;                     // 128 * (C + 1)
  float* ms_s = gq_s + kHD * (C + 1);                  // 128 * (C + 1)
  const int j = threadIdx.x, h = j >> 5, e = j & 31;
  float dwo[C], dwv[C];
#pragma unroll
  for (int c = 0; c < C; ++c) { dwo[c] = 0.f; dwv[c] = 0.f; }
  const int r0 = blockIdx.x * rows_per_block, r1 = min(a.R, r0 + rows_per_block);
  for (int r = r0; r < r1; ++r) {
    float gqv[C], ms[C];
#pragma unroll
    for (int c = 0; c < C; ++c) gqv[c] = 0.f;
    for (int ch = 0; ch < a.nchunk; ++ch) {
      const float* p = a.dpart + (((size_t)r * a.nchunk + ch) * kHD + j) * T::CP;
#pragma unroll
      for (int c = 0; c < C; ++c) gqv[c] += p[c];
    }
    const float* mp = a.msm + ((size_t)r * kHD + j) * T::PS + 2;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      ms[c] = mp[c];
      gq_s[j * (C + 1) + c] = gqv[c];
      ms_s[j * (C + 1) + c] = ms[c];
    }
    float sd = 0.f, hacc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) hacc[c] = 0.f;
    for (int ee = 0; ee < 32; ++ee) {
      const float* wv = a.wqkv + (size_t)(2 * kHD + h * 32 + ee) * C;
      float cx = 0.f, dc = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        cx = fmaf(ms[c], __ldg(wv + c), cx);
        dc = fmaf(__ldg(a.wout + (size_t)c * kHD + h * 32 + ee), gqv[c], dc);
      }
      sd = fmaf(dc, cx, sd);
#pragma unroll
      for (int c = 0; c < C; ++c) hacc[c] = fmaf(dc, __ldg(wv + c), hacc[c]);
      ctx_s[j * 33 + ee] = cx;
      dctx_s[j * 33 + ee] = dc;
    }
    a.sd[(size_t)r * kHD + j] = sd;
    float* ho = a.hmat + ((size_t)r * kHD + j) * T::CP;
#pragma unroll
    for (int c = 0; c < T::CP; ++c) ho[c] = (c < C) ? hacc[c < C ? c : 0] : 0.f;
    __syncthreads();
    // thread (h, e): dWout[c'][h*32+e] += sum_d ctx[d][e] Gq[d][c'];  dWv[h*32+e][c] += sum_d dctx[d][e] Ms[d][c]
    for (int d = 0; d < 32; ++d) {
      const float cx = ctx_s[(h * 32 + d) * 33 + e], dc = dctx_s[(h * 32 + d) * 33 + e];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        dwo[c] = fmaf(cx, gq_s[(h * 32 + d) * (C + 1) + c], dwo[c]);
        dwv[c] = fmaf(dc, ms_s[(h * 32 + d) * (C + 1) + c], dwv[c]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int c = 0; c < C; ++c) {
    atomicAdd(a.dwout + (size_t)c * kHD + j, dwo[c]);
    atomicAdd(a.dwqkv + (size_t)(2 * kHD + j) * C + c, dwv[c]);
  }
}

// ------------------------------------------------------------------------------------------- backward: k path
template <int C>
__global__ void __launch_bounds__(128, (C <= 4 ? LA_OCC4 : (C <= 8 ? LA_OCC8 : LA_OCCBIG))) la_bwd_kv_kernel(LAArgs a) {
  using T = TC<C>;
  extern __shared__ float4 dyn_smem4[];
  float* xn_s = reinterpret_cast<float*>(dyn_smem4);   // TA<C>::SIZE (natural A-operand layout)
  float* xnT_s = xn_s + TA<C>::SIZE;                   // C * XT (see la_bwd_q_kernel)
  float* yp_s = xnT_s + C * XT;                        // 4 * SP * YS
  float* scr = yp_s + 4 * SP * T::YS;                  // 4 warps * 16 * RS
  float* inv_s = scr + 4 * 16 * RS;                    // SP
  float* acc_s = inv_s + SP;                           // C (d g_pre)
  constexpr bool kAsync = (C <= LA_KV_ASYNC_MAXC);     // prefetch through shared memory (see la_bwd_q_kernel)
  float* pf_s = acc_s + C;                             // kAsync: 4 * C * SP: x (two alternating slots), dxnq, dres
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
  const int r = blockIdx.y;
  const int n_begin = blockIdx.x * a.chunk, n_end = min(a.L, n_begin + a.chunk);
  const float sqrtC = sqrtf((float)C);
  float* scrK = scr + h * 16 * RS;

  // C = 4: log2e is folded into Wk, and the per-channel constants (softmax offset, -sd) into the spare k-slots of the
  // xn operand, so exp2 / the softmax backward take the MMA outputs as they come
  constexpr bool kFold = (C == 4);
  uint32_t bwk[4][T::KC][2], bh[4][T::KC][2], bkT[4][T::CT][2], bhT[4][T::CT][2];
  float cn[4][2], cd[4][2];
#pragma unroll
  for (int dt = 0; dt < 4; ++dt) {
#pragma unroll
    for (int ks = 0; ks < T::KC; ++ks)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = 8 * ks + 2 * t + i, d = h * 32 + 8 * dt + g;
        bwk[dt][ks][i] = f2tf(c < C ? a.wqkv[(size_t)(kHD + d) * C + c] * (kFold ? kLog2e : 1.f) : 0.f);
        bh[dt][ks][i] = f2tf(a.hmat[((size_t)r * kHD + d) * T::CP + c]);               // B[k = c][n = d] = H[d][c]
        if (kFold && (c == C || c == C + 1)) {
          // spare k-slots (the A rows carry 1.0 there): the softmax constant and -sd of channel d, split hi + lo
          const size_t jd = (size_t)r * kHD + d;
          const float cnd = kTfBias - (a.msm[jd * T::PS] * kLog2e + log2f(a.msm[jd * T::PS + 1]));
          const float sdd = -a.sd[jd];
          const float cn_hi = __uint_as_float(f2tf(cnd)), sd_hi = __uint_as_float(f2tf(sdd));
          bwk[dt][ks][i] = (c == C) ? __float_as_uint(cn_hi) : f2tf(cnd - cn_hi);
          bh[dt][ks][i] = (c == C) ? __float_as_uint(sd_hi) : f2tf(sdd - sd_hi);
        }
      }
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int c = 8 * ct + g, d = h * 32 + 8 * dt + 2 * t + i;
        bkT[dt][ct][i] = f2tf(c < C ? a.wqkv[(size_t)(kHD + d) * C + c] : 0.f);        // B[k = d][n = c] = Wk[d][c]
        bhT[dt][ct][i] = f2tf(a.hmat[((size_t)r * kHD + d) * T::CP + c]);              // B[k = d][n = c] = H[d][c]
      }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const size_t jd = (size_t)r * kHD + h * 32 + 8 * dt + 2 * t + i;
      // softmax_L(k) = 2^(k log2e + cn); the + kTfBias pre-scales ks (and d k_raw = ks (..)) by (1 + 2^-11) so that the
      // MMA's operand truncation is unbiased without explicit rounding
      cn[dt][i] = kFold ? 0.f : kTfBias - (a.msm[jd * T::PS] * kLog2e + log2f(a.msm[jd * T::PS + 1]));
      cd[dt][i] = kFold ? 0.f : a.sd[jd];
    }
  }
  float dwk[2][T::CT][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 4; ++i) dwk[mt][ct][i] = 0.f;
  if (threadIdx.x < C) acc_s[threadIdx.x] = 0.f;

  float xv[C], xcur[C], dqv[C], drv[C];
  int slot = 0;
  if (kAsync) {
    prefetch_x<C>(a.x, r, a.L, n_begin, n_end, pf_s);
    cp_async_commit();
  } else {
    load_x<C>(a.x, r, a.L, n_begin, n_end, xv);
  }
  for (int n0 = n_begin; n0 < n_end; n0 += SP) {
    if (kAsync) {
      cp_async_wait0();
      take_x<C>(pf_s + slot * C * SP, xv);
    }
    stage_xn<C, C, (C == 4), true>(xv, a.g_pre, xn_s, xnT_s, inv_s);
    if (!kAsync) {
#pragma unroll
      for (int c = 0; c < C; ++c) xcur[c] = xv[c];
    }
    __syncthreads();
    if (kAsync) {  // epilogue inputs of this sub-tile and x of the next one, in flight during the slab loop
      prefetch_x<C>(a.dxnq, r, a.L, n0, n_end, pf_s + 2 * C * SP);
      prefetch_x<C>(a.dres, r, a.L, n0, n_end, pf_s + 3 * C * SP);
      if (n0 + SP < n_end) prefetch_x<C>(a.x, r, a.L, n0 + SP, n_end, pf_s + (slot ^ 1) * C * SP);
      cp_async_commit();
    } else {
      load_x<C>(a.dxnq, r, a.L, n0, n_end, dqv);   // epilogue inputs of this sub-tile, in flight during the slab loop
      load_x<C>(a.dres, r, a.L, n0, n_end, drv);
      if (n0 + SP < n_end) load_x<C>(a.x, r, a.L, n0 + SP, n_end, xv);
    }
    const int nslab = min(SP / 16, (n_end - n0 + 15) / 16);
    for (int s = 0; s < nslab; ++s) {
      float kk[4][4], dks[4][4];
      {
        uint32_t ax[T::KC][4];
        load_ax_nat<C>(xn_s, s, g, t, ax);
#pragma unroll
        for (int dt = 0; dt < 4; ++dt) {
          mma_kc<T::KC>(kk[dt], ax, bwk[dt]);
          mma_kc<T::KC>(dks[dt], ax, bh[dt]);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (kFold) {
              kk[dt][i] = fexp2(kk[dt][i]);                                // softmax_L(k)
              dks[dt][i] = kk[dt][i] * dks[dt][i];                         // d k_raw
            } else {
              kk[dt][i] = fexp2(fmaf(kk[dt][i], kLog2e, cn[dt][i & 1]));
              dks[dt][i] = kk[dt][i] * (dks[dt][i] - cd[dt][i & 1]);
            }
          }
        }
      }
      const uint32_t (&rk)[4][4] = reinterpret_cast<const uint32_t(&)[4][4]>(kk);
      const uint32_t (&rd)[4][4] = reinterpret_cast<const uint32_t(&)[4][4]>(dks);
      store_tile16x32(scrK, rd, g, t);
      {
        float dxn[T::CT][4];
#pragma unroll
        for (int ct = 0; ct < T::CT; ++ct) {
          mma8_acc_z(dxn[ct], rd[0], bkT[0][ct][0], bkT[0][ct][1]);
          mma8_acc(dxn[ct], rk[0], bhT[0][ct][0], bhT[0][ct][1]);
#pragma unroll
          for (int kd = 1; kd < 4; ++kd) {
            mma8_acc(dxn[ct], rd[kd], bkT[kd][ct][0], bkT[kd][ct][1]);
            mma8_acc(dxn[ct], rk[kd], bhT[kd][ct][0], bhT[kd][ct][1]);
          }
        }
#pragma unroll
        for (int ct = 0; ct < T::CT; ++ct)
          if (8 * ct + 2 * t < C) {
            float* p0 = yp_s + ((size_t)h * SP + 16 * s + g) * T::YS + 8 * ct + 2 * t;
            *reinterpret_cast<float2*>(p0) = make_float2(dxn[ct][0], dxn[ct][1]);
            *reinterpret_cast<float2*>(p0 + 8 * T::YS) = make_float2(dxn[ct][2], dxn[ct][3]);
          }
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        uint32_t Bxn[T::CT][2];
        load_bT<C>(xnT_s, s, j, g, t, Bxn);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          uint32_t Ak[4];
          load_At(scrK, mt, j, g, t, Ak);
#pragma unroll
          for (int ct = 0; ct < T::CT; ++ct) mma8(dwk[mt][ct], Ak[0], Ak[1], Ak[2], Ak[3], Bxn[ct][0], Bxn[ct][1]);
        }
      }
      __syncwarp();
    }
    __syncthreads();
    {  // thread j = position: RMSNorm_pre backward + residual gradient
      const int j = threadIdx.x, n = n0 + j;
      const bool ok = n < n_end;
      if (kAsync) {
        cp_async_wait0();
        take_x<C>(pf_s + slot * C * SP, xcur);
        take_x<C>(pf_s + 2 * C * SP, dqv);
        take_x<C>(pf_s + 3 * C * SP, drv);
        slot ^= 1;
      }
      const float inv = inv_s[j];
      float uh[C], duh[C];
      float dot = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const size_t idx = ((size_t)r * C + c) * a.L + n;
        const float dxn = ok ? yp_s[(0 * SP + j) * T::YS + c] + yp_s[(1 * SP + j) * T::YS + c] +
                                   yp_s[(2 * SP + j) * T::YS + c] + yp_s[(3 * SP + j) * T::YS + c] + dqv[c]
                             : 0.f;
        uh[c] = xcur[c] * inv;
        const float dgc = warp_sum(dxn * uh[c] * sqrtC);
        if (lane == 0) atomicAdd(acc_s + c, dgc);
        duh[c] = dxn * a.g_pre[c] * sqrtC;
        dot = fmaf(duh[c], uh[c], dot);
      }
      if (ok) {
        const bool big = inv < 1e12f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const size_t idx = ((size_t)r * C + c) * a.L + n;
          const float d = big ? (duh[c] - uh[c] * dot) * inv : duh[c] * inv;
          a.dx[idx] = drv[c] + d;
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int ct = 0; ct < T::CT; ++ct)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int d = h * 32 + 16 * mt + g + 8 * (i >> 1), c = 8 * ct + 2 * t + (i & 1);
        if (c < C) atomicAdd(a.dwqkv + (size_t)(kHD + d) * C + c, dwk[mt][ct][i]);
      }
  __syncthreads();
  if (threadIdx.x < C) atomicAdd(a.dg_pre + threadIdx.x, acc_s[threadIdx.x]);
}

// DQ_LA_TC=0 selects the mma.sync kernels of this file everywhere (cross-check / A-B timing); default: tcgen05 kernels
static bool la_tc_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DQ_LA_TC"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

template <int C>
static int la_fwd(const LAArgs& a, cudaStream_t st) {
  using T = TC<C>;
  dim3 grid((unsigned)a.nchunk, (unsigned)a.R);
  la_stats_kernel<C><<<grid, 128, 0, st>>>(a);
  DQ_LAUNCH_CHECK();
  la_combine_kernel<C><<<(unsigned)a.R, 128, 0, st>>>(a);
  DQ_LAUNCH_CHECK();
  size_t smem = sizeof(float) * (TA<C>::SIZE + 4 * SP * T::YS);
  cudaFuncSetAttribute(la_out_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  la_out_kernel<C><<<grid, 128, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

template <int C>
static int la_bwd(const LAArgs& a, cudaStream_t st) {
  using T = TC<C>;
  dim3 grid((unsigned)a.nchunk, (unsigned)a.R);
  // tcgen05 / TMEM kernel (linattn_tc.cu) where it wins: per launch of a 64-sample micro-batch 9.43 -> 5.89 ms (C = 4),
  // 3.95 -> 3.24 (C = 8), 1.82 -> 1.18 (C = 12); at C = 16 (L <= 1250: 5-10 tiles per CTA, fixed cost dominates, spills) it
  // measured 1.21 vs 0.71 ms, so the mma.sync kernel keeps that level (profiles/r2_launches_summary.csv vs r1d)
  if (la_tc_enabled() && C <= 12) {
    const int rc = la_bwd_q_tc(a, C, st);
    if (rc != 0) return rc;
  } else {
    size_t smem = sizeof(float) * ((C == 4 ? 1 : 2) * TA<C>::SIZE + 2 * C * XT + 4 * SP * T::YS + 4 * 2 * 16 * RS + 2 * C +
                                   (C == 4 ? 3 * C * SP : 0));
    cudaFuncSetAttribute(la_bwd_q_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    la_bwd_q_kernel<C><<<grid, 128, smem, st>>>(a);
    DQ_LAUNCH_CHECK();
  }
  {
    constexpr int kRows = 8;
    size_t smem = sizeof(float) * (2 * kHD * 33 + 2 * kHD * (C + 1));
    cudaFuncSetAttribute(la_bwd_combine_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    la_bwd_combine_kernel<C><<<(unsigned)((a.R + kRows - 1) / kRows), 128, smem, st>>>(a, kRows);
    DQ_LAUNCH_CHECK();
  }
  {
    size_t smem = sizeof(float) * (TA<C>::SIZE + C * XT + 4 * SP * T::YS + 4 * 16 * RS + SP + C + (C <= LA_KV_ASYNC_MAXC ? 4 * C * SP : 0));
    cudaFuncSetAttribute(la_bwd_kv_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    la_bwd_kv_kernel<C><<<grid, 128, smem, st>>>(a);
    DQ_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace dq

using namespace dq;

// chunking policy shared by forward and backward (the Python side sizes `part`/`dpart` from dq_la_nchunk):
// at most ~8192 positions per CTA, chunks of equal size rounded up to whole 128-position sub-tiles
static int la_nchunk(int L) { return (L + 8191) / 8192; }
static int la_chunk(int L) {
  int n = la_nchunk(L);
  int c = (L + n - 1) / n;
  return (c + SP - 1) / SP * SP;
}
DQ_API int dq_la_nchunk(int L) { int c = la_chunk(L); return (L + c - 1) / c; }

DQ_API int dq_linattn_fwd(const float* x, const float* g_pre, const float* wqkv, const float* wout, const float* bout,
                          const float* g_out, float* part, float* msm, float* gmat, float* ypre, float* out, int C,
                          int R, int L, void* stream) {
  LAArgs a{};
  a.x = x; a.g_pre = g_pre; a.wqkv = wqkv; a.wout = wout; a.bout = bout; a.g_out = g_out;
  a.part = part; a.msm = msm; a.gmat = gmat; a.ypre = ypre; a.out = out;
  a.R = R; a.L = L; a.chunk = la_chunk(L); a.nchunk = (L + a.chunk - 1) / a.chunk;
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || L <= 0) return 0;
  switch (C) {
    case 4: return la_fwd<4>(a, st);
    case 8: return la_fwd<8>(a, st);
    case 12: return la_fwd<12>(a, st);
    case 16: return la_fwd<16>(a, st);
    case 24: return la_fwd<24>(a, st);
    case 32: return la_fwd<32>(a, st);
    default: return -3;
  }
}

DQ_API int dq_linattn_bwd(const float* x, const float* dres, const float* ypre, const float* msm, const float* gmat,
                          const float* g_pre, const float* wqkv, const float* wout, const float* g_out, float* dxnq,
                          float* dpart, float* hmat, float* sd, float* dx, float* dwqkv, float* dwout, float* dbout,
                          float* dg_out, float* dg_pre, int C, int R, int L, void* stream) {
  LAArgs a{};
  a.x = x; a.dres = dres; a.ypre = const_cast<float*>(ypre); a.msm = const_cast<float*>(msm);
  a.gmat = const_cast<float*>(gmat); a.g_pre = g_pre; a.wqkv = wqkv; a.wout = wout; a.g_out = g_out;
  a.dxnq = dxnq; a.dpart = dpart; a.hmat = hmat; a.sd = sd; a.dx = dx;
  a.dwqkv = dwqkv; a.dwout = dwout; a.dbout = dbout; a.dg_out = dg_out; a.dg_pre = dg_pre;
  a.R = R; a.L = L; a.chunk = la_chunk(L); a.nchunk = (L + a.chunk - 1) / a.chunk;
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || L <= 0) return 0;
  switch (C) {
    case 4: return la_bwd<4>(a, st);
    case 8: return la_bwd<8>(a, st);
    case 12: return la_bwd<12>(a, st);
    case 16: return la_bwd<16>(a, st);
    case 24: return la_bwd<24>(a, st);
    case 32: return la_bwd<32>(a, st);
    default: return -3;
  }
}
