// Fused backward of one stride-1 Conv1d (K = 1 or 3, "same" padding) of the down/up path together with the
// backward of its Block epilogue (reference /root/reference/dquartic/model/unet1d.py: Block.forward 248-268,
// RMSNorm 140, ResnetBlock.forward 302-323 incl. the 1x1 res_conv 300/323):
//
//      du  = d(RMSNorm * (scale+1) + shift -> SiLU)^T dy            (pointwise over channels; skipped if u == null)
//      dx  = conv_transpose(du, W) (+ dadd)                         (dual destination = backward of the skip concat)
//      dW += du (x) x,  db += sum du,  dg / d scale / d shift += ...
//
// One pass over HBM: dy, u and x are read once, dx is written once (the three-kernel version wrote du and re-read
// it, and re-read du / x once per 4x4 channel tile of dW).  A persistent CTA walks a contiguous range of
// (row, 128*P-position) tiles; per tile
//   phase 1: thread-per-position epilogue backward -> du tile (+1 halo each side) and x tile into shared memory
//   phase 2: dx for the thread's positions from the du tile (taps from shared memory, weights broadcast)
//   phase 3: dW as a small GEMM over the tile: thread (ci, segment) keeps dW[:, ci, :] in registers for the whole
//            CTA lifetime, streaming du / x rows with 128-bit shared loads
// and the parameter gradients leave the CTA once (shared-memory combine, then one global atomic per value).
// HBM-bound: algorithmic bytes per position = 4 * (2 * COUT + 2 * cin) (+ 4 * c1 with dadd / accumulate).
#include "common.cuh"

namespace dq {

struct ConvBwdFusedArgs {
  const float* dy;    // (R, COUT, L) gradient of the block output
  const float* u;     // (R, COUT, L) saved pre-norm conv output, or null: plain conv (du = dy)
  const float* g;     // (COUT) RMSNorm gain or null
  const float* ss;    // per-sample scale/shift (scale = ss[s*ss_stride + c], shift = [.. + COUT + c]) or null
  const float* x1;    // (R, c1, L) forward source 1
  const float* x2;    // (R, c2, L) forward source 2 or null
  const float* w;     // (COUT, c1+c2, K)
  const float* dadd;  // optional (R, c1, L): added to dx1 (identity-skip gradient)
  float* dx1;         // (R, c1, L) or null
  float* dx2;         // (R, c2, L) or null
  float* dw;          // (COUT, cin, K) accumulated
  float* db;          // (COUT) accumulated or null
  float* dg;          // (COUT) accumulated or null
  float* dss;         // same layout as ss, accumulated, or null
  int c1, c2, R, L, rows_per_sample, ss_stride, act, acc1, acc2, tiles_per_row, total_tiles, tiles_per_cta;
  // optional second, 1x1 convolution over the same input (ResnetBlock.res_conv, unet1d.py:299/322): its output gradient
  // dyo (R, COUT, L), weight wres (COUT, cin); dx gets wres^T dyo added, dwres / dbres are accumulated
  int al8 = 0;        // every tensor base is 8-byte aligned (set by the launcher)
  const float* dyo = nullptr;
  const float* wres = nullptr;
  float* dwres = nullptr;
  float* dbres = nullptr;
};

// VEC == 4: thread t owns positions 4t .. 4t+3 of the tile (128-bit global accesses; needs L % 4 == 0)
// VEC == 1: thread t owns positions t + 128 i (coalesced scalar accesses)
template <int COUT, int K, int P, int VEC>
__global__ void __launch_bounds__(128) conv_bwd_fused_kernel(ConvBwdFusedArgs a) {
  constexpr int TL = 128 * P;
  constexpr int DS = TL + 4;          // row stride of the smem tiles (= 4 mod 32); position p lives at index p + 4
  constexpr int H = (K - 1) / 2;      // halo
  constexpr int NPA = 4 * COUT;       // per-thread phase-1 accumulators: dg, dscale, dshift, db
  static_assert(VEC == 1 || (VEC == 4 && P == 4), "vector mode needs 4 positions per thread");
  extern __shared__ float4 dyn_smem4[];
  float* du_s = reinterpret_cast<float*>(dyn_smem4);   // COUT * DS + 8
  const int cin = a.c1 + a.c2;
  float* x_s = du_s + COUT * DS + 8;                   // cin * DS + 8
  float* w_s = x_s + cin * DS + 8;                     // COUT * cin * 4   [(co*cin + ci)*4 + k]
  float* dw_s = w_s + COUT * cin * 4;                  // COUT * cin * K   combine buffer
  float* red = dw_s + COUT * cin * K;                  // 4 * NPA
  const int tid = threadIdx.x;

  for (int i = tid; i < COUT * cin * 4; i += 128) {
    const int k = i & 3, pc = i >> 2;
    w_s[i] = (k < K) ? a.w[(size_t)pc * K + k] : 0.f;
  }
  for (int i = tid; i < COUT * cin * K; i += 128) dw_s[i] = 0.f;

  // phase-3 role: input channel ci, position segment seg
  const int nseg = max(1, 128 / cin);
  const int ci3 = tid % cin, seg = tid / cin;
  const bool p3_active = seg < nseg && tid < nseg * cin;
  const int SL = ((TL + nseg - 1) / nseg + 3) & ~3;
  const int q_begin = seg * SL, q_end = min(TL, q_begin + SL);
  float dwacc[COUT][K];
#pragma unroll
  for (int co = 0; co < COUT; ++co)
#pragma unroll
    for (int k = 0; k < K; ++k) dwacc[co][k] = 0.f;
  float pacc[NPA];
#pragma unroll
  for (int i = 0; i < NPA; ++i) pacc[i] = 0.f;

  const float sqrtC = sqrtf((float)COUT);
  const int t_begin = blockIdx.x * a.tiles_per_cta, t_end = min(a.total_tiles, t_begin + a.tiles_per_cta);
  int cur_sample = -1;

  auto flush_sample = [&](int sample) {   // per-sample scale/shift gradients leave the CTA when the sample changes
    float v[2 * COUT];
#pragma unroll
    for (int c = 0; c < 2 * COUT; ++c) { v[c] = pacc[COUT + c]; pacc[COUT + c] = 0.f; }
    const float tot = block_reduce_vec<2 * COUT>(v, red);
    if (a.dss && a.ss && tid < 2 * COUT) atomicAdd(a.dss + (size_t)sample * a.ss_stride + tid, tot);
  };

  for (int tile = t_begin; tile < t_end; ++tile) {
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int sample = r / a.rows_per_sample;
    if (sample != cur_sample) {
      if (cur_sample >= 0 && a.u) flush_sample(cur_sample);
      cur_sample = sample;
    }
    __syncthreads();  // previous tile's phases 2/3 are done with the tiles (also covers the w_s / dw_s init)

    // ---------------------------------------------------------------- phase 1: du tile and x tile
    {
      float gl[COUT], scale1[COUT], shift[COUT];
#pragma unroll
      for (int c = 0; c < COUT; ++c) {
        gl[c] = a.g ? a.g[c] : 1.f;
        scale1[c] = a.ss ? a.ss[(size_t)sample * a.ss_stride + c] + 1.f : 1.f;
        shift[c] = a.ss ? a.ss[(size_t)sample * a.ss_stride + COUT + c] : 0.f;
      }
      // P own positions, then (threads 0 / 1 only) the left / right halo position
      auto du_at = [&](const float (&dyv)[COUT], const float (&uvin)[COUT], float (&duv)[COUT], bool accumulate) {
        if (!a.u) {
#pragma unroll
          for (int c = 0; c < COUT; ++c) { duv[c] = dyv[c]; if (accumulate) pacc[3 * COUT + c] += dyv[c]; }
          return;
        }
        float uv[COUT];
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) { uv[c] = uvin[c]; s2 = fmaf(uv[c], uv[c], s2); }
        const float nrm = sqrtf(s2);
        const float inv = a.g ? 1.f / fmaxf(nrm, 1e-12f) : 1.f;
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          const float uh = uv[c] * inv;
          const float n = a.g ? uh * gl[c] * sqrtC : uv[c];
          const float z = fmaf(n, scale1[c], shift[c]);
          const float d = dyv[c] * act_bwd(z, a.act);
          const float dn = d * scale1[c];
          if (accumulate) {
            pacc[c] += dn * uh * sqrtC;        // d g
            pacc[COUT + c] += d * n;           // d scale
            pacc[2 * COUT + c] += d;           // d shift
          }
          const float duh = a.g ? dn * gl[c] * sqrtC : dn;
          duv[c] = duh;
          dot = fmaf(duh, uh, dot);
          uv[c] = uh;
        }
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          float d;
          if (!a.g) d = duv[c];
          else if (nrm > 1e-12f) d = (duv[c] - uv[c] * dot) * inv;
          else d = duv[c] * inv;
          duv[c] = d;
          if (accumulate) pacc[3 * COUT + c] += d;   // d bias
        }
      };
      const size_t rowbase = (size_t)r * COUT * a.L;
      if (VEC == 4) {
        const int l = tl0 + 4 * tid;
        const bool ok = l < a.L;
        float4 dy4[COUT], u4[COUT];
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          dy4[c] = ok ? __ldg(reinterpret_cast<const float4*>(a.dy + rowbase + (size_t)c * a.L + l)) : make_float4(0.f, 0.f, 0.f, 0.f);
          u4[c] = (ok && a.u) ? __ldg(reinterpret_cast<const float4*>(a.u + rowbase + (size_t)c * a.L + l)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float o[4][COUT];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float dyv[COUT], uv[COUT];
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            dyv[c] = i == 0 ? dy4[c].x : i == 1 ? dy4[c].y : i == 2 ? dy4[c].z : dy4[c].w;
            uv[c] = i == 0 ? u4[c].x : i == 1 ? u4[c].y : i == 2 ? u4[c].z : u4[c].w;
          }
          du_at(dyv, uv, o[i], ok);
          if (!ok) {
#pragma unroll
            for (int c = 0; c < COUT; ++c) o[i][c] = 0.f;
          }
        }
#pragma unroll
        for (int c = 0; c < COUT; ++c)
          *reinterpret_cast<float4*>(du_s + c * DS + 4 + 4 * tid) = make_float4(o[0][c], o[1][c], o[2][c], o[3][c]);
      } else {
#pragma unroll
        for (int i = 0; i < P; ++i) {
          const int l = tl0 + tid + 128 * i;
          const bool ok = l < a.L;
          float dyv[COUT], uv[COUT], o[COUT];
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            dyv[c] = ok ? __ldg(a.dy + rowbase + (size_t)c * a.L + l) : 0.f;
            uv[c] = (ok && a.u) ? __ldg(a.u + rowbase + (size_t)c * a.L + l) : 0.f;
          }
          du_at(dyv, uv, o, ok);
#pragma unroll
          for (int c = 0; c < COUT; ++c) du_s[c * DS + 4 + tid + 128 * i] = ok ? o[c] : 0.f;
        }
      }
      if (H > 0 && tid < 2) {  // halo positions tl0 - 1 (thread 0) and tl0 + TL (thread 1): no accumulation
        const int l = tid == 0 ? tl0 - 1 : tl0 + TL;
        const bool ok = l >= 0 && l < a.L;
        float dyv[COUT], uv[COUT], o[COUT];
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          dyv[c] = ok ? __ldg(a.dy + rowbase + (size_t)c * a.L + l) : 0.f;
          uv[c] = (ok && a.u) ? __ldg(a.u + rowbase + (size_t)c * a.L + l) : 0.f;
        }
        du_at(dyv, uv, o, false);
#pragma unroll
        for (int c = 0; c < COUT; ++c) du_s[c * DS + (tid == 0 ? 3 : TL + 4)] = ok ? o[c] : 0.f;
      }
      // x tile
      for (int ci = 0; ci < cin; ++ci) {
        const float* xr = (ci < a.c1) ? a.x1 + ((size_t)r * a.c1 + ci) * a.L : a.x2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.L;
        if (VEC == 4) {
          const int l = tl0 + 4 * tid;
          *reinterpret_cast<float4*>(x_s + ci * DS + 4 + 4 * tid) =
              (l < a.L) ? __ldg(reinterpret_cast<const float4*>(xr + l)) : make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
#pragma unroll
          for (int i = 0; i < P; ++i) {
            const int l = tl0 + tid + 128 * i;
            x_s[ci * DS + 4 + tid + 128 * i] = (l < a.L) ? __ldg(xr + l) : 0.f;
          }
        }
      }
      if (H > 0) {
        for (int i = tid; i < 2 * cin; i += 128) {
          const int ci = i >> 1, right = i & 1;
          const int l = right ? tl0 + TL : tl0 - 1;
          const float* xr = (ci < a.c1) ? a.x1 + ((size_t)r * a.c1 + ci) * a.L : a.x2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.L;
          x_s[ci * DS + (right ? TL + 4 : 3)] = (l >= 0 && l < a.L) ? __ldg(xr + l) : 0.f;
        }
      }
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 2: dx for the thread's positions
    if (a.dx1 || a.dx2) {
      for (int cb = 0; cb < cin; cb += 4) {
        float acc[4][P];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int i = 0; i < P; ++i) acc[j][i] = 0.f;
#pragma unroll 2
        for (int co = 0; co < COUT; ++co) {
          float dn[P][K];   // dn[i][k] = du[co][pos_i + H - k]
          if (VEC == 4) {
            const float4 m = *reinterpret_cast<const float4*>(du_s + co * DS + 4 + 4 * tid);
            if (K == 3) {
              const float lft = du_s[co * DS + 3 + 4 * tid], rgt = du_s[co * DS + 8 + 4 * tid];
              const float d6[6] = {lft, m.x, m.y, m.z, m.w, rgt};
#pragma unroll
              for (int i = 0; i < P; ++i)
#pragma unroll
                for (int k = 0; k < K; ++k) dn[i][k] = d6[i + 2 - k];
            } else {
              dn[0][0] = m.x; dn[1][0] = m.y; dn[2][0] = m.z; dn[3][0] = m.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < P; ++i)
#pragma unroll
              for (int k = 0; k < K; ++k) dn[i][k] = du_s[co * DS + 4 + tid + 128 * i + H - k];
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (cb + j < cin) {
              const float4 w4 = *reinterpret_cast<const float4*>(w_s + (co * cin + cb + j) * 4);
              const float wk[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
              for (int i = 0; i < P; ++i)
#pragma unroll
                for (int k = 0; k < K; ++k) acc[j][i] = fmaf(dn[i][k], wk[k], acc[j][i]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ci = cb + j;
          if (ci >= cin) continue;
          float* dst;
          int accf;
          const float* add = nullptr;
          if (ci < a.c1) {
            dst = a.dx1 ? a.dx1 + ((size_t)r * a.c1 + ci) * a.L : nullptr;
            accf = a.acc1;
            if (a.dadd) add = a.dadd + ((size_t)r * a.c1 + ci) * a.L;
          } else {
            dst = a.dx2 ? a.dx2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.L : nullptr;
            accf = a.acc2;
          }
          if (!dst) continue;
          if (VEC == 4) {
            const int l = tl0 + 4 * tid;
            if (l < a.L) {
              float4 v = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
              if (add) { const float4 q = __ldg(reinterpret_cast<const float4*>(add + l)); v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w; }
              if (accf) { const float4 q = *reinterpret_cast<const float4*>(dst + l); v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w; }
              *reinterpret_cast<float4*>(dst + l) = v;
            }
          } else {
#pragma unroll
            for (int i = 0; i < P; ++i) {
              const int l = tl0 + tid + 128 * i;
              if (l < a.L) {
                float v = acc[j][i];
                if (add) v += __ldg(add + l);
                if (accf) v += dst[l];
                dst[l] = v;
              }
            }
          }
        }
      }
    }

    // ---------------------------------------------------------------- phase 3: dW[:, ci3, :] over this thread's segment
    if (p3_active) {
      const float* xr = x_s + ci3 * DS + 4;
      for (int q = q_begin; q < q_end; q += 4) {
        const float4 xm = *reinterpret_cast<const float4*>(xr + q);
        float x6[6] = {0.f, xm.x, xm.y, xm.z, xm.w, 0.f};
        if (K == 3) { x6[0] = xr[q - 1]; x6[5] = xr[q + 4]; }
#pragma unroll
        for (int co = 0; co < COUT; ++co) {
          const float4 d4 = *reinterpret_cast<const float4*>(du_s + co * DS + 4 + q);
          const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
          for (int k = 0; k < K; ++k)
#pragma unroll
            for (int i = 0; i < 4; ++i) dwacc[co][k] = fmaf(dd[i], x6[i + k + 1 - H], dwacc[co][k]);
        }
      }
    }
  }

  // ------------------------------------------------------------------ leave: parameter gradients
  if (cur_sample >= 0 && a.u) flush_sample(cur_sample);
  if (p3_active) {
#pragma unroll
    for (int co = 0; co < COUT; ++co)
#pragma unroll
      for (int k = 0; k < K; ++k) atomicAdd(dw_s + (co * cin + ci3) * K + k, dwacc[co][k]);
  }
  {
    float v[2 * COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) { v[c] = pacc[c]; v[COUT + c] = pacc[3 * COUT + c]; }
    const float tot = block_reduce_vec<2 * COUT>(v, red);   // includes the __syncthreads that publishes dw_s
    if (tid < COUT) { if (a.dg && a.g && a.u) atomicAdd(a.dg + tid, tot); }
    else if (tid < 2 * COUT) { if (a.db) atomicAdd(a.db + tid - COUT, tot); }
  }
  for (int i = tid; i < COUT * cin * K; i += 128) atomicAdd(a.dw + i, dw_s[i]);
}

// =====================================================================================================================
// Pipelined variant (L % 4 == 0): the raw dy / u / x rows of a tile are brought into shared memory by 1-D bulk
// async copies (cp.async.bulk, the TMA engine) that complete on an mbarrier, two tiles deep, so the HBM latency of
// tile t+1 / t+2 hides behind the arithmetic of tile t and no thread spends issue slots on global address math.
// A row of a stage holds positions [tl0-4, tl0+TL+4) at indices [0, TL+8); row stride TS = TL + 36 (= 4 mod 32).
__device__ __forceinline__ uint32_t cf_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cf_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void cf_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cf_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void cf_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ float cf_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float cf_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float cf_rsqrt(float x) {
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// TF32 helpers of the tensor-core variant of the backward kernel
__device__ __forceinline__ uint32_t cf_rtf(float x) { return __float_as_uint(x) + 0x1000u; }   // RN-even-ish: + half ulp, HW truncates
__device__ __forceinline__ uint32_t cf_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void cf_mma8(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cf_mma8_z(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.f));
}
// acc{0,1} += x * w{0,1} as ONE packed FFMA2 (Blackwell fma.rn.f32x2): halves the issue slots of the FMA-bound loops
__device__ __forceinline__ void cf_fma2(float& a0, float& a1, float x, float w0, float w1) {
  unsigned long long acc, xx, ww;
  asm("mov.b64 %0, {%1, %2};" : "=l"(acc) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(xx) : "f"(x));
  asm("mov.b64 %0, {%1, %2};" : "=l"(ww) : "f"(w0), "f"(w1));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(xx), "l"(ww));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(acc));
}
// d SiLU(z) / dz with single-MUFU exp / reciprocal (|rel err| ~ 1e-6)
__device__ __forceinline__ float cf_dsilu(float z) {
  const float s = cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
  return s * fmaf(z, 1.f - s, 1.f);
}

// EPI = false: plain conv (du = dy).  EPI = true: RMSNorm (g) + optional per-sample scale/shift + SiLU epilogue.
// BULK = true: rows are 16-byte aligned, one cp.async.bulk per row.  BULK = false: any alignment (L % 4 != 0, i.e. the
// L = 1250 / 625 levels): every thread stages its share of the tile with 4-byte cp.async (LDGSTS) that arrive on the same
// mbarrier; everything downstream of the staging is identical.
// NCI > 0: phases 2 and 3 run on the tensor cores (mma.sync m16n8k8 TF32, fp32 accumulate) with NCI n8-tiles over the
// input channels; du is stored TF32-rounded by phase 1, x / dyo fragments are rounded when loaded, weights once.
// Used for COUT >= 8, where the FFMA form of the two contractions (2 * 3 * COUT * cin FMAs per position) is what bounds
// the kernel.  Fragment k-slots are permuted (slot t <-> channel 2t, slot t+4 <-> channel 2t+1) so that with the row
// stride TS = 4 (mod 32) every fragment load covers the 32 banks once.
// UP2: the forward input was the nearest-x2 upsampling of HALF-rate rows (Upsample = nearest x2 + Conv1d k3,
// unet1d.py:93-96): x1 / dx1 are (R, c1, L / 2); the half-rate rows are staged (x_up[q] = x[q >> 1] is resolved when the
// wgrad taps are read) and d x_up is folded pairwise before it is stored - the upsampled tensor and its gradient never
// exist (they were two extra passes, dq_upsample2x / dq_fold2x, and doubled the x / dx bytes of this kernel).
// DOWN2: backward of Downsample = Conv1d(k4, stride 2, pad 1) (unet1d.py:110): dy is (R, COUT, L / 2) and its HALF-rate rows
// are staged; d x[2j] = W1 dy[j] + W3 dy[j-1], d x[2j+1] = W0 dy[j+1] + W2 dy[j]; dW_k = sum_m dy[m] x[2m + k - 1] - no
// space-to-depth copy of x, no depth-to-space pass over dx, no weight re-packing (dq_s2d / dq_d2s / dq_down_w).
template <int COUT, int K, int P, int NT, bool EPI, bool BULK, bool RES = false, int NCI = 0, bool UP2 = false,
          bool DOWN2 = false>
// (no minimum-blocks argument: an explicit `1` makes ptxas spend 152 instead of 128 registers on the 4-channel variants -
// three instead of four resident CTAs, level-0 ResnetBlock backward 1362 -> 1495 us; asking for three CTAs of the
// tensor-core variants changes nothing at 8 channels and spills at 12 / 16, DESIGN.md section 4)
// (the 4-channel res_conv variant is the exception: shared memory limits it to two CTAs anyway, and with the explicit `1`
// it keeps 161 registers instead of spilling at 128: 2131 -> 2046 us at level 0; 0 = no request)
__global__ void __launch_bounds__(NT, (RES && NCI == 0 && COUT == 4) ? 1 : 0) conv_bwd_fused_tma_kernel(ConvBwdFusedArgs a) {
  constexpr bool MMA = NCI > 0;
  static_assert(!MMA || (EPI && K == 3), "MMA variant: conv3 with epilogue");
  static_assert(!UP2 || (!EPI && !RES && !MMA && K == 3 && P >= 2), "UP2: plain conv3, FFMA contractions, pairs per thread");
  static_assert(!DOWN2 || (!EPI && !RES && !MMA && !UP2 && K == 4 && P >= 2), "DOWN2: plain conv k4 s2, FFMA contractions");
  constexpr int KCO = (COUT + 7) / 8;                    // k8 / n8 tiles over the output channels (rows >= COUT: zero weights)
  constexpr int MCI = (NCI + 1) / 2 > 0 ? (NCI + 1) / 2 : 1;   // m16 tiles over the input channels (phase 3)
  constexpr int TL = NT * P;
  constexpr int TS = TL + 36;
  constexpr int H = (K - 1) / 2;
  constexpr int NW = NT / 32;
  constexpr int DYR = EPI ? 2 * COUT : COUT;             // dy rows, [u rows]
  static_assert(P == 1 || P == 2 || P == 4, "P");
  extern __shared__ float4 dyn_smem4[];
  const int cin = a.c1 + a.c2;                           // multiple of 4 (checked by the launcher), as is c1
  const int rows = DYR + cin + (RES ? COUT : 0);         // RES: + the res_conv output-gradient rows
  float* stage0 = reinterpret_cast<float*>(dyn_smem4);
  const int stage_floats = rows * TS;
  float* w_s = stage0 + 2 * stage_floats;                // COUT * cin * 4
  float* dw_s = w_s + (MMA ? 0 : COUT * cin * 4);        // COUT * cin * K (MMA: weights live in fragments, no w_s)
  float* wres_s = dw_s + COUT * cin * K;                 // RES: COUT * cin
  float* dwres_s = wres_s + (RES ? COUT * cin : 0);      // RES: COUT * cin
  float* red = dwres_s + (RES ? COUT * cin : 0);         // NW * 2 * COUT
  uint64_t* bars = reinterpret_cast<uint64_t*>(red + NW * 2 * COUT);
  // MMA variant: the identity-skip gradient (dadd) and the destination's old contents (acc1) of the tile are copied
  // into shared memory during phase 1 ([c1][TS] each, position p at index p + 4): read from global memory in the
  // phase-2 epilogue they were its long-scoreboard stall (ncu: block1 backward took 2x block2 at 12 channels)
  float* add_s = reinterpret_cast<float*>(bars + 2);
  constexpr bool STG = MMA && !RES;   // (the res_conv variant has neither dadd nor an accumulating destination)
  const bool st_add = STG && a.dadd != nullptr && a.dx1 != nullptr, st_acc = STG && a.acc1 != 0 && a.dx1 != nullptr;
  float* acc_s = add_s + (st_add ? a.c1 * TS : 0);
  const int tid = threadIdx.x;
  const uint32_t bar0 = cf_smem_u32(bars), bar1 = bar0 + 8;

  if (tid == 0) {
    cf_mbar_init(bar0, BULK ? 1 : NT);
    cf_mbar_init(bar1, BULK ? 1 : NT);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (!MMA)
    for (int i = tid; i < COUT * cin * 4; i += NT) {
      const int k = i & 3, pc = i >> 2;
      w_s[i] = (k < K) ? a.w[(size_t)pc * K + k] : 0.f;
    }
  for (int i = tid; i < COUT * cin * K; i += NT) dw_s[i] = 0.f;
  if (RES)
    for (int i = tid; i < COUT * cin; i += NT) { wres_s[i] = a.wres[i]; dwres_s[i] = 0.f; }
  // stage slots that no copy ever fills (beyond a row end) must hold finite values: 0 * stale stays 0
  for (int i = tid; i < 2 * stage_floats; i += NT) stage0[i] = 0.f;
  __syncthreads();

  const int t_begin = blockIdx.x * a.tiles_per_cta, t_end = min(a.total_tiles, t_begin + a.tiles_per_cta);
  const int n_tiles = t_end - t_begin;

  // BULK: one lane per row issues that row's bulk copy; lane 0 posts the expected byte count first
  auto issue = [&](int tile, int s) {
    if (!BULK) {
      // unaligned rows: one warp per row (the row pointer is computed once per warp and row), lanes stride over the
      // elements with 8-byte copies when every row of the tensor starts 8-byte aligned (even L), else 4-byte ones
      const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
      const int l_lo = max(0, tl0 - 4), l_hi = min(a.L, tl0 + TL + 4);
      const int w = l_hi - l_lo, doff = l_lo - (tl0 - 4);
      float* st = stage0 + s * stage_floats;
      const bool even = ((a.L | w | l_lo) & 1) == 0 && a.al8;
      for (int row = tid >> 5; row < rows; row += NW) {
        if ((UP2 && row >= DYR) || (DOWN2 && row < DYR)) {   // half-rate source rows: window [tl0 / 2 - 4, tl0 / 2 + TL / 2 + 4)
          const int Lh = a.L >> 1, h0 = (tl0 >> 1) - 4;
          const int h_lo = max(0, h0), h_hi = min(Lh, h0 + TL / 2 + 8), wh = h_hi - h_lo;
          const float* srch = (DOWN2 ? a.dy + ((size_t)r * COUT + row) * Lh : a.x1 + ((size_t)r * a.c1 + (row - DYR)) * Lh) + h_lo;
          const uint32_t dsth = cf_smem_u32(st + row * TS + (h_lo - h0));
          if (((Lh | wh | h_lo) & 1) == 0 && a.al8) {
            for (int e = (tid & 31) * 2; e < wh; e += 64)
              asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dsth + 4u * (uint32_t)e), "l"(srch + e) : "memory");
          } else {
            for (int e = tid & 31; e < wh; e += 32)
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dsth + 4u * (uint32_t)e), "l"(srch + e) : "memory");
          }
          continue;
        }
        const float* src;
        if (row < COUT) src = a.dy + ((size_t)r * COUT + row) * a.L;
        else if (row < DYR) src = a.u + ((size_t)r * COUT + (row - COUT)) * a.L;
        else if (RES && row >= DYR + cin) src = a.dyo + ((size_t)r * COUT + (row - DYR - cin)) * a.L;
        else {
          const int ci = row - DYR;
          src = (ci < a.c1) ? a.x1 + ((size_t)r * a.c1 + ci) * a.L : a.x2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.L;
        }
        src += l_lo;
        const uint32_t dst = cf_smem_u32(st + row * TS + doff);
        if (even) {
          for (int e = (tid & 31) * 2; e < w; e += 64)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
        } else {
          for (int e = tid & 31; e < w; e += 32)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
        }
      }
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(s ? bar1 : bar0) : "memory");
      return;
    }
    {
      // the row copies are spread over ALL warps (row = warp + NW * lane): issued from one warp, the ~rows serialized
      // UBLKCP iterations made that warp the straggler of the next phase-1 barrier.  Thread 0 posts the expected byte
      // count; copies of other warps may complete first (the tx-count may go negative, the phase cannot complete
      // before thread 0's arrive).
      const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
      const int l_lo = max(0, tl0 - 4), l_hi = min(a.L, tl0 + TL + 4);
      const uint32_t bytes = (uint32_t)(l_hi - l_lo) * 4u;
      const uint32_t bar = s ? bar1 : bar0;
      const int row = (tid >> 5) + NW * (tid & 31);
      if (tid == 0 || row < rows) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      const int Lh = a.L >> 1, h0 = (tl0 >> 1) - 4;
      const int h_lo = max(0, h0), h_hi = min(Lh, h0 + TL / 2 + 8);
      const uint32_t bytes_h = (uint32_t)(h_hi - h_lo) * 4u;
      const uint32_t bytes_x = UP2 ? bytes_h : bytes, bytes_d = DOWN2 ? bytes_h : bytes;
      if (tid == 0) cf_mbar_expect_tx(bar, bytes_d * (uint32_t)(rows - cin) + bytes_x * (uint32_t)cin);
      float* st = stage0 + s * stage_floats;
      if (UP2 && row >= DYR && row < rows) {
        cf_bulk_g2s(cf_smem_u32(st + row * TS + (h_lo - h0)), a.x1 + ((size_t)r * a.c1 + (row - DYR)) * Lh + h_lo, bytes_x, bar);
      } else if (DOWN2 && row < DYR) {
        cf_bulk_g2s(cf_smem_u32(st + row * TS + (h_lo - h0)), a.dy + ((size_t)r * COUT + row) * Lh + h_lo, bytes_d, bar);
      } else
      if (row < rows) {
        const float* src;
        if (row < COUT) src = a.dy + ((size_t)r * COUT + row) * a.L;
        else if (row < DYR) src = a.u + ((size_t)r * COUT + (row - COUT)) * a.L;
        else if (RES && row >= DYR + cin) src = a.dyo + ((size_t)r * COUT + (row - DYR - cin)) * a.L;
        else {
          const int ci = row - DYR;
          src = (ci < a.c1) ? a.x1 + ((size_t)r * a.c1 + ci) * a.L : a.x2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.L;
        }
        cf_bulk_g2s(cf_smem_u32(st + row * TS + (l_lo - (tl0 - 4))), src + l_lo, bytes, bar);
      }
    }
  };
  // staged copies of a tile's dadd / old-dx1 rows: issued one tile ahead (after the end-of-tile barrier, before the stage
  // prefetch) and committed as a cp.async group of their own, so that waiting for them (before phase 2 of their tile)
  // never waits for the younger, uncommitted stage copies of the unaligned-row pipeline
  auto issue_add = [&](int tile) {
    if constexpr (STG) {
      if (st_add || st_acc) {   // CTA-uniform
        const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
        const int wv = min(TL, a.L - tl0);
        const int nrow = a.c1 * ((st_add ? 1 : 0) + (st_acc ? 1 : 0));
        for (int row = tid >> 5; row < nrow; row += NW) {
          const bool second = row >= a.c1;
          const int ci = second ? row - a.c1 : row;
          const float* src = ((st_add && !second) ? a.dadd : a.dx1) + ((size_t)r * a.c1 + ci) * a.L + tl0;
          const uint32_t dst = cf_smem_u32(add_s + row * TS + 4);
          if (BULK && (wv & 3) == 0 && (reinterpret_cast<size_t>(src) & 15) == 0) {
            for (int e = (tid & 31) * 4; e < wv; e += 128)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
          } else {
            for (int e = tid & 31; e < wv; e += 32)
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      }
    }
  };
  if (n_tiles > 0) issue_add(t_begin);
  if (n_tiles > 0) issue(t_begin, 0);
  if (n_tiles > 1) issue(t_begin + 1, 1);

  // phase-3 role: input channel ci3, position segment seg
  const int nseg = max(1, NT / cin);
  const int ci3 = tid % cin, seg = tid / cin;
  const bool p3_active = tid < nseg * cin;
  const int SL = ((TL + nseg - 1) / nseg + 3) & ~3;
  const int q_begin = seg * SL, q_end = min(TL, q_begin + SL);
  float dwacc[MMA ? 1 : COUT][K];
#pragma unroll
  for (int co = 0; co < (MMA ? 1 : COUT); ++co)
#pragma unroll
    for (int k = 0; k < K; ++k) dwacc[co][k] = 0.f;
  // MMA variant: weight fragments (B operand of phase 2) and the dW accumulators (phase 3), per warp
  const int lane_ = tid & 31, warp_ = tid >> 5, fg = lane_ >> 2, ft = lane_ & 3;
  uint32_t wB[MMA ? K : 1][KCO][MMA ? NCI : 1][2], wR[KCO][MMA && RES ? NCI : 1][2];
  float dWf[MMA ? K : 1][MCI][KCO][4], dRf[MCI][KCO][4];
  if constexpr (MMA) {
#pragma unroll
    for (int kc = 0; kc < KCO; ++kc)
#pragma unroll
      for (int nt = 0; nt < NCI; ++nt)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int co = 8 * kc + 2 * ft + i, ci = 8 * nt + fg;
          const bool in = ci < cin && co < COUT;
#pragma unroll
          for (int kk = 0; kk < K; ++kk) wB[kk][kc][nt][i] = cf_tf32(in ? a.w[((size_t)co * cin + ci) * K + kk] : 0.f);
          if constexpr (RES) wR[kc][nt][i] = cf_tf32(in ? a.wres[(size_t)co * cin + ci] : 0.f);
        }
#pragma unroll
    for (int mt = 0; mt < MCI; ++mt)
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int kk = 0; kk < K; ++kk) dWf[kk][mt][nt][i] = 0.f;
          dRf[mt][nt][i] = 0.f;
        }
  }
  // per-thread partial sums: S = sum d*uhat, T = sum d (current sample), B = sum du (bias), G = d g / sqrt(C)
  float accS[COUT], accT[COUT], accB[COUT], accG[COUT];
#pragma unroll
  for (int c = 0; c < COUT; ++c) accS[c] = accT[c] = accB[c] = accG[c] = 0.f;
  float dwres[RES ? COUT : 1], accR[RES ? COUT : 1];    // RES: dWres[:, ci3] of this thread's segment, sum of dyo
#pragma unroll
  for (int c = 0; c < (RES ? COUT : 1); ++c) dwres[c] = accR[c] = 0.f;
  const float sqrtC = sqrtf((float)COUT);
  const bool has_ss = a.ss != nullptr;
  int cur_sample = -1;

  auto block_sum2c = [&](float (&v)[2 * COUT]) -> float {   // thread i < 2*COUT returns the block total of v[i]
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int i = 0; i < 2 * COUT; ++i) {
      const float sres = warp_sum(v[i]);
      if (lane == 0) red[warp * 2 * COUT + i] = sres;
    }
    __syncthreads();
    float out = 0.f;
    if (tid < 2 * COUT)
      for (int w = 0; w < NW; ++w) out += red[w * 2 * COUT + tid];
    __syncthreads();
    return out;
  };
  // d scale[c] = g[c] sqrt(C) S[c], d shift[c] = T[c] leave the CTA when the sample changes; d g picks up scale1 * S
  auto flush_sample = [&](int sample) {
    float v[2 * COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) {
      const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + c] + 1.f : 1.f;
      accG[c] = fmaf(sc1, accS[c], accG[c]);
      v[c] = accS[c] * a.g[c] * sqrtC;
      v[COUT + c] = accT[c];
      accS[c] = 0.f; accT[c] = 0.f;
    }
    if (a.dss && has_ss) {   // CTA-uniform
      const float tot = block_sum2c(v);
      if (tid < 2 * COUT) atomicAdd(a.dss + (size_t)sample * a.ss_stride + tid, tot);
    }
  };

  for (int it = 0; it < n_tiles; ++it) {
    const int tile = t_begin + it, s = it & 1;
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int sample = r / a.rows_per_sample;
    if (EPI && sample != cur_sample) {
      if (cur_sample >= 0) flush_sample(cur_sample);
      cur_sample = sample;
    }
    float* du_s = stage0 + s * stage_floats;                 // dy rows, overwritten in place by du
    const float* u_t = du_s + COUT * TS;                     // [COUT][TS] (EPI only)
    float* x_t = du_s + DYR * TS;                            // [cin][TS]
    float* yo_t = x_t + cin * TS;                            // RES: [COUT][TS]
    cf_mbar_wait(s ? bar1 : bar0, (uint32_t)((it >> 1) & 1));

    // ---------------------------------------------------------------- phase 1: du tile (in place of dy)
    if (EPI) {
      float gs[COUT], shift[COUT];
#pragma unroll
      for (int c = 0; c < COUT; ++c) {
        const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + c] + 1.f : 1.f;
        gs[c] = a.g[c] * sqrtC * sc1;
        shift[c] = has_ss ? a.ss[(size_t)sample * a.ss_stride + COUT + c] : 0.f;
      }
      // inputs of non-existent positions are zeroed at load time, which makes every derived quantity exactly 0
      auto du_at = [&](float (&dv)[COUT], const float (&uvin)[COUT], bool accumulate) {   // dv: dy in, du out
        float uh[COUT];
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) s2 = fmaf(uvin[c], uvin[c], s2);
        const bool big = s2 > 1e-24f;                        // ||u|| > 1e-12 (F.normalize eps)
        const float inv = big ? cf_rsqrt(s2) : 1e12f;
        float dot = 0.f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          uh[c] = uvin[c] * inv;
          const float z = fmaf(uh[c], gs[c], shift[c]);
          const float d = dv[c] * cf_dsilu(z);
          if (accumulate) { accS[c] = fmaf(d, uh[c], accS[c]); accT[c] += d; }
          dv[c] = d * gs[c];                                 // d u-hat
          dot = fmaf(dv[c], uh[c], dot);
        }
        const float k = big ? dot : 0.f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          dv[c] = (dv[c] - uh[c] * k) * inv;
          if (accumulate) accB[c] += dv[c];
        }
      };
      {
        const int idx = 4 + P * tid;
        float dyv[P][COUT], uv[P][COUT];
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (P == 4) {
            const float4 d4 = *reinterpret_cast<const float4*>(du_s + c * TS + idx);
            dyv[0][c] = d4.x; dyv[1][c] = d4.y; dyv[2][c] = d4.z; dyv[3][c] = d4.w;
            const float4 u4 = *reinterpret_cast<const float4*>(u_t + c * TS + idx);
            uv[0][c] = u4.x; uv[1][c] = u4.y; uv[2][c] = u4.z; uv[3][c] = u4.w;
          } else if constexpr (P == 2) {
            const float2 d2 = *reinterpret_cast<const float2*>(du_s + c * TS + idx);
            dyv[0][c] = d2.x; dyv[P - 1][c] = d2.y;
            const float2 u2 = *reinterpret_cast<const float2*>(u_t + c * TS + idx);
            uv[0][c] = u2.x; uv[P - 1][c] = u2.y;
          } else {
            dyv[0][c] = du_s[c * TS + idx];
            uv[0][c] = u_t[c * TS + idx];
          }
        }
        // positions at or beyond the row end do not exist (with unaligned rows a thread's group can straddle the end)
        const int nvalid = a.L - (tl0 + P * tid);
        if (nvalid < P) {
#pragma unroll
          for (int i = 0; i < P; ++i)
            if (i >= nvalid) {
#pragma unroll
              for (int c = 0; c < COUT; ++c) { dyv[i][c] = 0.f; uv[i][c] = 0.f; }
            }
        }
#pragma unroll
        for (int i = 0; i < P; ++i) du_at(dyv[i], uv[i], true);
        if constexpr (MMA) {   // operands of the TF32 contractions: round to nearest once, here
#pragma unroll
          for (int i = 0; i < P; ++i)
#pragma unroll
            for (int c = 0; c < COUT; ++c) dyv[i][c] = __uint_as_float(cf_rtf(dyv[i][c]));
        }
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (P == 4) *reinterpret_cast<float4*>(du_s + c * TS + idx) = make_float4(dyv[0][c], dyv[1][c], dyv[2][c], dyv[3][c]);
          else if constexpr (P == 2) *reinterpret_cast<float2*>(du_s + c * TS + idx) = make_float2(dyv[0][c], dyv[P - 1][c]);
          else du_s[c * TS + idx] = dyv[0][c];
        }
      }
      if (H > 0 && tid < 32) {
        // halo positions tl0 - 1 (lanes 0-15) and tl0 + TL (lanes 16-31), one CHANNEL per lane with shuffle reductions:
        // a serial per-thread evaluation here made warp 0 / 3 the stragglers of the phase-1 barrier (13-18 % of the
        // kernel in ncu's stall samples)
        const int side = tid >> 4, c = tid & 15;
        const int idx = side == 0 ? 3 : TL + 4;
        const int l = tl0 - 4 + idx;
        const bool ok = l >= 0 && l < a.L && c < COUT;
        const int cc = c < COUT ? c : 0;
        const float dyv = ok ? du_s[cc * TS + idx] : 0.f;
        const float uvv = ok ? u_t[cc * TS + idx] : 0.f;
        float s2 = uvv * uvv;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        const bool big = s2 > 1e-24f;
        const float inv = big ? cf_rsqrt(s2) : 1e12f;
        const float uh = uvv * inv;
        // this lane's channel constants straight from memory (indexing the register arrays by lane would spill them)
        const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + cc] + 1.f : 1.f;
        const float gsc = a.g[cc] * sqrtC * sc1;
        const float shc = has_ss ? a.ss[(size_t)sample * a.ss_stride + COUT + cc] : 0.f;
        const float z = fmaf(uh, gsc, shc);
        const float d = dyv * cf_dsilu(z);
        float dv = d * gsc;
        float dot = dv * uh;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
        dv = (dv - uh * (big ? dot : 0.f)) * inv;
        if (MMA) dv = __uint_as_float(cf_rtf(dv));
        if (c < COUT) du_s[c * TS + idx] = ok ? dv : 0.f;
      }
    } else {
      // plain conv: du = dy already sits in the stage; zero the non-existent positions and accumulate the bias gradient
      // (DOWN2: the dy tile has TL / 2 half-rate positions, handled by the first half of the threads)
      const int idx = 4 + P * tid;
      const int nvalid = DOWN2 ? (a.L >> 1) - ((tl0 >> 1) + P * tid) : a.L - (tl0 + P * tid);
      if (DOWN2 && P * tid >= TL / 2) {
      } else
      if (nvalid >= P) {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (P == 4) { const float4 d4 = *reinterpret_cast<const float4*>(du_s + c * TS + idx); accB[c] += (d4.x + d4.y) + (d4.z + d4.w); }
          else if constexpr (P == 2) { const float2 d2 = *reinterpret_cast<const float2*>(du_s + c * TS + idx); accB[c] += d2.x + d2.y; }
          else accB[c] += du_s[c * TS + idx];
        }
      } else {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
#pragma unroll
          for (int i = 0; i < P; ++i) {
            if (i < nvalid) accB[c] += du_s[c * TS + idx + i];
            else du_s[c * TS + idx + i] = 0.f;
          }
        }
      }
      if (H > 0 && tid < COUT) {
        if (tl0 == 0) du_s[tid * TS + 3] = 0.f;
        if (a.L <= tl0 + TL) du_s[tid * TS + (DOWN2 ? ((a.L - tl0) >> 1) : (a.L - tl0)) + 4] = 0.f;
      }
    }
    if constexpr (RES) {   // bias gradient of the 1x1 conv; non-existent positions are zeroed for phase 3
      const int idx = 4 + P * tid;
      const int nvalid = a.L - (tl0 + P * tid);
      if (nvalid >= P) {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (P == 4) { const float4 d4 = *reinterpret_cast<const float4*>(yo_t + c * TS + idx); accR[c] += (d4.x + d4.y) + (d4.z + d4.w); }
          else if constexpr (P == 2) { const float2 d2 = *reinterpret_cast<const float2*>(yo_t + c * TS + idx); accR[c] += d2.x + d2.y; }
          else accR[c] += yo_t[c * TS + idx];
        }
      } else {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
#pragma unroll
          for (int i = 0; i < P; ++i) {
            if (i < nvalid) accR[c] += yo_t[c * TS + idx + i];
            else yo_t[c * TS + idx + i] = 0.f;
          }
        }
      }
    }
    // x rows: exact zeros at the two out-of-range neighbours a valid du can touch (row start / row end)
    if (H > 0 && tid < cin) {
      if (tl0 == 0) x_t[tid * TS + 3] = 0.f;
      if (a.L <= tl0 + TL) x_t[tid * TS + (UP2 ? ((a.L - tl0) >> 1) : (a.L - tl0)) + 4] = 0.f;
    }
    if constexpr (STG) {
      if (st_add || st_acc) asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();

    // ---------------------------------------------------------------- phase 2: dx for the thread's positions
    if constexpr (MMA) {
      if (a.dx1 || a.dx2) {
        // warp w: slabs of 16 positions w, w + NW, ..; D[pos][ci] = sum_k A_k[pos][co] W_k[co][ci] (+ dyo wres)
        // destination rows of this thread's channel pairs (ci = 8nt + 2ft, +1), fixed for the whole tile
        float* dstp[NCI];
        const float* addp[NCI];   // shared-memory copies of the tile (dadd rows, then the old dx1 rows)
        const float* oldp[NCI];
        bool accp[NCI];
#pragma unroll
        for (int nt = 0; nt < NCI; ++nt) {
          const int ci = 8 * nt + 2 * ft;
          dstp[nt] = nullptr; addp[nt] = nullptr; oldp[nt] = nullptr; accp[nt] = false;
          if (ci < a.c1) {
            if (a.dx1) dstp[nt] = a.dx1 + ((size_t)r * a.c1 + ci) * a.L + tl0 + fg;
            if (st_add) addp[nt] = add_s + ci * TS + 4 + fg;
            if (st_acc) oldp[nt] = acc_s + ci * TS + 4 + fg;
          } else if (ci < cin) {
            if (a.dx2) dstp[nt] = a.dx2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.L + tl0 + fg;
            accp[nt] = a.acc2 != 0;
          }
        }
        const bool full = tl0 + TL <= a.L;   // CTA-uniform: no per-position bound checks
        for (int sl = warp_; sl < TL / 16; sl += NW) {
          const int p0 = 16 * sl;
          float d[NCI][4];
#pragma unroll
          for (int kk = 0; kk < K; ++kk)
#pragma unroll
            for (int kc = 0; kc < KCO; ++kc) {
              // channel rows >= COUT (COUT = 12) meet zero weights: any finite row will do
              const float* ap = du_s + min(8 * kc + 2 * ft, COUT - 2) * TS + 4 + p0 + fg + H - kk;
              const uint32_t a0 = __float_as_uint(ap[0]), a1 = __float_as_uint(ap[8]);
              const uint32_t a2 = __float_as_uint(ap[TS]), a3 = __float_as_uint(ap[TS + 8]);
#pragma unroll
              for (int nt = 0; nt < NCI; ++nt) {
                if (kk == 0 && kc == 0) cf_mma8_z(d[nt], a0, a1, a2, a3, wB[kk][kc][nt][0], wB[kk][kc][nt][1]);
                else cf_mma8(d[nt], a0, a1, a2, a3, wB[kk][kc][nt][0], wB[kk][kc][nt][1]);
              }
            }
          if constexpr (RES) {
#pragma unroll
            for (int kc = 0; kc < KCO; ++kc) {
              const float* ap = yo_t + min(8 * kc + 2 * ft, COUT - 2) * TS + 4 + p0 + fg;
              const uint32_t a0 = cf_rtf(ap[0]), a1 = cf_rtf(ap[8]), a2 = cf_rtf(ap[TS]), a3 = cf_rtf(ap[TS + 8]);
#pragma unroll
              for (int nt = 0; nt < NCI; ++nt) cf_mma8(d[nt], a0, a1, a2, a3, wR[kc][nt][0], wR[kc][nt][1]);
            }
          }
          // thread holds (pos p0+fg | p0+fg+8, ci 8nt+2ft | +1)
          const bool ok0 = full || tl0 + p0 + fg < a.L, ok1 = full || tl0 + p0 + fg + 8 < a.L;
#pragma unroll
          for (int nt = 0; nt < NCI; ++nt) {
            if (!dstp[nt]) continue;   // warp-uniform per nt only when c1 is a multiple of 8; divergence is harmless
            float* q0 = dstp[nt] + p0;
            float* q1 = q0 + a.L;
            if (addp[nt] || oldp[nt] || accp[nt]) {
              float e[4] = {0.f, 0.f, 0.f, 0.f};
              if (addp[nt]) {
                const float* z0 = addp[nt] + p0;
                const float* z1 = z0 + TS;
                if (ok0) { e[0] += z0[0]; e[1] += z1[0]; }
                if (ok1) { e[2] += z0[8]; e[3] += z1[8]; }
              }
              if (oldp[nt]) {
                const float* z0 = oldp[nt] + p0;
                const float* z1 = z0 + TS;
                if (ok0) { e[0] += z0[0]; e[1] += z1[0]; }
                if (ok1) { e[2] += z0[8]; e[3] += z1[8]; }
              }
              if (accp[nt]) {
                if (ok0) { e[0] += q0[0]; e[1] += q1[0]; }
                if (ok1) { e[2] += q0[8]; e[3] += q1[8]; }
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) d[nt][i] += e[i];
            }
            if (ok0) { q0[0] = d[nt][0]; q1[0] = d[nt][1]; }
            if (ok1) { q0[8] = d[nt][2]; q1[8] = d[nt][3]; }
          }
        }
      }
    } else
    if (a.dx1 || a.dx2) {
      const int l = tl0 + P * tid;
      const bool ok = l < a.L;
      for (int cb = 0; cb < cin; cb += 4) {
        float* dst;
        const float* add = nullptr;
        int accf;
        if (UP2) {
          dst = a.dx1 ? a.dx1 + ((size_t)r * a.c1 + cb) * (a.L >> 1) + (l >> 1) : nullptr;
          accf = a.acc1;
        } else if (cb < a.c1) {
          dst = a.dx1 ? a.dx1 + ((size_t)r * a.c1 + cb) * a.L + l : nullptr;
          accf = a.acc1;
          if (a.dadd) add = a.dadd + ((size_t)r * a.c1 + cb) * a.L + l;
        } else {
          dst = a.dx2 ? a.dx2 + ((size_t)r * a.c2 + (cb - a.c1)) * a.L + l : nullptr;
          accf = a.acc2;
        }
        if (!dst) continue;   // CTA-uniform
        // accumulate / identity-skip inputs are fetched BEFORE the FMA loop so that their latency hides behind it
        float acc[4][P];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int i = 0; i < P; ++i) acc[j][i] = 0.f;
        if (!UP2 && ok && (add || accf)) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float* d = dst + (size_t)j * a.L;
            const float* q = add ? add + (size_t)j * a.L : nullptr;
            if constexpr (BULK && P == 4) {
              if (q) { const float4 v = __ldg(reinterpret_cast<const float4*>(q)); acc[j][0] += v.x; acc[j][1] += v.y; acc[j][2] += v.z; acc[j][P - 1] += v.w; }
              if (accf) { const float4 v = *reinterpret_cast<const float4*>(d); acc[j][0] += v.x; acc[j][1] += v.y; acc[j][2] += v.z; acc[j][P - 1] += v.w; }
            } else if constexpr (BULK && P == 2) {
              if (q) { const float2 v = __ldg(reinterpret_cast<const float2*>(q)); acc[j][0] += v.x; acc[j][P - 1] += v.y; }
              if (accf) { const float2 v = *reinterpret_cast<const float2*>(d); acc[j][0] += v.x; acc[j][P - 1] += v.y; }
            } else {
#pragma unroll
              for (int i = 0; i < P; ++i)
                if (l + i < a.L) {
                  if (q) acc[j][i] += __ldg(q + i);
                  if (accf) acc[j][i] += d[i];
                }
            }
          }
        }
        if constexpr (DOWN2) {
#pragma unroll 4
          for (int co = 0; co < COUT; ++co) {
            float dh[P / 2 + 2];   // dy[co][j0 - 1 .. j0 + P / 2], j0 = (this thread's first position) / 2
            const float* hb = du_s + co * TS + 4 + ((P * tid) >> 1);
#pragma unroll
            for (int e = 0; e < P / 2 + 2; ++e) dh[e] = hb[e - 1];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 w4 = *reinterpret_cast<const float4*>(w_s + (co * cin + cb + j) * 4);
#pragma unroll
              for (int pp = 0; pp < P / 2; ++pp) {
                acc[j][2 * pp] = fmaf(dh[pp + 1], w4.y, fmaf(dh[pp], w4.w, acc[j][2 * pp]));
                acc[j][2 * pp + 1] = fmaf(dh[pp + 2], w4.x, fmaf(dh[pp + 1], w4.z, acc[j][2 * pp + 1]));
              }
            }
          }
        } else
#pragma unroll 4
        for (int co = 0; co < COUT; ++co) {
          float dwin[P + 2];   // du[co][pos - 1 .. pos + P]
          const float* dr = du_s + co * TS + 4 + P * tid;
          if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(dr); dwin[1] = m.x; dwin[2] = m.y; dwin[3] = m.z; dwin[P] = m.w; }
          else if constexpr (P == 2) { const float2 m = *reinterpret_cast<const float2*>(dr); dwin[1] = m.x; dwin[P] = m.y; }
          else dwin[1] = dr[0];
          if constexpr (K == 3) { dwin[0] = dr[-1]; dwin[P + 1] = dr[P]; }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 w4 = *reinterpret_cast<const float4*>(w_s + (co * cin + cb + j) * 4);
            const float wk[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int i = 0; i < P; ++i)
#pragma unroll
              for (int k = 0; k < K; ++k) acc[j][i] = fmaf(dwin[i + 1 + H - k], wk[k], acc[j][i]);
          }
        }
        if constexpr (RES) {   // + wres^T dyo (1x1: no halo)
#pragma unroll 4
          for (int co = 0; co < COUT; ++co) {
            float yo[P];
            const float* yr = yo_t + co * TS + 4 + P * tid;
            if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(yr); yo[0] = m.x; yo[1] = m.y; yo[2] = m.z; yo[P - 1] = m.w; }
            else if constexpr (P == 2) { const float2 m = *reinterpret_cast<const float2*>(yr); yo[0] = m.x; yo[P - 1] = m.y; }
            else yo[0] = yr[0];
            const float4 w4 = *reinterpret_cast<const float4*>(wres_s + co * cin + cb);
            const float wj[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int i = 0; i < P; ++i) acc[j][i] = fmaf(yo[i], wj[j], acc[j][i]);
          }
        }
        if constexpr (UP2) {   // d x[m] = d x_up[2m] + d x_up[2m + 1]: both halves of a pair live in this thread
          if (ok) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float* d = dst + (size_t)j * (a.L >> 1);
              float f[P / 2];
#pragma unroll
              for (int m = 0; m < P / 2; ++m) f[m] = acc[j][2 * m] + acc[j][2 * m + 1];
              if constexpr (BULK && P == 4) {
                if (accf) { const float2 v = *reinterpret_cast<const float2*>(d); f[0] += v.x; f[P / 2 - 1] += v.y; }
                *reinterpret_cast<float2*>(d) = make_float2(f[0], f[P / 2 - 1]);
              } else {
#pragma unroll
                for (int m = 0; m < P / 2; ++m)
                  if (l + 2 * m < a.L) d[m] = accf ? d[m] + f[m] : f[m];
              }
            }
          }
        } else
        if (ok) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float* d = dst + (size_t)j * a.L;
            if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(d) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][P - 1]);
            else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(d) = make_float2(acc[j][0], acc[j][P - 1]);
            else {
#pragma unroll
              for (int i = 0; i < P; ++i) if (l + i < a.L) d[i] = acc[j][i];
            }
          }
        }
      }
    }

    // ---------------------------------------------------------------- phase 3: dW[:, ci3, :] over this thread's segment
    if constexpr (MMA) {
      // dW_k[ci][co] += sum_pos x[ci][pos] du[co][pos + H - k]: A = x (rows ci, k-slots = 8 positions), B_k = shifted du
      for (int chn = warp_; chn < TL / 8; chn += NW) {
        const int p0 = 8 * chn;
        uint32_t ax[MCI][4];
#pragma unroll
        for (int mt = 0; mt < MCI; ++mt) {
          // rows >= cin of the m16 tile do not exist (their dW rows are dropped): re-read the last real row instead
          const float* xp = x_t + min(16 * mt + fg, cin - 1) * TS + 4 + p0 + ft;
          const float* xq = x_t + min(16 * mt + fg + 8, cin - 1) * TS + 4 + p0 + ft;
          ax[mt][0] = cf_rtf(xp[0]); ax[mt][1] = cf_rtf(xq[0]); ax[mt][2] = cf_rtf(xp[4]); ax[mt][3] = cf_rtf(xq[4]);
        }
#pragma unroll
        for (int nt = 0; nt < KCO; ++nt) {
          const float* bp = du_s + min(8 * nt + fg, COUT - 1) * TS + 4 + p0 + ft + H;
#pragma unroll
          for (int kk = 0; kk < K; ++kk) {
            const uint32_t b0 = __float_as_uint(bp[-kk]), b1 = __float_as_uint(bp[4 - kk]);
#pragma unroll
            for (int mt = 0; mt < MCI; ++mt) cf_mma8(dWf[kk][mt][nt], ax[mt][0], ax[mt][1], ax[mt][2], ax[mt][3], b0, b1);
          }
          if constexpr (RES) {
            const float* yp = yo_t + min(8 * nt + fg, COUT - 1) * TS + 4 + p0 + ft;
            const uint32_t b0 = cf_rtf(yp[0]), b1 = cf_rtf(yp[4]);
#pragma unroll
            for (int mt = 0; mt < MCI; ++mt) cf_mma8(dRf[mt][nt], ax[mt][0], ax[mt][1], ax[mt][2], ax[mt][3], b0, b1);
          }
        }
      }
    } else
    if (p3_active) {
      const float* xr = x_t + ci3 * TS + 4;
      for (int q = q_begin; q < q_end; q += 4) {
        float4 xm;
        float x6[6];
        if constexpr (UP2) {   // x_up[q - 1 .. q + 4] = x[q/2 - 1], x[q/2] (x2), x[q/2 + 1] (x2), x[q/2 + 2]
          const float* hr = xr + (q >> 1);
          const float h0 = hr[0], h1 = hr[1];
          x6[0] = hr[-1]; x6[1] = h0; x6[2] = h0; x6[3] = h1; x6[4] = h1; x6[5] = hr[2];
          xm = make_float4(h0, h0, h1, h1);
        } else {
          xm = *reinterpret_cast<const float4*>(xr + q);
          x6[0] = 0.f; x6[1] = xm.x; x6[2] = xm.y; x6[3] = xm.z; x6[4] = xm.w; x6[5] = 0.f;
          if constexpr (K >= 3) { x6[0] = xr[q - 1]; x6[5] = xr[q + 4]; }
        }
        if constexpr (DOWN2) {   // output positions m0 = q / 2, m0 + 1 read x[2m + k - 1] = x6[k], x6[k + 2]
#pragma unroll
          for (int co = 0; co < COUT; ++co) {
            const float d0 = du_s[co * TS + 4 + (q >> 1)], d1 = du_s[co * TS + 5 + (q >> 1)];
#pragma unroll
            for (int k = 0; k < K; ++k) dwacc[co][k] = fmaf(d0, x6[k], fmaf(d1, x6[k + 2], dwacc[co][k]));
          }
        } else
#pragma unroll
        for (int co = 0; co < COUT; ++co) {
          const float4 d4 = *reinterpret_cast<const float4*>(du_s + co * TS + 4 + q);
          const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
          for (int k = 0; k < K; ++k)
#pragma unroll
            for (int i = 0; i < 4; ++i) dwacc[co][k] = fmaf(dd[i], x6[i + k + 1 - H], dwacc[co][k]);
        }
        if constexpr (RES) {
#pragma unroll
          for (int co = 0; co < COUT; ++co) {
            const float4 y4 = *reinterpret_cast<const float4*>(yo_t + co * TS + 4 + q);
            dwres[co] = fmaf(y4.x, xm.x, fmaf(y4.y, xm.y, fmaf(y4.z, xm.z, fmaf(y4.w, xm.w, dwres[co]))));
          }
        }
      }
    }
    __syncthreads();   // everyone is done with stage s
    if (it + 1 < n_tiles) issue_add(tile + 1);
    if (it + 2 < n_tiles) issue(tile + 2, s);
  }

  // ------------------------------------------------------------------ leave: parameter gradients
  if (EPI && cur_sample >= 0) flush_sample(cur_sample);
  if constexpr (MMA) {   // thread holds dW_k[ci = 16mt + fg (+8)][co = 8nt + 2ft (+1)]
#pragma unroll
    for (int mt = 0; mt < MCI; ++mt)
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int ci = 16 * mt + fg + 8 * (i >> 1), co = 8 * nt + 2 * ft + (i & 1);
          if (ci < cin && co < COUT) {
#pragma unroll
            for (int kk = 0; kk < K; ++kk) atomicAdd(dw_s + (co * cin + ci) * K + kk, dWf[kk][mt][nt][i]);
            if constexpr (RES) atomicAdd(dwres_s + co * cin + ci, dRf[mt][nt][i]);
          }
        }
  } else
  if (p3_active) {
#pragma unroll
    for (int co = 0; co < COUT; ++co)
#pragma unroll
      for (int k = 0; k < K; ++k) atomicAdd(dw_s + (co * cin + ci3) * K + k, dwacc[co][k]);
  }
  {
    float v[2 * COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) { v[c] = accG[c] * sqrtC; v[COUT + c] = accB[c]; }
    const float tot = block_sum2c(v);   // its barriers also publish dw_s
    if (tid < COUT) { if (EPI && a.dg) atomicAdd(a.dg + tid, tot); }
    else if (tid < 2 * COUT) { if (a.db) atomicAdd(a.db + tid - COUT, tot); }
  }
  for (int i = tid; i < COUT * cin * K; i += NT) atomicAdd(a.dw + i, dw_s[i]);
  if constexpr (RES) {
    if (!MMA && p3_active) {
#pragma unroll
      for (int co = 0; co < COUT; ++co) atomicAdd(dwres_s + co * cin + ci3, dwres[co]);
    }
    float v[2 * COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) { v[c] = accR[c]; v[COUT + c] = 0.f; }
    const float tot = block_sum2c(v);   // its barriers also publish dwres_s
    if (tid < COUT && a.dbres) atomicAdd(a.dbres + tid, tot);
    for (int i = tid; i < COUT * cin; i += NT) atomicAdd(a.dwres + i, dwres_s[i]);
  }
}

template <int COUT, int K, int P, int NT, bool EPI, bool BULK, bool RES = false, int NCI = 0, bool UP2 = false,
          bool DOWN2 = false>
static int launch_fused_tma(ConvBwdFusedArgs a, cudaStream_t st) {
  constexpr int TL = NT * P, TS = TL + 36, NW = NT / 32;
  const int cin = a.c1 + a.c2;
  const int rows = (EPI ? 2 * COUT : COUT) + cin + (RES ? COUT : 0);
  a.tiles_per_row = (a.L + TL - 1) / TL;
  a.total_tiles = a.tiles_per_row * a.R;
  a.al8 = ((((size_t)a.dy | (size_t)a.u | (size_t)a.x1 | (size_t)a.x2 | (size_t)a.dyo) & 7) == 0) ? 1 : 0;
  size_t smem = sizeof(float) * ((size_t)2 * rows * TS + (NCI > 0 ? 0 : (size_t)COUT * cin * 4) + (size_t)COUT * cin * K +
                                 (RES ? (size_t)2 * COUT * cin : 0) + NW * 2 * COUT) + 16;
  if (NCI > 0 && !RES && a.dx1)   // staged copies of dadd / the old dx1 tile (see the kernel)
    smem += sizeof(float) * (size_t)a.c1 * TS * ((a.dadd ? 1 : 0) + (a.acc1 ? 1 : 0));
  if (smem > 220 * 1024) return -6;
  auto kern = conv_bwd_fused_tma_kernel<COUT, K, P, NT, EPI, BULK, RES, NCI, UP2, DOWN2>;
  static int sm_count = 0;
  if (!sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem);
  if (occ < 1) return -6;
  int grid = min(a.total_tiles, sm_count * occ);
  a.tiles_per_cta = (a.total_tiles + grid - 1) / grid;
  grid = (a.total_tiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
  kern<<<(unsigned)grid, NT, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}
template <int COUT, int K, int P, int NT, bool BULK>
static int launch_fused_tma_epi(const ConvBwdFusedArgs& a, cudaStream_t st) {
  return a.u ? launch_fused_tma<COUT, K, P, NT, true, BULK>(a, st) : launch_fused_tma<COUT, K, P, NT, false, BULK>(a, st);
}

template <int COUT, int K, int P, int VEC>
static int launch_fused(ConvBwdFusedArgs a, cudaStream_t st) {
  constexpr int TL = 128 * P, DS = TL + 4;
  const int cin = a.c1 + a.c2;
  a.tiles_per_row = (a.L + TL - 1) / TL;
  a.total_tiles = a.tiles_per_row * a.R;
  size_t smem = sizeof(float) * ((size_t)COUT * DS + 8 + (size_t)cin * DS + 8 + (size_t)COUT * cin * 4 + (size_t)COUT * cin * K + 4 * 4 * COUT);
  auto kern = conv_bwd_fused_kernel<COUT, K, P, VEC>;
  static int sm_count = 0;
  if (!sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 128, smem);
  if (occ < 1) return -6;
  int grid = min(a.total_tiles, sm_count * occ);
  a.tiles_per_cta = (a.total_tiles + grid - 1) / grid;
  grid = (a.total_tiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
  kern<<<(unsigned)grid, 128, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

template <int K>
static int dispatch_fused(const ConvBwdFusedArgs& a, int cout, cudaStream_t st) {
  const bool v4 = (a.L % 4 == 0);
  // 16-byte aligned rows of the staged inputs: bulk-async-copy pipeline
  const bool al = v4 && ((((size_t)a.dy | (size_t)a.x1 | (size_t)a.u | (size_t)a.x2) & 15) == 0);
  // the FFMA variants (bulk pipeline with NCI == 0, and conv_bwd_fused_kernel with VEC = 4) also read dadd / the old dx
  // and store dx with float4 / float2 accesses; the tensor-core variants store dx scalar and check each dadd / old-dx row
  // before their 16-byte copies, so only `al` applies to them (a null pointer is 0: it never vetoes)
  const bool alv = al && ((((size_t)a.dadd | (size_t)a.dx1 | (size_t)a.dx2) & 15) == 0);
  // the pipelined kernel covers: plain conv, or RMSNorm (+ scale/shift) + SiLU epilogue; channel counts in fours
  const bool epi_ok = !a.u || (a.g && a.act == 1);
  const int cin = a.c1 + a.c2;
  const bool ch4 = (a.c1 & 3) == 0 && (a.c2 & 3) == 0;
  if constexpr (K == 3) {
    // conv3 + RMSNorm / SiLU epilogue at 8 .. 16 channels: tensor-core contractions (NCI = n8 tiles over cin)
    if (!a.dyo && a.L >= 128 && a.u && a.g && a.act == 1 && ch4 && cin <= 32) {
      const int nci = (cin + 7) / 8;
      if (al) {
        if (cout == 8 && nci == 1) return launch_fused_tma<8, 3, 2, 128, true, true, false, 1>(a, st);
        if (cout == 8 && nci == 2) return launch_fused_tma<8, 3, 2, 128, true, true, false, 2>(a, st);
        if (cout == 12 && nci == 2) return launch_fused_tma<12, 3, 2, 128, true, true, false, 2>(a, st);
        if (cout == 16 && nci == 2) return launch_fused_tma<16, 3, 1, 128, true, true, false, 2>(a, st);
      } else {
        if (cout == 12 && nci == 2) return launch_fused_tma<12, 3, 1, 128, true, false, false, 2>(a, st);
        if (cout == 16 && nci == 2) return launch_fused_tma<16, 3, 1, 128, true, false, false, 2>(a, st);
      }
    }
  }
  if (a.dyo) {   // conv3 + epilogue with the 1x1 res_conv over the same input: pipelined kernel only
    if constexpr (K == 3) {
      const bool al2 = al && (((size_t)a.dyo & 15) == 0);
      if (a.L >= 128 && a.u && a.g && a.act == 1 && ch4 && !a.dadd) {
        const int nci = (cin + 7) / 8;
        if (al2) {
          if (cout == 4 && alv) return launch_fused_tma<4, 3, 4, 128, true, true, true>(a, st);
          if (cout == 8) {
            if (nci == 1) return launch_fused_tma<8, 3, 2, 128, true, true, true, 1>(a, st);
            if (nci == 2) return launch_fused_tma<8, 3, 2, 128, true, true, true, 2>(a, st);
            if (alv) return launch_fused_tma<8, 3, 2, 128, true, true, true>(a, st);
          }
          if (cout == 12 && nci == 3) return launch_fused_tma<12, 3, 1, 128, true, true, true, 3>(a, st);
          if (cout == 16 && nci == 4) return launch_fused_tma<16, 3, 1, 128, true, true, true, 4>(a, st);
        } else {
          if (cout == 12 && nci == 3) return launch_fused_tma<12, 3, 1, 128, true, false, true, 3>(a, st);
          if (cout == 16 && nci == 4) return launch_fused_tma<16, 3, 1, 128, true, false, true, 4>(a, st);
        }
      }
    }
    return 1;    // not covered: the caller runs the two convolutions separately
  }
  if (a.L >= 128 && epi_ok && ch4) {
    if (alv) {
      switch (cout) {
        case 4: return launch_fused_tma_epi<4, K, 4, 128, true>(a, st);
        case 8: return launch_fused_tma_epi<8, K, 2, 128, true>(a, st);
        case 12: return launch_fused_tma_epi<12, K, 2, 128, true>(a, st);
        case 16: return launch_fused_tma_epi<16, K, 1, 128, true>(a, st);
        default: break;
      }
    } else {
      switch (cout) {
        case 4: return launch_fused_tma_epi<4, K, 4, 128, false>(a, st);
        case 8: return launch_fused_tma_epi<8, K, 2, 128, false>(a, st);
        case 12: return launch_fused_tma_epi<12, K, 1, 128, false>(a, st);
        case 16: return launch_fused_tma_epi<16, K, 1, 128, false>(a, st);
        default: break;
      }
    }
  }
  // VEC = 4 reads dy / u / x1 / x2 / dadd / the old dx and stores dx as float4: every one of them must be 16-byte aligned
  switch (cout) {
    case 1: return alv ? launch_fused<1, K, 4, 4>(a, st) : launch_fused<1, K, 4, 1>(a, st);
    case 4: return alv ? launch_fused<4, K, 4, 4>(a, st) : launch_fused<4, K, 4, 1>(a, st);
    case 8: return alv ? launch_fused<8, K, 4, 4>(a, st) : launch_fused<8, K, 4, 1>(a, st);
    case 12: return launch_fused<12, K, 2, 1>(a, st);
    case 16: return launch_fused<16, K, 2, 1>(a, st);
    case 24: return launch_fused<24, K, 1, 1>(a, st);
    case 32: return launch_fused<32, K, 1, 1>(a, st);
    default: return -3;
  }
}

// =====================================================================================================================
// Pipelined forward of a stride-1 Conv1d (K = 1 or 3) with the fused Block epilogue (bias, RMSNorm over channels,
// per-sample scale/shift, SiLU/GELU, residual add): Block.forward unet1d.py:248-268, ResnetBlock 302-323.
// The input rows (both concat sources, and the residual rows) of a tile arrive by bulk async copies, two tiles deep;
// a thread owns P consecutive positions and all COUT output channels (needed for the channel RMSNorm), reads its
// taps with one 128/64-bit shared load + 2 neighbours per input channel and the weights as broadcast float4.
struct ConvFwdTmaArgs {
  const float* x1; const float* x2; const float* w; const float* bias; const float* g; const float* ss;
  const float* res; float* u; float* y;
  int c1, c2, R, L, rows_per_sample, ss_stride, act, tiles_per_row, total_tiles, tiles_per_cta;
  // K = 7 (init_conv over cat(ConditionalScaleShift(cond), x), unet1d.py:1107-1117): source-1 channel c is
  // x * (in_ss[c] + 1) + in_ss[c1 + c] per sample at existing positions (the zero padding stays zero)
  const float* in_ss = nullptr;
  int in_ss_stride = 0;
};
// UP2: the input is the nearest-x2 upsampling of half-length rows (Upsample, unet1d.py:93-96): the half-rate rows are staged
// and x_up[q] = x_half[q >> 1] is resolved when the taps are read, so the upsampled tensor never exists.

// DN2: Downsample = Conv1d(k4, stride 2, pad 1) (unet1d.py:110): a.L is the OUTPUT length, the input rows are 2 a.L long;
// a thread owns P output positions m and reads x[2m - 1 .. 2m + 2] per tap window from the staged full-rate rows
// (row stride 2 TL + 8), single source, no residual.
template <int COUT, int K, int P, int NT, bool BULK, bool UP2, bool DN2 = false>
__global__ void __launch_bounds__(NT) conv_fwd_tma_kernel(ConvFwdTmaArgs a) {
  constexpr int TL = NT * P;
  constexpr int TS = DN2 ? 2 * TL + 8 : TL + 36;
  constexpr int H = (K - 1) / 2;
  static_assert(P == 1 || P == 2 || P == 4, "P");
  static_assert(COUT % 4 == 0, "COUT");
  static_assert(!DN2 || (K == 4 && !UP2), "DN2: k4 s2");
  static_assert(K != 7 || (!UP2 && !DN2), "k7: plain stride-1 mode");
  extern __shared__ float4 dyn_smem4[];
  const int cin = a.c1 + a.c2;
  const bool has_res = a.res != nullptr;
  const int rows = cin + (has_res ? COUT : 0);
  float* stage0 = reinterpret_cast<float*>(dyn_smem4);
  const int stage_floats = rows * TS;
  float* w_s = stage0 + 2 * stage_floats;                 // [(ci*K + k) * COUT + co]
  uint64_t* bars = reinterpret_cast<uint64_t*>(w_s + cin * K * COUT);
  const int tid = threadIdx.x;
  const uint32_t bar0 = cf_smem_u32(bars), bar1 = bar0 + 8;
  if (tid == 0) {
    cf_mbar_init(bar0, BULK ? 1 : NT);
    cf_mbar_init(bar1, BULK ? 1 : NT);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < cin * K * COUT; i += NT) {
    const int co = i % COUT, ck = i / COUT;
    w_s[i] = a.w[(size_t)co * cin * K + ck];
  }
  __syncthreads();
  const int t_begin = blockIdx.x * a.tiles_per_cta, t_end = min(a.total_tiles, t_begin + a.tiles_per_cta);
  const int n_tiles = t_end - t_begin;

  auto issue = [&](int tile, int s) {
    if (!BULK) {   // any alignment: 4-byte cp.async from every thread, arriving on the same mbarrier
      const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
      const int Lx = UP2 ? a.L / 2 : DN2 ? 2 * a.L : a.L, x0 = UP2 ? tl0 / 2 : DN2 ? 2 * tl0 : tl0,
                xw_ = UP2 ? TL / 2 : DN2 ? 2 * TL : TL;   // staged input window
      const int l_lo = max(0, x0 - 4), l_hi = min(Lx, x0 + xw_ + 4);
      const int w = l_hi - l_lo, doff = l_lo - (x0 - 4);
      float* st = stage0 + s * stage_floats;
      for (int row = tid >> 5; row < rows; row += NT / 32) {   // one warp per row: the row pointer is computed once per warp
        const float* src;
        if (row < a.c1) src = a.x1 + ((size_t)r * a.c1 + row) * Lx;
        else if (row < cin) src = a.x2 + ((size_t)r * a.c2 + (row - a.c1)) * Lx;
        else src = a.res + ((size_t)r * COUT + (row - cin)) * a.L;
        src += l_lo;
        const uint32_t dst = cf_smem_u32(st + row * TS + doff);
        for (int e = tid & 31; e < w; e += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
      }
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(s ? bar1 : bar0) : "memory");
      return;
    }
    if (tid < 32) {
      const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
      const int Lx = UP2 ? a.L / 2 : DN2 ? 2 * a.L : a.L, x0 = UP2 ? tl0 / 2 : DN2 ? 2 * tl0 : tl0,
                xw_ = UP2 ? TL / 2 : DN2 ? 2 * TL : TL;
      const int l_lo = max(0, x0 - 4), l_hi = min(Lx, x0 + xw_ + 4);
      const uint32_t bytes = (uint32_t)(l_hi - l_lo) * 4u;
      const uint32_t bar = s ? bar1 : bar0;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (tid == 0) cf_mbar_expect_tx(bar, bytes * (uint32_t)rows);
      __syncwarp();
      float* st = stage0 + s * stage_floats;
      for (int row = tid; row < rows; row += 32) {
        const float* src;
        if (row < a.c1) src = a.x1 + ((size_t)r * a.c1 + row) * Lx;
        else if (row < cin) src = a.x2 + ((size_t)r * a.c2 + (row - a.c1)) * Lx;
        else src = a.res + ((size_t)r * COUT + (row - cin)) * a.L;
        cf_bulk_g2s(cf_smem_u32(st + row * TS + (l_lo - (x0 - 4))), src + l_lo, bytes, bar);
      }
    }
  };
  if (n_tiles > 0) issue(t_begin, 0);
  if (n_tiles > 1) issue(t_begin + 1, 1);

  const float sqrtC = sqrtf((float)COUT);
  const bool has_g = a.g != nullptr, has_ss = a.ss != nullptr;
  float bias[COUT];
#pragma unroll
  for (int c = 0; c < COUT; ++c) bias[c] = a.bias ? a.bias[c] : 0.f;

  for (int it = 0; it < n_tiles; ++it) {
    const int tile = t_begin + it, s = it & 1;
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int sample = r / a.rows_per_sample;
    float* x_t = stage0 + s * stage_floats;
    cf_mbar_wait(s ? bar1 : bar0, (uint32_t)((it >> 1) & 1));
    if (H > 0) {   // zero padding at the two row ends (positions -1 .. -H and L .. L + H - 1)
      if (tid < cin) {
#pragma unroll
        for (int h = 0; h < (K == 7 ? 3 : 1); ++h) {
          if (tl0 == 0) x_t[tid * TS + 3 - h] = 0.f;
          if (a.L <= tl0 + TL) x_t[tid * TS + (UP2 ? (a.L - tl0) / 2 : DN2 ? 2 * (a.L - tl0) : a.L - tl0) + 4 + h] = 0.f;
        }
      }
      if constexpr (K == 7) {
        if (a.in_ss) {   // ConditionalScaleShift on source 1, in place, existing positions of the window only
          for (int ci = 0; ci < a.c1; ++ci) {
            const float sc = a.in_ss[(size_t)sample * a.in_ss_stride + ci] + 1.f;
            const float sh = a.in_ss[(size_t)sample * a.in_ss_stride + a.c1 + ci];
            for (int j = tid; j < TL + 8; j += NT) {
              const int l = tl0 - 4 + j;
              if (l >= 0 && l < a.L) x_t[ci * TS + j] = fmaf(x_t[ci * TS + j], sc, sh);
            }
          }
        }
        __syncthreads();
      } else
      if (tl0 == 0 || a.L <= tl0 + TL) __syncthreads();   // uniform per tile
    }
    const int l = tl0 + P * tid;
    const bool ok = l < a.L;
    float acc[P][COUT];
#pragma unroll
    for (int i = 0; i < P; ++i)
#pragma unroll
      for (int c = 0; c < COUT; ++c) acc[i][c] = bias[c];
#pragma unroll 2
    for (int ci = 0; ci < cin; ++ci) {
      float xw[DN2 ? 2 * P + 2 : K == 7 ? P + 6 : P + 2];
      if constexpr (K == 7) {   // xw[e] = x[l - 3 + e]
        const float* xb = x_t + ci * TS + 4 + P * tid;
#pragma unroll
        for (int e = 0; e < 3; ++e) { xw[e] = xb[e - 3]; xw[P + 3 + e] = xb[P + e]; }
        if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(xb); xw[3] = m.x; xw[4] = m.y; xw[5] = m.z; xw[6] = m.w; }
        else {
#pragma unroll
          for (int e = 0; e < P; ++e) xw[3 + e] = xb[e];
        }
      }
      if constexpr (DN2) {   // xw[e] = x[2 m0 - 1 + e], m0 = this thread's first output position
        const float* xb = x_t + ci * TS + 4 + 2 * P * tid;
        xw[0] = xb[-1];
        if constexpr (P >= 2) {
#pragma unroll
          for (int v = 0; v < P / 2; ++v) {
            const float4 m = *reinterpret_cast<const float4*>(xb + 4 * v);
            xw[4 * v + 1] = m.x; xw[4 * v + 2] = m.y; xw[4 * v + 3] = m.z; xw[4 * v + 4] = m.w;
          }
        } else {
          const float2 m = *reinterpret_cast<const float2*>(xb);
          xw[1] = m.x; xw[2] = m.y;
        }
        xw[2 * P + 1] = xb[2 * P];
      }
      if constexpr (UP2) {
        // x_up[tl0 + P tid + i - 1] = x_half[(P tid + i - 1) >> 1]  (index -1 >> 1 = -1: the zeroed left neighbour)
        const float* xh = x_t + ci * TS + 4;
        if constexpr (P == 4) {
          const float2 m = *reinterpret_cast<const float2*>(xh + 2 * tid);
          xw[0] = xh[2 * tid - 1]; xw[1] = m.x; xw[2] = m.x; xw[3] = m.y; xw[P] = m.y; xw[P + 1] = xh[2 * tid + 2];
        } else {
#pragma unroll
          for (int i = 0; i < P + 2; ++i) xw[i] = xh[(P * (int)tid + i - 1) >> 1];
        }
      }
      const float* xr = x_t + ci * TS + 4 + P * tid;
      if constexpr (UP2 || DN2 || K == 7) {
      } else if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(xr); xw[1] = m.x; xw[2] = m.y; xw[3] = m.z; xw[P] = m.w; }
      else if constexpr (P == 2) { const float2 m = *reinterpret_cast<const float2*>(xr); xw[1] = m.x; xw[P] = m.y; }
      else xw[1] = xr[0];
      if constexpr (K == 3 && !UP2) { xw[0] = xr[-1]; xw[P + 1] = xr[P]; }
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float4* wp = reinterpret_cast<const float4*>(w_s + (ci * K + k) * COUT);
#pragma unroll
        for (int c4 = 0; c4 < COUT / 4; ++c4) {
          const float4 w4 = wp[c4];
#pragma unroll
          for (int i = 0; i < P; ++i) {
            const float xv = DN2 ? xw[2 * i + k] : K == 7 ? xw[i + k] : xw[i + 1 + k - H];
            cf_fma2(acc[i][4 * c4 + 0], acc[i][4 * c4 + 1], xv, w4.x, w4.y);
            cf_fma2(acc[i][4 * c4 + 2], acc[i][4 * c4 + 3], xv, w4.z, w4.w);
          }
        }
      }
    }
    if (ok) {
      const size_t base = (size_t)r * COUT * a.L + l;
      if (a.u) {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(a.u + base + (size_t)c * a.L) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
          else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(a.u + base + (size_t)c * a.L) = make_float2(acc[0][c], acc[P - 1][c]);
          else {
#pragma unroll
            for (int i = 0; i < P; ++i) if (l + i < a.L) a.u[base + (size_t)c * a.L + i] = acc[i][c];
          }
        }
      }
      float gs[COUT], sh[COUT];
#pragma unroll
      for (int c = 0; c < COUT; ++c) {
        const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + c] + 1.f : 1.f;
        gs[c] = (has_g ? a.g[c] * sqrtC : 1.f) * sc1;
        sh[c] = has_ss ? a.ss[(size_t)sample * a.ss_stride + COUT + c] : 0.f;
      }
#pragma unroll
      for (int i = 0; i < P; ++i) {
        float inv = 1.f;
        if (has_g) {
          float s2 = 0.f;
#pragma unroll
          for (int c = 0; c < COUT; ++c) s2 = fmaf(acc[i][c], acc[i][c], s2);
          inv = s2 > 1e-24f ? cf_rsqrt(s2) : 1e12f;
        }
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          float z = fmaf(acc[i][c] * inv, gs[c], sh[c]);
          if (a.act == 1) z = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
          else if (a.act == 2) z = act_fwd(z, 2);
          if (has_res) z += x_t[(cin + c) * TS + 4 + P * tid + i];
          acc[i][c] = z;
        }
      }
#pragma unroll
      for (int c = 0; c < COUT; ++c) {
        if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(a.y + base + (size_t)c * a.L) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
        else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(a.y + base + (size_t)c * a.L) = make_float2(acc[0][c], acc[P - 1][c]);
        else {
#pragma unroll
          for (int i = 0; i < P; ++i) if (l + i < a.L) a.y[base + (size_t)c * a.L + i] = acc[i][c];
        }
      }
    }
    __syncthreads();   // everyone is done with stage s
    if (it + 2 < n_tiles) issue(tile + 2, s);
  }
}

template <int COUT, int K, int P, int NT, bool BULK, bool UP2, bool DN2 = false>
static int launch_fwd_tma(ConvFwdTmaArgs a, cudaStream_t st) {
  constexpr int TL = NT * P, TS = DN2 ? 2 * TL + 8 : TL + 36;
  const int cin = a.c1 + a.c2;
  const int rows = cin + (a.res ? COUT : 0);
  a.tiles_per_row = (a.L + TL - 1) / TL;
  a.total_tiles = a.tiles_per_row * a.R;
  size_t smem = sizeof(float) * ((size_t)2 * rows * TS + (size_t)cin * K * COUT) + 16;
  if (smem > 220 * 1024) return -6;
  auto kern = conv_fwd_tma_kernel<COUT, K, P, NT, BULK, UP2, DN2>;
  static int sm_count = 0;
  if (!sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem);
  if (occ < 1) return -6;
  int grid = min(a.total_tiles, sm_count * occ);
  a.tiles_per_cta = (a.total_tiles + grid - 1) / grid;
  grid = (a.total_tiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
  kern<<<(unsigned)grid, NT, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

// Returns 1 if the pipelined kernel took the call, 0 if the shape is not eligible, < 0 on error.  up == 2: x1 has
// L / 2 columns (nearest-x2 upsampling folded into the tap reads), K == 3, single source, no residual.
int conv_fwd_tma_try(const float* x1, int c1, const float* x2, int c2, const float* w, const float* bias, int cout, int K,
                     const float* g, const float* ss, int ss_stride, int act, const float* res, float* u, float* y, int R,
                     int L, int rows_per_sample, int up, cudaStream_t st, const float* in_ss, int in_ss_stride) {
  if (L < 128 || c1 + c2 > 64) return 0;
  if (up == -2) { if (K != 4 || x2 || res) return 0; }   // Downsample: k4, stride 2, pad 1; L = output length
  else if (K == 7) { if (up != 1 || res || (cout != 4 && cout != 8)) return 0; }
  else if (K != 1 && K != 3) return 0;
  if (in_ss && K != 7) return 0;
  if (up == 2 && (K != 3 || x2 || res || (L & 1))) return 0;
  const int Lx = up == 2 ? L / 2 : up == -2 ? 2 * L : L;
  const bool al = (L % 4 == 0) && (Lx % 4 == 0) && ((((size_t)x1 | (size_t)x2 | (size_t)res | (size_t)u | (size_t)y) & 15) == 0);
  ConvFwdTmaArgs a{x1, x2, w, bias, g, ss, res, u, y, c1, c2, R, L, rows_per_sample, ss_stride, act, 0, 0, 0};
  a.in_ss = in_ss; a.in_ss_stride = in_ss_stride;
  int rc;
#define DQ_FWD_CASE(CO, KK, PA, PU) \
  case CO: rc = al ? launch_fwd_tma<CO, KK, PA, 128, true, false>(a, st) : launch_fwd_tma<CO, KK, PU, 128, false, false>(a, st); break;
#define DQ_FWD_CASE_UP(CO, PA, PU) \
  case CO: rc = al ? launch_fwd_tma<CO, 3, PA, 128, true, true>(a, st) : launch_fwd_tma<CO, 3, PU, 128, false, true>(a, st); break;
#define DQ_FWD_CASE_DN(CO, PA) \
  case CO: rc = al ? launch_fwd_tma<CO, 4, PA, 128, true, false, true>(a, st) : launch_fwd_tma<CO, 4, PA, 128, false, false, true>(a, st); break;
  if (K == 7) {
    switch (cout) {
      DQ_FWD_CASE(4, 7, 4, 4)
      DQ_FWD_CASE(8, 7, 4, 2)
      default: return 0;
    }
  } else if (up == -2) {
    switch (cout) {
      DQ_FWD_CASE_DN(4, 4)
      DQ_FWD_CASE_DN(8, 2)
      DQ_FWD_CASE_DN(12, 2)
      DQ_FWD_CASE_DN(16, 2)
      default: return 0;
    }
  } else if (up == 2) {
    switch (cout) {
      DQ_FWD_CASE_UP(4, 4, 4)
      DQ_FWD_CASE_UP(8, 4, 2)
      DQ_FWD_CASE_UP(12, 2, 2)
      DQ_FWD_CASE_UP(16, 2, 2)
      default: return 0;
    }
  } else if (K == 3) {
    switch (cout) {
      DQ_FWD_CASE(4, 3, 4, 4)
      DQ_FWD_CASE(8, 3, 4, 2)
      DQ_FWD_CASE(12, 3, 2, 1)
      DQ_FWD_CASE(16, 3, 2, 1)
      default: return 0;
    }
  } else {
    switch (cout) {
      DQ_FWD_CASE(4, 1, 4, 4)
      DQ_FWD_CASE(8, 1, 4, 2)
      DQ_FWD_CASE(12, 1, 2, 1)
      DQ_FWD_CASE(16, 1, 2, 1)
      default: return 0;
    }
  }
#undef DQ_FWD_CASE
#undef DQ_FWD_CASE_UP
#undef DQ_FWD_CASE_DN
  return rc == 0 ? 1 : rc;
}

// =====================================================================================================================
// Fused ResnetBlock forward (unet1d.py:302-323): h1 = Block1(x, scale/shift), out = Block2(h1) + (res_conv(x) | x) in ONE
// pass.  The h1 tile (with one halo position each side) lives in shared memory, the skip path reads the staged x rows:
// HBM traffic per position drops from 4 (2 cin + 5 C) B to 4 (cin + [3 C saved for backward] + C) B.
struct ResFwdArgs {
  const float* x1; const float* x2;
  const float* w1; const float* b1; const float* g1; const float* ss;   // block1 (+ per-sample scale/shift)
  const float* w2; const float* b2; const float* g2;                    // block2
  const float* wres; const float* bres;                                 // 1x1 skip conv or null (identity: cin == COUT)
  float* u1; float* h1; float* u2;                                      // optional outputs saved for backward
  float* out;
  int c1, c2, R, L, rows_per_sample, ss_stride, tiles_per_row, total_tiles, tiles_per_cta;
};

template <int COUT, int P, int NT, bool BULK>
__global__ void __launch_bounds__(NT) resblock_fwd_tma_kernel(ResFwdArgs a) {
  constexpr int TL = NT * P;
  constexpr int TS = TL + 36;
  static_assert(P == 1 || P == 2 || P == 4, "P");
  static_assert(COUT % 4 == 0 && COUT <= 16, "COUT");
  extern __shared__ float4 dyn_smem4[];
  const int cin = a.c1 + a.c2;
  const bool has_res = a.wres != nullptr;
  float* stage0 = reinterpret_cast<float*>(dyn_smem4);
  const int stage_floats = cin * TS;
  float* h1_s = stage0 + 2 * stage_floats;                // COUT * TS   (position p at index p + 4)
  float* w1_s = h1_s + COUT * TS;                         // [(ci*3 + k) * COUT + co]
  float* w2_s = w1_s + cin * 3 * COUT;                    // [(c*3 + k) * COUT + co]
  float* wr_s = w2_s + COUT * 3 * COUT;                   // [ci * COUT + co]  (has_res)
  uint64_t* bars = reinterpret_cast<uint64_t*>(wr_s + cin * COUT);
  const int tid = threadIdx.x;
  const uint32_t bar0 = cf_smem_u32(bars), bar1 = bar0 + 8;
  if (tid == 0) {
    cf_mbar_init(bar0, BULK ? 1 : NT);
    cf_mbar_init(bar1, BULK ? 1 : NT);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < cin * 3 * COUT; i += NT) { const int co = i % COUT, ck = i / COUT; w1_s[i] = a.w1[(size_t)co * cin * 3 + ck]; }
  for (int i = tid; i < COUT * 3 * COUT; i += NT) { const int co = i % COUT, ck = i / COUT; w2_s[i] = a.w2[(size_t)co * COUT * 3 + ck]; }
  if (has_res)
    for (int i = tid; i < cin * COUT; i += NT) { const int co = i % COUT, ci = i / COUT; wr_s[i] = a.wres[(size_t)co * cin + ci]; }
  __syncthreads();
  const int t_begin = blockIdx.x * a.tiles_per_cta, t_end = min(a.total_tiles, t_begin + a.tiles_per_cta);
  const int n_tiles = t_end - t_begin;

  auto issue = [&](int tile, int s) {
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int l_lo = max(0, tl0 - 4), l_hi = min(a.L, tl0 + TL + 4);
    float* st = stage0 + s * stage_floats;
    if (!BULK) {
      const int w = l_hi - l_lo, doff = l_lo - (tl0 - 4);
      for (int row = tid >> 5; row < cin; row += NT / 32) {   // one warp per row
        const float* src = (row < a.c1 ? a.x1 + ((size_t)r * a.c1 + row) * a.L : a.x2 + ((size_t)r * a.c2 + (row - a.c1)) * a.L) + l_lo;
        const uint32_t dst = cf_smem_u32(st + row * TS + doff);
        for (int e = tid & 31; e < w; e += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
      }
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(s ? bar1 : bar0) : "memory");
      return;
    }
    if (tid < 32) {
      const uint32_t bytes = (uint32_t)(l_hi - l_lo) * 4u;
      const uint32_t bar = s ? bar1 : bar0;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (tid == 0) cf_mbar_expect_tx(bar, bytes * (uint32_t)cin);
      __syncwarp();
      for (int row = tid; row < cin; row += 32) {
        const float* src = row < a.c1 ? a.x1 + ((size_t)r * a.c1 + row) * a.L : a.x2 + ((size_t)r * a.c2 + (row - a.c1)) * a.L;
        cf_bulk_g2s(cf_smem_u32(st + row * TS + (l_lo - (tl0 - 4))), src + l_lo, bytes, bar);
      }
    }
  };
  if (n_tiles > 0) issue(t_begin, 0);
  if (n_tiles > 1) issue(t_begin + 1, 1);

  const float sqrtC = sqrtf((float)COUT);
  const bool has_ss = a.ss != nullptr;

  for (int it = 0; it < n_tiles; ++it) {
    const int tile = t_begin + it, s = it & 1;
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int sample = r / a.rows_per_sample;
    float* x_t = stage0 + s * stage_floats;
    cf_mbar_wait(s ? bar1 : bar0, (uint32_t)((it >> 1) & 1));
    // conv zero padding at the row ends (positions -1 and L) wherever they fall inside the staged window
    const bool edge = tl0 == 0 || a.L < tl0 + TL + 4;
    if (edge) {
      if (tid < cin) {
        if (tl0 == 0) x_t[tid * TS + 3] = 0.f;
        if (a.L < tl0 + TL + 4) x_t[tid * TS + (a.L - tl0 + 4)] = 0.f;
      }
      __syncthreads();
    }
    const int l = tl0 + P * tid;
    const int nvalid = a.L - l;                       // positions l + i with i < nvalid exist
    const size_t base = (size_t)r * COUT * a.L + l;

    // ------------------------------------------------------------ block 1: conv k3 + RMSNorm + scale/shift + SiLU -> h1 tile
    {
      float acc[P][COUT];
#pragma unroll
      for (int i = 0; i < P; ++i)
#pragma unroll
        for (int c = 0; c < COUT; ++c) acc[i][c] = a.b1[c];
#pragma unroll 2
      for (int ci = 0; ci < cin; ++ci) {
        float xw[P + 2];
        const float* xr = x_t + ci * TS + 4 + P * tid;
        if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(xr); xw[1] = m.x; xw[2] = m.y; xw[3] = m.z; xw[P] = m.w; }
        else if constexpr (P == 2) { const float2 m = *reinterpret_cast<const float2*>(xr); xw[1] = m.x; xw[P] = m.y; }
        else xw[1] = xr[0];
        xw[0] = xr[-1]; xw[P + 1] = xr[P];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float4* wp = reinterpret_cast<const float4*>(w1_s + (ci * 3 + k) * COUT);
#pragma unroll
          for (int c4 = 0; c4 < COUT / 4; ++c4) {
            const float4 w4 = wp[c4];
#pragma unroll
            for (int i = 0; i < P; ++i) {
              const float xv = xw[i + k];
              cf_fma2(acc[i][4 * c4 + 0], acc[i][4 * c4 + 1], xv, w4.x, w4.y);
              cf_fma2(acc[i][4 * c4 + 2], acc[i][4 * c4 + 3], xv, w4.z, w4.w);
            }
          }
        }
      }
      if (a.u1 && nvalid > 0) {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(a.u1 + base + (size_t)c * a.L) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
          else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(a.u1 + base + (size_t)c * a.L) = make_float2(acc[0][c], acc[P - 1][c]);
          else {
#pragma unroll
            for (int i = 0; i < P; ++i) if (i < nvalid) a.u1[base + (size_t)c * a.L + i] = acc[i][c];
          }
        }
      }
      float gs[COUT], sh[COUT];
#pragma unroll
      for (int c = 0; c < COUT; ++c) {
        const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + c] + 1.f : 1.f;
        gs[c] = a.g1[c] * sqrtC * sc1;
        sh[c] = has_ss ? a.ss[(size_t)sample * a.ss_stride + COUT + c] : 0.f;
      }
#pragma unroll
      for (int i = 0; i < P; ++i) {
        float s2 = 0.f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) s2 = fmaf(acc[i][c], acc[i][c], s2);
        const float inv = s2 > 1e-24f ? cf_rsqrt(s2) : 1e12f;
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          float z = fmaf(acc[i][c] * inv, gs[c], sh[c]);
          z = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
          acc[i][c] = (i < nvalid) ? z : 0.f;          // conv2 sees zero padding beyond the row end
        }
      }
#pragma unroll
      for (int c = 0; c < COUT; ++c) {
        if constexpr (P == 4) *reinterpret_cast<float4*>(h1_s + c * TS + 4 + P * tid) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
        else if constexpr (P == 2) *reinterpret_cast<float2*>(h1_s + c * TS + 4 + P * tid) = make_float2(acc[0][c], acc[P - 1][c]);
        else h1_s[c * TS + 4 + tid] = acc[0][c];
      }
      if (a.h1 && nvalid > 0) {
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(a.h1 + base + (size_t)c * a.L) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
          else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(a.h1 + base + (size_t)c * a.L) = make_float2(acc[0][c], acc[P - 1][c]);
          else {
#pragma unroll
            for (int i = 0; i < P; ++i) if (i < nvalid) a.h1[base + (size_t)c * a.L + i] = acc[i][c];
          }
        }
      }
    }
    if (tid < 32) {
      // h1 at the two halo positions tl0 - 1 (lanes 0-15) and tl0 + TL (lanes 16-31): one output channel per lane
      const int side = tid >> 4, c = tid & 15;
      const int idx = side == 0 ? 3 : TL + 4;
      const int lp = tl0 - 4 + idx;
      const bool ok = lp >= 0 && lp < a.L;
      const int cc = c < COUT ? c : 0;
      float acc = a.b1[cc];
      for (int ci = 0; ci < cin; ++ci) {
        const float* xr = x_t + ci * TS + idx;
#pragma unroll
        for (int k = 0; k < 3; ++k) acc = fmaf(xr[k - 1], w1_s[(ci * 3 + k) * COUT + cc], acc);
      }
      if (c >= COUT) acc = 0.f;
      float s2 = acc * acc;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      const float inv = s2 > 1e-24f ? cf_rsqrt(s2) : 1e12f;
      const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + cc] + 1.f : 1.f;
      const float shc = has_ss ? a.ss[(size_t)sample * a.ss_stride + COUT + cc] : 0.f;
      float z = fmaf(acc * inv, a.g1[cc] * sqrtC * sc1, shc);
      z = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
      if (c < COUT) h1_s[c * TS + idx] = ok ? z : 0.f;
    }
    __syncthreads();

    // ------------------------------------------------------------ block 2: conv k3 + RMSNorm + SiLU, + skip -> out
    {
      float acc[P][COUT];
#pragma unroll
      for (int i = 0; i < P; ++i)
#pragma unroll
        for (int c = 0; c < COUT; ++c) acc[i][c] = a.b2[c];
#pragma unroll 2
      for (int ci = 0; ci < COUT; ++ci) {
        float xw[P + 2];
        const float* xr = h1_s + ci * TS + 4 + P * tid;
        if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(xr); xw[1] = m.x; xw[2] = m.y; xw[3] = m.z; xw[P] = m.w; }
        else if constexpr (P == 2) { const float2 m = *reinterpret_cast<const float2*>(xr); xw[1] = m.x; xw[P] = m.y; }
        else xw[1] = xr[0];
        xw[0] = xr[-1]; xw[P + 1] = xr[P];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float4* wp = reinterpret_cast<const float4*>(w2_s + (ci * 3 + k) * COUT);
#pragma unroll
          for (int c4 = 0; c4 < COUT / 4; ++c4) {
            const float4 w4 = wp[c4];
#pragma unroll
            for (int i = 0; i < P; ++i) {
              const float xv = xw[i + k];
              cf_fma2(acc[i][4 * c4 + 0], acc[i][4 * c4 + 1], xv, w4.x, w4.y);
              cf_fma2(acc[i][4 * c4 + 2], acc[i][4 * c4 + 3], xv, w4.z, w4.w);
            }
          }
        }
      }
      if (nvalid > 0) {
        if (a.u2) {
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(a.u2 + base + (size_t)c * a.L) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
            else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(a.u2 + base + (size_t)c * a.L) = make_float2(acc[0][c], acc[P - 1][c]);
            else {
#pragma unroll
              for (int i = 0; i < P; ++i) if (i < nvalid) a.u2[base + (size_t)c * a.L + i] = acc[i][c];
            }
          }
        }
#pragma unroll
        for (int i = 0; i < P; ++i) {
          float s2 = 0.f;
#pragma unroll
          for (int c = 0; c < COUT; ++c) s2 = fmaf(acc[i][c], acc[i][c], s2);
          const float inv = (s2 > 1e-24f ? cf_rsqrt(s2) : 1e12f) * sqrtC;
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            float z = acc[i][c] * inv * a.g2[c];
            acc[i][c] = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
          }
        }
        // skip path from the staged x rows
        if (has_res) {
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            const float bb = a.bres ? a.bres[c] : 0.f;
#pragma unroll
            for (int i = 0; i < P; ++i) acc[i][c] += bb;
          }
          for (int ci = 0; ci < cin; ++ci) {
            float xv[P];
            const float* xr = x_t + ci * TS + 4 + P * tid;
            if constexpr (P == 4) { const float4 m = *reinterpret_cast<const float4*>(xr); xv[0] = m.x; xv[1] = m.y; xv[2] = m.z; xv[P - 1] = m.w; }
            else if constexpr (P == 2) { const float2 m = *reinterpret_cast<const float2*>(xr); xv[0] = m.x; xv[P - 1] = m.y; }
            else xv[0] = xr[0];
            const float4* wp = reinterpret_cast<const float4*>(wr_s + ci * COUT);
#pragma unroll
            for (int c4 = 0; c4 < COUT / 4; ++c4) {
              const float4 w4 = wp[c4];
#pragma unroll
              for (int i = 0; i < P; ++i) {
                acc[i][4 * c4 + 0] = fmaf(xv[i], w4.x, acc[i][4 * c4 + 0]);
                acc[i][4 * c4 + 1] = fmaf(xv[i], w4.y, acc[i][4 * c4 + 1]);
                acc[i][4 * c4 + 2] = fmaf(xv[i], w4.z, acc[i][4 * c4 + 2]);
                acc[i][4 * c4 + 3] = fmaf(xv[i], w4.w, acc[i][4 * c4 + 3]);
              }
            }
          }
        } else {
#pragma unroll
          for (int c = 0; c < COUT; ++c) {
            const float* xr = x_t + c * TS + 4 + P * tid;
#pragma unroll
            for (int i = 0; i < P; ++i) acc[i][c] += xr[i];
          }
        }
#pragma unroll
        for (int c = 0; c < COUT; ++c) {
          if constexpr (BULK && P == 4) *reinterpret_cast<float4*>(a.out + base + (size_t)c * a.L) = make_float4(acc[0][c], acc[1][c], acc[2][c], acc[P - 1][c]);
          else if constexpr (BULK && P == 2) *reinterpret_cast<float2*>(a.out + base + (size_t)c * a.L) = make_float2(acc[0][c], acc[P - 1][c]);
          else {
#pragma unroll
            for (int i = 0; i < P; ++i) if (i < nvalid) a.out[base + (size_t)c * a.L + i] = acc[i][c];
          }
        }
      }
    }
    __syncthreads();   // everyone is done with stage s and the h1 tile
    if (it + 2 < n_tiles) issue(tile + 2, s);
  }
}

template <int COUT, int P, int NT, bool BULK>
static int launch_resblock(ResFwdArgs a, cudaStream_t st) {
  constexpr int TL = NT * P, TS = TL + 36;
  const int cin = a.c1 + a.c2;
  a.tiles_per_row = (a.L + TL - 1) / TL;
  a.total_tiles = a.tiles_per_row * a.R;
  size_t smem = sizeof(float) * ((size_t)2 * cin * TS + (size_t)COUT * TS + (size_t)cin * 3 * COUT + (size_t)COUT * 3 * COUT + (size_t)cin * COUT) + 32;
  if (smem > 220 * 1024) return -6;
  auto kern = resblock_fwd_tma_kernel<COUT, P, NT, BULK>;
  static int sm_count = 0;
  if (!sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem);
  if (occ < 1) return -6;
  int grid = min(a.total_tiles, sm_count * occ);
  a.tiles_per_cta = (a.total_tiles + grid - 1) / grid;
  grid = (a.total_tiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
  kern<<<(unsigned)grid, NT, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}


// =====================================================================================================================
// Tensor-core form of the fused ResnetBlock forward for 8 / 12 / 16 channels (where 3 * cin * COUT FMAs per position and
// conv bound the FFMA kernel above: 25-60 % of HBM).  Same staging pipeline; a warp owns slabs of 16 positions and keeps
// everything in mma.sync m16n8k8 (TF32 operands, fp32 accumulate) fragment layout:
//   block 1: U1[pos][co] = b1 + sum_k X_k[pos][ci] W1_k[ci][co]  -> RMSNorm over co (quad shuffle) -> scale/shift -> SiLU
//            -> h1 tile in shared memory (TF32-rounded; the unrounded values go to the saved h1)
//   block 2: U2 = b2 + sum_k H1_k W2_k -> RMSNorm -> SiLU, + skip (1x1 conv of x as one more MMA chain, or x itself)
// k-slots are permuted (slot t <-> channel 2t, t+4 <-> 2t+1): with TS = 4 (mod 32) every fragment access is conflict-free.
// The two halo positions of the h1 tile are evaluated by one warp in fp32 FFMA (as in the kernel above).
template <int COUT, int KCI, int TL, int NT, bool BULK>
__global__ void __launch_bounds__(NT) resblock_fwd_mma_kernel(ResFwdArgs a) {
  constexpr int TS = TL + 36;
  constexpr int NW = NT / 32;
  constexpr int KCO = (COUT + 7) / 8;
  extern __shared__ float4 dyn_smem4[];
  const int cin = a.c1 + a.c2;
  const bool has_res = a.wres != nullptr;
  float* stage0 = reinterpret_cast<float*>(dyn_smem4);
  const int stage_floats = cin * TS;
  float* h1_s = stage0 + 2 * stage_floats;                // COUT * TS   (position p at index p + 4)
  float* w1_s = h1_s + COUT * TS;                         // [(ci*3 + k) * COUT + co]   (halo evaluation only)
  uint64_t* bars = reinterpret_cast<uint64_t*>(w1_s + ((cin * 3 * COUT + 3) & ~3));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, fg = lane >> 2, ft = lane & 3;
  const uint32_t bar0 = cf_smem_u32(bars), bar1 = bar0 + 8;
  if (tid == 0) {
    cf_mbar_init(bar0, BULK ? 1 : NT);
    cf_mbar_init(bar1, BULK ? 1 : NT);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < cin * 3 * COUT; i += NT) { const int co = i % COUT, ck = i / COUT; w1_s[i] = a.w1[(size_t)co * cin * 3 + ck]; }
  for (int i = tid; i < COUT * TS; i += NT) h1_s[i] = 0.f;
  for (int i = tid; i < 2 * stage_floats; i += NT) stage0[i] = 0.f;   // slots no copy fills stay finite
  // weight fragments (B operands): b0 = W[co = 8nt + fg][c = 8kc + 2ft], b1 = W[co][c + 1]
  uint32_t W1f[3][KCI][KCO][2], W2f[3][KCO][KCO][2], Wrf[KCI][KCO][2];
  float bias1[KCO][2], bias2[KCO][2], biasr[KCO][2], gg1[KCO][2], gg2[KCO][2];
  const float sqrtC = sqrtf((float)COUT);
#pragma unroll
  for (int nt = 0; nt < KCO; ++nt) {
    const int co = 8 * nt + fg;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
      for (int kc = 0; kc < KCI; ++kc) {
        const int ci = 8 * kc + 2 * ft + i;
        const bool in = ci < cin && co < COUT;
#pragma unroll
        for (int k = 0; k < 3; ++k) W1f[k][kc][nt][i] = cf_tf32(in ? a.w1[((size_t)co * cin + ci) * 3 + k] : 0.f);
        Wrf[kc][nt][i] = cf_tf32(in && has_res ? a.wres[(size_t)co * cin + ci] : 0.f);
      }
#pragma unroll
      for (int kc = 0; kc < KCO; ++kc) {
        const int c = 8 * kc + 2 * ft + i;
        const bool in = c < COUT && co < COUT;
#pragma unroll
        for (int k = 0; k < 3; ++k) W2f[k][kc][nt][i] = cf_tf32(in ? a.w2[((size_t)co * COUT + c) * 3 + k] : 0.f);
      }
      // per-thread channel constants of the accumulator columns co' = 8nt + 2ft + i
      const int cq = 8 * nt + 2 * ft + i;
      const bool inq = cq < COUT;
      bias1[nt][i] = inq ? a.b1[cq] : 0.f;
      bias2[nt][i] = inq ? a.b2[cq] : 0.f;
      biasr[nt][i] = (inq && has_res && a.bres) ? a.bres[cq] : 0.f;
      gg1[nt][i] = inq ? a.g1[cq] * sqrtC : 0.f;
      gg2[nt][i] = inq ? a.g2[cq] * sqrtC : 0.f;
    }
  }
  __syncthreads();
  const int t_begin = blockIdx.x * a.tiles_per_cta, t_end = min(a.total_tiles, t_begin + a.tiles_per_cta);
  const int n_tiles = t_end - t_begin;

  auto issue = [&](int tile, int s) {
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int l_lo = max(0, tl0 - 4), l_hi = min(a.L, tl0 + TL + 4);
    float* st = stage0 + s * stage_floats;
    if (!BULK) {
      const int w = l_hi - l_lo, doff = l_lo - (tl0 - 4);
      for (int row = warp; row < cin; row += NW) {   // one warp per row
        const float* src = (row < a.c1 ? a.x1 + ((size_t)r * a.c1 + row) * a.L : a.x2 + ((size_t)r * a.c2 + (row - a.c1)) * a.L) + l_lo;
        const uint32_t dst = cf_smem_u32(st + row * TS + doff);
        for (int e = lane; e < w; e += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (uint32_t)e), "l"(src + e) : "memory");
      }
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(s ? bar1 : bar0) : "memory");
      return;
    }
    if (tid < 32) {
      const uint32_t bytes = (uint32_t)(l_hi - l_lo) * 4u;
      const uint32_t bar = s ? bar1 : bar0;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (tid == 0) cf_mbar_expect_tx(bar, bytes * (uint32_t)cin);
      __syncwarp();
      for (int row = tid; row < cin; row += 32) {
        const float* src = row < a.c1 ? a.x1 + ((size_t)r * a.c1 + row) * a.L : a.x2 + ((size_t)r * a.c2 + (row - a.c1)) * a.L;
        cf_bulk_g2s(cf_smem_u32(st + row * TS + (l_lo - (tl0 - 4))), src + l_lo, bytes, bar);
      }
    }
  };
  if (n_tiles > 0) issue(t_begin, 0);
  if (n_tiles > 1) issue(t_begin + 1, 1);

  const bool has_ss = a.ss != nullptr;
  float gs1[KCO][2], sh1[KCO][2];
  int cur_sample = -1;

  // fragment (rows = positions p0 + fg, + 8; columns = channels 8nt + 2ft, + 1) -> (R, COUT, L) tensor
  auto store_frag = [&](float* dst, const float (&v)[KCO][4], bool ok0, bool ok1) {
#pragma unroll
    for (int nt = 0; nt < KCO; ++nt) {
      if (8 * nt + 2 * ft < COUT) {
        float* q = dst + (size_t)(8 * nt + 2 * ft) * a.L;
        if (ok0) { q[0] = v[nt][0]; q[a.L] = v[nt][1]; }
        if (ok1) { q[8] = v[nt][2]; q[a.L + 8] = v[nt][3]; }
      }
    }
  };
  // RMSNorm over the COUT channels of rows fg / fg + 8 of a fragment set: 1 / max(||u||, 1e-12)
  auto inv_norm = [&](const float (&v)[KCO][4], float& inv0, float& inv1) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < KCO; ++nt) {
      s0 = fmaf(v[nt][0], v[nt][0], fmaf(v[nt][1], v[nt][1], s0));
      s1 = fmaf(v[nt][2], v[nt][2], fmaf(v[nt][3], v[nt][3], s1));
    }
    s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
    s0 += __shfl_xor_sync(0xffffffffu, s0, 2); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
    inv0 = s0 > 1e-24f ? cf_rsqrt(s0) : 1e12f;
    inv1 = s1 > 1e-24f ? cf_rsqrt(s1) : 1e12f;
  };

  for (int it = 0; it < n_tiles; ++it) {
    const int tile = t_begin + it, s = it & 1;
    const int r = tile / a.tiles_per_row, tl0 = (tile - r * a.tiles_per_row) * TL;
    const int sample = r / a.rows_per_sample;
    if (sample != cur_sample) {
      cur_sample = sample;
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int cq = 8 * nt + 2 * ft + i;
          const bool inq = cq < COUT && has_ss;
          gs1[nt][i] = gg1[nt][i] * (inq ? a.ss[(size_t)sample * a.ss_stride + cq] + 1.f : 1.f);
          sh1[nt][i] = inq ? a.ss[(size_t)sample * a.ss_stride + COUT + cq] : 0.f;
        }
    }
    float* x_t = stage0 + s * stage_floats;
    cf_mbar_wait(s ? bar1 : bar0, (uint32_t)((it >> 1) & 1));
    // conv zero padding at the row ends (positions -1 and L) wherever they fall inside the staged window
    const bool edge = tl0 == 0 || a.L < tl0 + TL + 4;
    if (edge) {
      if (tid < cin) {
        if (tl0 == 0) x_t[tid * TS + 3] = 0.f;
        if (a.L < tl0 + TL + 4) x_t[tid * TS + (a.L - tl0 + 4)] = 0.f;
      }
      __syncthreads();
    }
    const size_t rbase = (size_t)r * COUT * a.L + tl0 + fg;
    const bool full = tl0 + TL <= a.L;

    // ------------------------------------------------------------ block 1 -> h1 tile
    for (int sl = warp; sl < TL / 16; sl += NW) {
      const int p0 = 16 * sl;
      const bool ok0 = full || tl0 + p0 + fg < a.L, ok1 = full || tl0 + p0 + fg + 8 < a.L;
      float u[KCO][4];
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt) { u[nt][0] = u[nt][2] = bias1[nt][0]; u[nt][1] = u[nt][3] = bias1[nt][1]; }
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int kc = 0; kc < KCI; ++kc) {
          const float* ap = x_t + min(8 * kc + 2 * ft, cin - 2) * TS + 4 + p0 + fg + k - 1;
          const uint32_t a0 = cf_rtf(ap[0]), a1 = cf_rtf(ap[8]), a2 = cf_rtf(ap[TS]), a3 = cf_rtf(ap[TS + 8]);
#pragma unroll
          for (int nt = 0; nt < KCO; ++nt) cf_mma8(u[nt], a0, a1, a2, a3, W1f[k][kc][nt][0], W1f[k][kc][nt][1]);
        }
      if (a.u1) store_frag(a.u1 + rbase + p0, u, ok0, ok1);
      float inv0, inv1;
      inv_norm(u, inv0, inv1);
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float z = fmaf(u[nt][i] * (i < 2 ? inv0 : inv1), gs1[nt][i & 1], sh1[nt][i & 1]);
          z = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
          u[nt][i] = ((i < 2) ? ok0 : ok1) ? z : 0.f;       // conv2 sees zero padding beyond the row end
        }
      if (a.h1) store_frag(a.h1 + rbase + p0, u, ok0, ok1);
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt)
        if (8 * nt + 2 * ft < COUT) {
          float* hp = h1_s + (8 * nt + 2 * ft) * TS + 4 + p0 + fg;
          hp[0] = __uint_as_float(cf_rtf(u[nt][0])); hp[TS] = __uint_as_float(cf_rtf(u[nt][1]));
          hp[8] = __uint_as_float(cf_rtf(u[nt][2])); hp[TS + 8] = __uint_as_float(cf_rtf(u[nt][3]));
        }
    }
    if (tid < 32) {
      // h1 at the two halo positions tl0 - 1 (lanes 0-15) and tl0 + TL (lanes 16-31): one output channel per lane
      const int side = tid >> 4, c = tid & 15;
      const int idx = side == 0 ? 3 : TL + 4;
      const int lp = tl0 - 4 + idx;
      const bool ok = lp >= 0 && lp < a.L;
      const int cc = c < COUT ? c : 0;
      float acc = a.b1[cc];
      for (int ci = 0; ci < cin; ++ci) {
        const float* xr = x_t + ci * TS + idx;
#pragma unroll
        for (int k = 0; k < 3; ++k) acc = fmaf(xr[k - 1], w1_s[(ci * 3 + k) * COUT + cc], acc);
      }
      if (c >= COUT) acc = 0.f;
      float s2 = acc * acc;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
      const float inv = s2 > 1e-24f ? cf_rsqrt(s2) : 1e12f;
      const float sc1 = has_ss ? a.ss[(size_t)sample * a.ss_stride + cc] + 1.f : 1.f;
      const float shc = has_ss ? a.ss[(size_t)sample * a.ss_stride + COUT + cc] : 0.f;
      float z = fmaf(acc * inv, a.g1[cc] * sqrtC * sc1, shc);
      z = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z));
      if (c < COUT) h1_s[c * TS + idx] = ok ? __uint_as_float(cf_rtf(z)) : 0.f;
    }
    __syncthreads();

    // ------------------------------------------------------------ block 2 + skip -> out
    for (int sl = warp; sl < TL / 16; sl += NW) {
      const int p0 = 16 * sl;
      const bool ok0 = full || tl0 + p0 + fg < a.L, ok1 = full || tl0 + p0 + fg + 8 < a.L;
      float u[KCO][4];
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt) { u[nt][0] = u[nt][2] = bias2[nt][0]; u[nt][1] = u[nt][3] = bias2[nt][1]; }
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int kc = 0; kc < KCO; ++kc) {
          const float* ap = h1_s + min(8 * kc + 2 * ft, COUT - 2) * TS + 4 + p0 + fg + k - 1;
          const uint32_t a0 = __float_as_uint(ap[0]), a1 = __float_as_uint(ap[8]);
          const uint32_t a2 = __float_as_uint(ap[TS]), a3 = __float_as_uint(ap[TS + 8]);
#pragma unroll
          for (int nt = 0; nt < KCO; ++nt) cf_mma8(u[nt], a0, a1, a2, a3, W2f[k][kc][nt][0], W2f[k][kc][nt][1]);
        }
      if (a.u2) store_frag(a.u2 + rbase + p0, u, ok0, ok1);
      float inv0, inv1;
      inv_norm(u, inv0, inv1);
      float sk[KCO][4];
      if (has_res) {   // CTA-uniform
#pragma unroll
        for (int nt = 0; nt < KCO; ++nt) { sk[nt][0] = sk[nt][2] = biasr[nt][0]; sk[nt][1] = sk[nt][3] = biasr[nt][1]; }
#pragma unroll
        for (int kc = 0; kc < KCI; ++kc) {
          const float* ap = x_t + min(8 * kc + 2 * ft, cin - 2) * TS + 4 + p0 + fg;
          const uint32_t a0 = cf_rtf(ap[0]), a1 = cf_rtf(ap[8]), a2 = cf_rtf(ap[TS]), a3 = cf_rtf(ap[TS + 8]);
#pragma unroll
          for (int nt = 0; nt < KCO; ++nt) cf_mma8(sk[nt], a0, a1, a2, a3, Wrf[kc][nt][0], Wrf[kc][nt][1]);
        }
      } else {         // identity skip (cin == COUT): exact fp32 x
#pragma unroll
        for (int nt = 0; nt < KCO; ++nt) {
          const float* xp = x_t + min(8 * nt + 2 * ft, COUT - 2) * TS + 4 + p0 + fg;
          sk[nt][0] = xp[0]; sk[nt][1] = xp[TS]; sk[nt][2] = xp[8]; sk[nt][3] = xp[TS + 8];
        }
      }
#pragma unroll
      for (int nt = 0; nt < KCO; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float z = u[nt][i] * (i < 2 ? inv0 : inv1) * gg2[nt][i & 1];
          u[nt][i] = z * cf_rcp(1.f + cf_ex2(-1.4426950408889634f * z)) + sk[nt][i];
        }
      store_frag(a.out + rbase + p0, u, ok0, ok1);
    }
    __syncthreads();   // everyone is done with stage s and the h1 tile
    if (it + 2 < n_tiles) issue(tile + 2, s);
  }
}

template <int COUT, int KCI, int TL, int NT, bool BULK>
static int launch_resblock_mma(ResFwdArgs a, cudaStream_t st) {
  constexpr int TS = TL + 36;
  const int cin = a.c1 + a.c2;
  a.tiles_per_row = (a.L + TL - 1) / TL;
  a.total_tiles = a.tiles_per_row * a.R;
  size_t smem = sizeof(float) * ((size_t)2 * cin * TS + (size_t)COUT * TS + (size_t)((cin * 3 * COUT + 3) & ~3)) + 32;
  if (smem > 220 * 1024) return -6;
  auto kern = resblock_fwd_mma_kernel<COUT, KCI, TL, NT, BULK>;
  static int sm_count = 0;
  if (!sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem);
  if (occ < 1) return -6;
  int grid = min(a.total_tiles, sm_count * occ);
  a.tiles_per_cta = (a.total_tiles + grid - 1) / grid;
  grid = (a.total_tiles + a.tiles_per_cta - 1) / a.tiles_per_cta;
  kern<<<(unsigned)grid, NT, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

}  // namespace dq

using namespace dq;

// Fused backward of a stride-1 Conv1d(K in {1,3}, pad (K-1)/2) and (if u != NULL) its RMSNorm / scale-shift /
// activation epilogue.  dx1/dx2 NULL = not needed; acc = accumulate into the destination; dadd (shape of dx1) is added
// to dx1.  dw / db / dg / dss are accumulated.
DQ_API int dq_conv_bwd_fused(const float* dy, const float* u, const float* g, const float* ss, int ss_stride, int act,
                             const float* x1, int c1, const float* x2, int c2, const float* w, const float* dadd,
                             float* dx1, int acc1, float* dx2, int acc2, float* dw, float* db, float* dg, float* dss,
                             int cout, int K, int R, int L, int rows_per_sample, void* stream) {
  ConvBwdFusedArgs a{dy, u, g, ss, x1, x2, w, dadd, dx1, dx2, dw, db, dg, dss, c1, c2, R, L, rows_per_sample, ss_stride,
                     act, acc1, acc2, 0, 0, 0};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || L <= 0) return 0;
  if (c1 + c2 > 64) return -3;
  if (K == 3) return dispatch_fused<3>(a, cout, st);
  if (K == 1) return dispatch_fused<1>(a, cout, st);
  return -2;
}

// Backward of Upsample = nearest x2 + Conv1d(k3, pad 1) (unet1d.py:93-96) in ONE pass: dy (R, cout, 2 Lh), x / dx
// (R, cin, Lh) at half rate; dw (cout, cin, 3) and db accumulated; dx NULL = not needed, acc = accumulate into dx.
// Returns 1 (nothing launched) if the shape is not covered: dq_upsample2x + dq_conv_bwd_fused + dq_fold2x instead.
DQ_API int dq_upconv_bwd_fused(const float* dy, const float* x, const float* w, float* dx, int acc, float* dw, float* db,
                               int cout, int cin, int R, int Lh, int rows_per_sample, void* stream) {
  ConvBwdFusedArgs a{dy, nullptr, nullptr, nullptr, x, nullptr, w, nullptr, dx, nullptr, dw, db, nullptr, nullptr, cin, 0, R,
                     2 * Lh, rows_per_sample, 0, 0, acc, 0, 0, 0, 0};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || Lh <= 0) return 0;
  if ((cin & 3) || cin > 64 || 2 * Lh < 128) return 1;
  const bool al = (Lh % 4 == 0) && ((((size_t)dy | (size_t)x | (size_t)dx) & 15) == 0);
  switch (cout) {
    case 4: return al ? launch_fused_tma<4, 3, 4, 128, false, true, false, 0, true>(a, st)
                      : launch_fused_tma<4, 3, 4, 128, false, false, false, 0, true>(a, st);
    case 8: return al ? launch_fused_tma<8, 3, 2, 128, false, true, false, 0, true>(a, st)
                      : launch_fused_tma<8, 3, 2, 128, false, false, false, 0, true>(a, st);
    case 12: return al ? launch_fused_tma<12, 3, 2, 128, false, true, false, 0, true>(a, st)
                       : launch_fused_tma<12, 3, 2, 128, false, false, false, 0, true>(a, st);
    case 16: return al ? launch_fused_tma<16, 3, 2, 128, false, true, false, 0, true>(a, st)
                       : launch_fused_tma<16, 3, 2, 128, false, false, false, 0, true>(a, st);
    default: return 1;
  }
}

// Backward of Downsample = Conv1d(k4, stride 2, pad 1) (unet1d.py:110) in ONE pass: dy (R, cout, L / 2), x / dx (R, cin, L),
// w / dw (cout, cin, 4); dw and db accumulated; dx NULL = not needed, acc = accumulate into dx.  Returns 1 (nothing
// launched) if the shape is not covered: dq_s2d + dq_down_w + dq_conv_bwd_fused + dq_d2s instead.
DQ_API int dq_downconv_bwd_fused(const float* dy, const float* x, const float* w, float* dx, int acc, float* dw, float* db,
                                 int cout, int cin, int R, int L, int rows_per_sample, void* stream) {
  ConvBwdFusedArgs a{dy, nullptr, nullptr, nullptr, x, nullptr, w, nullptr, dx, nullptr, dw, db, nullptr, nullptr, cin, 0, R,
                     L, rows_per_sample, 0, 0, acc, 0, 0, 0, 0};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || L <= 0) return 0;
  if ((cin & 3) || cin > 64 || (L & 1) || L < 128) return 1;
  const bool al = (L % 8 == 0) && ((((size_t)dy | (size_t)x | (size_t)dx) & 15) == 0);
  switch (cout) {
    case 4: return al ? launch_fused_tma<4, 4, 4, 128, false, true, false, 0, false, true>(a, st)
                      : launch_fused_tma<4, 4, 4, 128, false, false, false, 0, false, true>(a, st);
    case 8: return al ? launch_fused_tma<8, 4, 2, 128, false, true, false, 0, false, true>(a, st)
                      : launch_fused_tma<8, 4, 2, 128, false, false, false, 0, false, true>(a, st);
    case 12: return al ? launch_fused_tma<12, 4, 2, 128, false, true, false, 0, false, true>(a, st)
                       : launch_fused_tma<12, 4, 2, 128, false, false, false, 0, false, true>(a, st);
    case 16: return al ? launch_fused_tma<16, 4, 2, 128, false, true, false, 0, false, true>(a, st)
                       : launch_fused_tma<16, 4, 2, 128, false, false, false, 0, false, true>(a, st);
    default: return 1;
  }
}

// dq_conv_bwd_fused (K = 3, with epilogue) plus the backward of ResnetBlock.res_conv, a 1x1 convolution over the same
// input (x1 | x2) whose output gradient is dyo: dx1 / dx2 = conv3^T du + wres^T dyo in ONE pass over x (the separate
// calls read x twice and read-modify-write dx).  dwres / dbres accumulated.  Returns 1 if the shape is not covered.
DQ_API int dq_conv_bwd_fused_res(const float* dy, const float* u, const float* g, const float* ss, int ss_stride, int act,
                                 const float* x1, int c1, const float* x2, int c2, const float* w, float* dx1, float* dx2,
                                 float* dw, float* db, float* dg, float* dss, const float* dyo, const float* wres,
                                 float* dwres, float* dbres, int cout, int R, int L, int rows_per_sample, void* stream) {
  ConvBwdFusedArgs a{dy, u, g, ss, x1, x2, w, nullptr, dx1, dx2, dw, db, dg, dss, c1, c2, R, L, rows_per_sample, ss_stride,
                     act, 0, 0, 0, 0, 0};
  a.dyo = dyo; a.wres = wres; a.dwres = dwres; a.dbres = dbres;
  if (R <= 0 || L <= 0) return 0;
  if (!dyo || !wres || !dwres || !dx1 || c1 + c2 > 64) return 1;
  return dispatch_fused<3>(a, cout, (cudaStream_t)stream);
}

// Fused ResnetBlock forward (unet1d.py:302-323).  Returns 0 on success, 1 if the shape is not covered (the caller then
// composes the block from dq_conv1d_fwd calls), < 0 / cudaError on failure.  u1 / h1 / u2 may be NULL (inference).
DQ_API int dq_resblock_fwd(const float* x1, int c1, const float* x2, int c2, const float* w1, const float* b1, const float* g1,
                           const float* ss, int ss_stride, const float* w2, const float* b2, const float* g2,
                           const float* wres, const float* bres, float* u1, float* h1, float* u2, float* out, int cout,
                           int R, int L, int rows_per_sample, void* stream) {
  if (R <= 0 || L <= 0) return 0;
  const int cin = c1 + c2;
  if (L < 128 || cin > 32 || (cin & 3) || (c1 & 3) || (!wres && cin != cout)) return 1;
  ResFwdArgs a{x1, x2, w1, b1, g1, ss, w2, b2, g2, wres, bres, u1, h1, u2, out, c1, c2, R, L, rows_per_sample, ss_stride, 0, 0, 0};
  const bool al = (L % 4 == 0) && ((((size_t)x1 | (size_t)x2 | (size_t)u1 | (size_t)h1 | (size_t)u2 | (size_t)out) & 15) == 0);
  cudaStream_t st = (cudaStream_t)stream;
  if (cout >= 8) {
    const int kci = (cin + 7) / 8;
    if (al) {
      // (cout 8, cin 8: the FFMA2 kernel is as fast — 6 warp-instructions per position of conv work either way)
      if (cout == 8 && kci == 2) return launch_resblock_mma<8, 2, 256, 128, true>(a, st);
      if (cout == 12 && kci == 2) return launch_resblock_mma<12, 2, 256, 128, true>(a, st);
      if (cout == 12 && kci == 3) return launch_resblock_mma<12, 3, 256, 128, true>(a, st);
      if (cout == 16 && kci == 2) return launch_resblock_mma<16, 2, 128, 128, true>(a, st);
      if (cout == 16 && kci == 4) return launch_resblock_mma<16, 4, 128, 128, true>(a, st);
    } else {
      if (cout == 12 && kci == 2) return launch_resblock_mma<12, 2, 128, 128, false>(a, st);
      if (cout == 12 && kci == 3) return launch_resblock_mma<12, 3, 128, 128, false>(a, st);
      if (cout == 16 && kci == 2) return launch_resblock_mma<16, 2, 128, 128, false>(a, st);
      if (cout == 16 && kci == 4) return launch_resblock_mma<16, 4, 128, 128, false>(a, st);
    }
  }
  switch (cout) {
    case 4: return al ? launch_resblock<4, 4, 128, true>(a, st) : launch_resblock<4, 4, 128, false>(a, st);
    case 8: return al ? launch_resblock<8, 4, 128, true>(a, st) : launch_resblock<8, 2, 128, false>(a, st);
    case 12: return al ? launch_resblock<12, 2, 128, true>(a, st) : launch_resblock<12, 1, 128, false>(a, st);
    case 16: return al ? launch_resblock<16, 2, 128, true>(a, st) : launch_resblock<16, 1, 128, false>(a, st);
    default: return 1;
  }
}
