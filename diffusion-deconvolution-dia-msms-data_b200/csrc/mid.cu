// Mid-stage helpers around the tcgen05 GEMMs: the mid activations are kept as row-major [M = b*RT][N = d*mz]
// matrices (the reference's "(b rt) d mz -> b (d mz) rt" rearrange, unet1d.py:1144/1148, is a pure re-indexing of
// this layout and is never materialised).  For the 3-tap convolution over RT each sample is stored with one zero
// halo row on either side: padded row m' = s*(RT+2) + 1 + r.
//
//   mid_pack          fp32 [M][N]            -> bf16 padded [Mp][N]           (GEMM A operand)
//   transpose_bf16    bf16 [rows][N]         -> bf16 [N][ld]                  (wgrad operands, K = rows)
//   rownorm_fwd       RMSNorm(N) * g, (scale+1, shift), SiLU, + residual      (Block.forward 260-266 at C = N)
//   rowstats / colbwd backward of the above, row statistics then a column-parallel pass
//   attn_core         RoPE + softmax(q k^T / sqrt(32)) v for the RT x RT cross attention (unet1d.py:560-565, 428-443)
#include "common.cuh"

namespace dq {

__device__ __forceinline__ int padded_row(int m, int rt, int pad) { return pad ? (m / rt) * (rt + 2) + 1 + (m % rt) : m; }

// ---------------------------------------------------------------------------------------------- pack / transpose
__global__ void __launch_bounds__(256) mid_pack_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                       int b, int rt, int N, int pad) {
  // grid.x over padded rows
  const int rows_p = pad ? rt + 2 : rt;
  const int mp = blockIdx.x;
  const int s = mp / rows_p, rr = mp % rows_p;
  const bool halo = pad && (rr == 0 || rr == rt + 1);
  const float* src = halo ? nullptr : x + ((size_t)s * rt + (pad ? rr - 1 : rr)) * N;
  __nv_bfloat16* dst = out + (size_t)mp * N;
  for (int c = threadIdx.x * 2; c < N; c += blockDim.x * 2) {
    float2 v = halo ? make_float2(0.f, 0.f) : *reinterpret_cast<const float2*>(src + c);
    *reinterpret_cast<__nv_bfloat162*>(dst + c) = __floats2bfloat162_rn(v.x, v.y);
  }
}

__global__ void __launch_bounds__(256) transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in,
                                                             __nv_bfloat16* __restrict__ out, int rows, int cols,
                                                             long ld_out, int row_shift) {
  // out[c][r] = in[r + row_shift][c] (zero outside): the tap shift of the RT convolution is applied here
  // because TMA cannot start a box at an odd element of the contiguous dimension.
  __shared__ __nv_bfloat16 tile[32][34];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    int r = r0 + i + row_shift, c = c0 + tx;
    tile[i][tx] = (r >= 0 && r < rows && c < cols) ? in[(size_t)r * cols + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    int c = c0 + i, r = r0 + tx;
    if (c < cols && r < rows) out[(size_t)c * ld_out + r] = tile[tx][i];
  }
}

// The same on 64 x 64 tiles with packed bf16x2 loads and stores (rows, cols, ld_out even; 4-byte aligned bases): the
// 32 x 32 version above moved 2 bytes per thread and access (1.6 TB/s on the 2304 x 10000 activation transposes).
__global__ void __launch_bounds__(256) transpose_bf16_64_kernel(const __nv_bfloat16* __restrict__ in,
                                                                __nv_bfloat16* __restrict__ out, int rows, int cols,
                                                                long ld_out, int row_shift) {
  __shared__ __nv_bfloat16 tile[64][66];
  const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const __nv_bfloat162 zero2 = __floats2bfloat162_rn(0.f, 0.f);
#pragma unroll
  for (int i = ty; i < 64; i += 8) {
    const int r = r0 + i + row_shift, c = c0 + 2 * tx;
    __nv_bfloat162 v = zero2;
    if (r >= 0 && r < rows && c < cols) v = *reinterpret_cast<const __nv_bfloat162*>(in + (size_t)r * cols + c);
    *reinterpret_cast<__nv_bfloat162*>(&tile[i][2 * tx]) = v;
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < 64; i += 8) {
    const int c = c0 + i, r = r0 + 2 * tx;
    if (c < cols && r < rows) {
      __nv_bfloat162 v;
      v.x = tile[2 * tx][i];
      v.y = tile[2 * tx + 1][i];
      *reinterpret_cast<__nv_bfloat162*>(out + (size_t)c * ld_out + r) = v;
    }
  }
}

// fp32 [rows][cols] -> bf16 [rows][cols] and/or bf16 transposed [cols][rows]   (weight refresh after AdamW)
__global__ void __launch_bounds__(256) cast_transpose_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                             __nv_bfloat16* __restrict__ out_t, int rows, int cols) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    int r = r0 + i, c = c0 + tx;
    float v = (r < rows && c < cols) ? in[(size_t)r * cols + c] : 0.f;
    tile[i][tx] = v;
    if (out && r < rows && c < cols) out[(size_t)r * cols + c] = __float2bfloat16(v);
  }
  __syncthreads();
  if (out_t) {
    for (int i = ty; i < 32; i += 8) {
      int c = c0 + i, r = r0 + tx;
      if (c < cols && r < rows) out_t[(size_t)c * rows + r] = __float2bfloat16(tile[tx][i]);
    }
  }
}

// The same for even rows / cols and 4-byte aligned bases (every weight of the mid stage): 64 x 64 tiles, 8-byte loads,
// packed bf16x2 stores in both layouts (the 32 x 32 version wrote 64-byte rows with 2-byte stores: 2.9 TB/s).
__global__ void __launch_bounds__(256) cast_transpose64_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                               __nv_bfloat16* __restrict__ out_t, int rows, int cols) {
  __shared__ float tile[64][65];
  const int c0 = blockIdx.x * 64, r0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = ty; i < 64; i += 8) {
    const int r = r0 + i, c = c0 + 2 * tx;
    float2 v = make_float2(0.f, 0.f);
    if (r < rows && c < cols) v = *reinterpret_cast<const float2*>(in + (size_t)r * cols + c);   // cols even: c + 1 < cols
    tile[i][2 * tx] = v.x;
    tile[i][2 * tx + 1] = v.y;
    if (out && r < rows && c < cols) *reinterpret_cast<__nv_bfloat162*>(out + (size_t)r * cols + c) = __floats2bfloat162_rn(v.x, v.y);
  }
  __syncthreads();
  if (out_t) {
#pragma unroll
    for (int i = ty; i < 64; i += 8) {
      const int c = c0 + i, r = r0 + 2 * tx;
      if (c < cols && r < rows)                                                                  // rows even: r + 1 < rows
        *reinterpret_cast<__nv_bfloat162*>(out_t + (size_t)c * rows + r) = __floats2bfloat162_rn(tile[2 * tx][i], tile[2 * tx + 1][i]);
    }
  }
}

// ---------------------------------------------------------------------------------------------- row norm forward
struct RowNormArgs {
  const float* u;        // [Mp or M][N]   (padded if upad)
  const float* g;        // (N) or null: no normalisation (plain activation / copy)
  const float* ss;       // per-sample scale at ss[s*ss_stride + c], shift at ss[s*ss_stride + N + c]; or null
  const float* res;      // fp32 [M][N] residual added after the activation, or null
  float* out_f32;        // [M][N] or null
  __nv_bfloat16* out_bf16;  // padded (opad) or plain [M][N], or null
  float* inv_out;        // (M) 1/max(norm,eps) saved for backward, or null
  int b, rt, N, upad, opad, ss_stride, act;
};

// 16-byte vector version (N a multiple of 4, every base pointer 16-byte aligned - 8 bytes for the bf16 output): one row per
// CTA, the row stays in registers between the norm pass and the apply pass when it fits (N <= 10240: the 10000-channel
// mid stage), so u is read once; float4 loads of g / scale / shift / residual, float4 + 8-byte bf16x4 stores.  Same
// arithmetic per element as rownorm_fwd_kernel; the sum of squares is accumulated in a different order.
__global__ void __launch_bounds__(256) rownorm_fwd4_kernel(RowNormArgs a) {
  __shared__ float red[8];
  constexpr int KEEP = 10;
  const int m = blockIdx.x, tid = threadIdx.x;
  const int s = m / a.rt;
  const int nv = a.N >> 2;
  const float4* u4 = reinterpret_cast<const float4*>(a.u + (size_t)padded_row(m, a.rt, a.upad) * a.N);
  const bool keep = nv <= KEEP * 256;
  float4 buf[KEEP];
  float sc = 1.f;
  if (a.g) {
    float s2 = 0.f;
    if (keep) {
#pragma unroll
      for (int k = 0; k < KEEP; ++k) {
        const int i = tid + k * 256;
        buf[k] = i < nv ? u4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        s2 = fmaf(buf[k].x, buf[k].x, fmaf(buf[k].y, buf[k].y, fmaf(buf[k].z, buf[k].z, fmaf(buf[k].w, buf[k].w, s2))));
      }
    } else {
      for (int i = tid; i < nv; i += 256) {
        const float4 v = u4[i];
        s2 = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, s2))));
      }
    }
    s2 = warp_sum(s2);
    if ((tid & 31) == 0) red[tid >> 5] = s2;
    __syncthreads();
    float tot = 0.f;
    for (int w = 0; w < 8; ++w) tot += red[w];
    const float inv = 1.f / fmaxf(sqrtf(tot), 1e-12f);
    if (a.inv_out && tid == 0) a.inv_out[m] = inv;
    sc = inv * sqrtf((float)a.N);
  } else if (keep) {
#pragma unroll
    for (int k = 0; k < KEEP; ++k) {
      const int i = tid + k * 256;
      buf[k] = i < nv ? u4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  const float4* g4 = a.g ? reinterpret_cast<const float4*>(a.g) : nullptr;
  // (the scale / shift columns of a producer start at an even, not necessarily 4-aligned column of SS: 8-byte loads)
  const float2* sc2 = a.ss ? reinterpret_cast<const float2*>(a.ss + (size_t)s * a.ss_stride) : nullptr;
  const float2* sh2 = a.ss ? reinterpret_cast<const float2*>(a.ss + (size_t)s * a.ss_stride + a.N) : nullptr;
  const float4* r4 = a.res ? reinterpret_cast<const float4*>(a.res + (size_t)m * a.N) : nullptr;
  float4* of4 = a.out_f32 ? reinterpret_cast<float4*>(a.out_f32 + (size_t)m * a.N) : nullptr;
  uint2* ob4 = a.out_bf16 ? reinterpret_cast<uint2*>(a.out_bf16 + (size_t)padded_row(m, a.rt, a.opad) * a.N) : nullptr;
  auto apply = [&](float4 v, int i) {
    float z[4] = {v.x, v.y, v.z, v.w};
    if (g4) { const float4 gg = g4[i]; z[0] = z[0] * sc * gg.x; z[1] = z[1] * sc * gg.y; z[2] = z[2] * sc * gg.z; z[3] = z[3] * sc * gg.w; }
    if (sc2) {
      const float2 a0 = sc2[2 * i], a1 = sc2[2 * i + 1], b0 = sh2[2 * i], b1 = sh2[2 * i + 1];
      z[0] = fmaf(z[0], a0.x + 1.f, b0.x); z[1] = fmaf(z[1], a0.y + 1.f, b0.y);
      z[2] = fmaf(z[2], a1.x + 1.f, b1.x); z[3] = fmaf(z[3], a1.y + 1.f, b1.y);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) z[j] = act_fwd(z[j], a.act);
    if (r4) { const float4 rr = r4[i]; z[0] += rr.x; z[1] += rr.y; z[2] += rr.z; z[3] += rr.w; }
    if (of4) of4[i] = make_float4(z[0], z[1], z[2], z[3]);
    if (ob4) {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(z[0], z[1]), hi = __floats2bfloat162_rn(z[2], z[3]);
      ob4[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
    }
  };
  if (keep) {
#pragma unroll
    for (int k = 0; k < KEEP; ++k) {
      const int i = tid + k * 256;
      if (i < nv) apply(buf[k], i);
    }
  } else {
    for (int i = tid; i < nv; i += 256) apply(u4[i], i);
  }
}

__global__ void __launch_bounds__(256) rownorm_fwd_kernel(RowNormArgs a) {
  __shared__ float red[8];
  const int m = blockIdx.x;
  const int s = m / a.rt;
  const float* ur = a.u + (size_t)padded_row(m, a.rt, a.upad) * a.N;
  float sc = 1.f;
  if (a.g) {
    float s2 = 0.f;
    for (int c = threadIdx.x; c < a.N; c += blockDim.x) { float v = ur[c]; s2 = fmaf(v, v, s2); }
    s2 = warp_sum(s2);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s2;
    __syncthreads();
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    float inv = 1.f / fmaxf(sqrtf(tot), 1e-12f);
    if (a.inv_out && threadIdx.x == 0) a.inv_out[m] = inv;
    sc = inv * sqrtf((float)a.N);
  }
  const float* ssr = a.ss ? a.ss + (size_t)s * a.ss_stride : nullptr;
  const float* rr = a.res ? a.res + (size_t)m * a.N : nullptr;
  float* of = a.out_f32 ? a.out_f32 + (size_t)m * a.N : nullptr;
  __nv_bfloat16* ob = a.out_bf16 ? a.out_bf16 + (size_t)padded_row(m, a.rt, a.opad) * a.N : nullptr;
  for (int c = threadIdx.x; c < a.N; c += blockDim.x) {
    float z = ur[c];
    if (a.g) z = z * sc * a.g[c];
    if (ssr) z = fmaf(z, ssr[c] + 1.f, ssr[a.N + c]);
    z = act_fwd(z, a.act);
    if (rr) z += rr[c];
    if (of) of[c] = z;
    if (ob) ob[c] = __float2bfloat16(z);
  }
}

// ---------------------------------------------------------------------------------------------- row norm backward
struct RowNormBwdArgs {
  const float* dh;       // fp32 [M][N] gradient of the output
  const float* u;        // forward input (padded if upad)
  const float* g; const float* ss;
  const float* inv;      // (M) from forward (required when g)
  float* dot;            // (M) scratch: sum_c dû û
  __nv_bfloat16* du_bf16;   // padded (opad) or plain; halo rows must be pre-zeroed by the caller
  float* du_f32;         // [M][N] or null
  int du_acc;            // accumulate into du_f32
  float* dg;             // (N) accumulated
  float* dss;            // same layout as ss, accumulated
  float* dbias;          // (N) accumulated column sums of du (bias gradient of the producing GEMM), or null
  int b, rt, N, upad, opad, ss_stride, act, dhpad;
};

__global__ void __launch_bounds__(256) rownorm_rowstats_kernel(RowNormBwdArgs a) {
  __shared__ float red[8];
  const int m = blockIdx.x, s = m / a.rt;
  const float* ur = a.u + (size_t)padded_row(m, a.rt, a.upad) * a.N;
  const float* dr = a.dh + (size_t)padded_row(m, a.rt, a.dhpad) * a.N;
  const float* ssr = a.ss ? a.ss + (size_t)s * a.ss_stride : nullptr;
  const float inv = a.inv[m], sq = sqrtf((float)a.N);
  float acc = 0.f;
  for (int c = threadIdx.x; c < a.N; c += blockDim.x) {
    float uh = ur[c] * inv;
    float n = uh * a.g[c] * sq;
    float sc1 = ssr ? ssr[c] + 1.f : 1.f;
    float z = ssr ? fmaf(n, sc1, ssr[a.N + c]) : n;
    float dz = dr[c] * act_bwd(z, a.act);
    float duh = dz * sc1 * a.g[c] * sq;
    acc = fmaf(duh, uh, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    a.dot[m] = tot;
  }
}

// grid (ceil(N/256), b): thread = column c of sample s, loops over the RT rows of that sample
__global__ void __launch_bounds__(256) rownorm_colbwd_kernel(RowNormBwdArgs a) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
  if (c >= a.N) return;
  const float sq = sqrtf((float)a.N);
  const float gc = a.g ? a.g[c] : 1.f;
  const float* ssr = a.ss ? a.ss + (size_t)s * a.ss_stride : nullptr;
  const float sc1 = ssr ? ssr[c] + 1.f : 1.f, sh = ssr ? ssr[a.N + c] : 0.f;
  float dgc = 0.f, dsc = 0.f, dsh = 0.f, dbc = 0.f;
  for (int r = 0; r < a.rt; ++r) {
    const int m = s * a.rt + r;
    const float uv = a.u[(size_t)padded_row(m, a.rt, a.upad) * a.N + c];
    const float d = a.dh[(size_t)padded_row(m, a.rt, a.dhpad) * a.N + c];
    float du;
    if (a.g) {
      const float inv = a.inv[m];
      const float uh = uv * inv;
      const float n = uh * gc * sq;
      const float z = fmaf(n, sc1, sh);
      const float dz = d * act_bwd(z, a.act);
      dsc = fmaf(dz, n, dsc);
      dsh += dz;
      const float dn = dz * sc1;
      dgc = fmaf(dn * uh, sq, dgc);
      const float duh = dn * gc * sq;
      du = (inv < 1e12f) ? (duh - uh * a.dot[m]) * inv : duh * inv;
    } else {
      const float z = fmaf(uv, sc1, sh);
      const float dz = d * act_bwd(z, a.act);
      dsc = fmaf(dz, uv, dsc);
      dsh += dz;
      du = dz * sc1;
    }
    dbc += du;
    if (a.du_bf16) a.du_bf16[(size_t)padded_row(m, a.rt, a.opad) * a.N + c] = __float2bfloat16(du);
    if (a.du_f32) {
      float* p = a.du_f32 + (size_t)m * a.N + c;
      *p = a.du_acc ? *p + du : du;
    }
  }
  if (a.dg && a.g) atomicAdd(a.dg + c, dgc);
  if (a.dbias) atomicAdd(a.dbias + c, dbc);
  if (a.dss && ssr) {
    atomicAdd(a.dss + (size_t)s * a.ss_stride + c, dsc);
    atomicAdd(a.dss + (size_t)s * a.ss_stride + a.N + c, dsh);
  }
}

// out[c] += sum_r x[r][c]      (bias gradients of the 1x1 projections)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ x, float* __restrict__ out, int rows,
                                                     int cols, int rows_per_block) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float acc = 0.f;
  for (int r = r0; r < r1; ++r) acc += x[(size_t)r * cols + c];
  atomicAdd(out + c, acc);
}

// ---------------------------------------------------------------------------------------------- attention core
// qv fp32 [M][256] (q | v), k fp32 [M][128]; heads 4 x 32; RoPE on the first 16 features (interleaved pairs) of q, k.
// One CTA per (sample, head).  P (b, 4, rt, rt) saved for backward.
__device__ __forceinline__ void rope_rows(float* t, int rt, const float* __restrict__ freqs, bool inverse) {
  for (int i = threadIdx.x; i < rt * 8; i += blockDim.x) {
    int n = i / 8, p = i % 8;
    float ang = (float)n * freqs[p];
    float sn, cs;
    sincosf(ang, &sn, &cs);
    if (inverse) sn = -sn;
    float x1 = t[n * 33 + 2 * p], x2 = t[n * 33 + 2 * p + 1];
    t[n * 33 + 2 * p] = x1 * cs - x2 * sn;
    t[n * 33 + 2 * p + 1] = x2 * cs + x1 * sn;
  }
}

__global__ void __launch_bounds__(128) attn_core_fwd_kernel(const float* __restrict__ qv, const float* __restrict__ k,
                                                            const float* __restrict__ freqs, float* __restrict__ P,
                                                            float* __restrict__ o_f32, __nv_bfloat16* __restrict__ o_bf16,
                                                            int rt) {
  extern __shared__ float sm[];
  float* q_s = sm;                 // rt*33
  float* k_s = q_s + rt * 33;
  float* v_s = k_s + rt * 33;
  float* p_s = v_s + rt * 33;      // rt*rt
  const int s = blockIdx.x >> 2, h = blockIdx.x & 3;
  for (int i = threadIdx.x; i < rt * 32; i += blockDim.x) {
    int n = i >> 5, d = i & 31;
    size_t m = (size_t)s * rt + n;
    q_s[n * 33 + d] = qv[m * 256 + h * 32 + d];
    v_s[n * 33 + d] = qv[m * 256 + 128 + h * 32 + d];
    k_s[n * 33 + d] = k[m * 128 + h * 32 + d];
  }
  __syncthreads();
  rope_rows(q_s, rt, freqs, false);
  rope_rows(k_s, rt, freqs, false);
  __syncthreads();
  const float scale = rsqrtf(32.f);
  for (int i = threadIdx.x; i < rt * rt; i += blockDim.x) {
    int qi = i / rt, kj = i % rt;
    float acc = 0.f;
#pragma unroll
    for (int d = 0; d < 32; ++d) acc = fmaf(q_s[qi * 33 + d], k_s[kj * 33 + d], acc);
    p_s[i] = acc * scale;
  }
  __syncthreads();
  for (int qi = threadIdx.x >> 5; qi < rt; qi += (blockDim.x >> 5)) {  // one warp per query row
    const int lane = threadIdx.x & 31;
    float mx = -INFINITY;
    for (int j = lane; j < rt; j += 32) mx = fmaxf(mx, p_s[qi * rt + j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < rt; j += 32) { float e = __expf(p_s[qi * rt + j] - mx); p_s[qi * rt + j] = e; sum += e; }
    sum = warp_sum(sum);
    float inv = 1.f / sum;
    for (int j = lane; j < rt; j += 32) {
      float pv = p_s[qi * rt + j] * inv;
      p_s[qi * rt + j] = pv;
      if (P) P[(((size_t)s * 4 + h) * rt + qi) * rt + j] = pv;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < rt * 32; i += blockDim.x) {
    int n = i >> 5, d = i & 31;
    float acc = 0.f;
    for (int j = 0; j < rt; ++j) acc = fmaf(p_s[n * rt + j], v_s[j * 33 + d], acc);
    size_t idx = ((size_t)s * rt + n) * 128 + h * 32 + d;
    if (o_f32) o_f32[idx] = acc;
    if (o_bf16) o_bf16[idx] = __float2bfloat16(acc);
  }
}

// backward: dO fp32 [M][128] -> dqv fp32 [M][256] (+ bf16 copy), dk fp32 [M][128]
__global__ void __launch_bounds__(128) attn_core_bwd_kernel(const float* __restrict__ qv, const float* __restrict__ k,
                                                            const float* __restrict__ freqs, const float* __restrict__ P,
                                                            const float* __restrict__ dO, float* __restrict__ dqv,
                                                            __nv_bfloat16* __restrict__ dqv_bf16, float* __restrict__ dk,
                                                            int rt) {
  extern __shared__ float sm[];
  float* q_s = sm;                 // rotated q, later dq
  float* k_s = q_s + rt * 33;      // rotated k, later dk
  float* v_s = k_s + rt * 33;
  float* do_s = v_s + rt * 33;
  float* p_s = do_s + rt * 33;     // P, rt*rt
  float* ds_s = p_s + rt * rt;     // dS, rt*rt
  const int s = blockIdx.x >> 2, h = blockIdx.x & 3;
  for (int i = threadIdx.x; i < rt * 32; i += blockDim.x) {
    int n = i >> 5, d = i & 31;
    size_t m = (size_t)s * rt + n;
    q_s[n * 33 + d] = qv[m * 256 + h * 32 + d];
    v_s[n * 33 + d] = qv[m * 256 + 128 + h * 32 + d];
    k_s[n * 33 + d] = k[m * 128 + h * 32 + d];
    do_s[n * 33 + d] = dO[m * 128 + h * 32 + d];
  }
  for (int i = threadIdx.x; i < rt * rt; i += blockDim.x) p_s[i] = P[((size_t)s * 4 + h) * rt * rt + i];
  __syncthreads();
  rope_rows(q_s, rt, freqs, false);
  rope_rows(k_s, rt, freqs, false);
  __syncthreads();
  // dP[i][j] = dO[i] . v[j] ; dS = P * (dP - sum_j P dP)
  for (int i = threadIdx.x; i < rt * rt; i += blockDim.x) {
    int qi = i / rt, kj = i % rt;
    float acc = 0.f;
#pragma unroll
    for (int d = 0; d < 32; ++d) acc = fmaf(do_s[qi * 33 + d], v_s[kj * 33 + d], acc);
    ds_s[i] = acc;
  }
  __syncthreads();
  for (int qi = threadIdx.x >> 5; qi < rt; qi += (blockDim.x >> 5)) {
    const int lane = threadIdx.x & 31;
    float t = 0.f;
    for (int j = lane; j < rt; j += 32) t = fmaf(p_s[qi * rt + j], ds_s[qi * rt + j], t);
    t = warp_sum(t);
    for (int j = lane; j < rt; j += 32) ds_s[qi * rt + j] = p_s[qi * rt + j] * (ds_s[qi * rt + j] - t);
  }
  __syncthreads();
  const float scale = rsqrtf(32.f);
  // dv[j][d] = sum_i P[i][j] dO[i][d]  -> written straight to global
  for (int i = threadIdx.x; i < rt * 32; i += blockDim.x) {
    int n = i >> 5, d = i & 31;
    float acc = 0.f;
    for (int qi = 0; qi < rt; ++qi) acc = fmaf(p_s[qi * rt + n], do_s[qi * 33 + d], acc);
    size_t idx = ((size_t)s * rt + n) * 256 + 128 + h * 32 + d;
    dqv[idx] = acc;
    if (dqv_bf16) dqv_bf16[idx] = __float2bfloat16(acc);
  }
  // dq_rot[i][d] = scale * sum_j dS[i][j] k_rot[j][d] ; dk_rot[j][d] = scale * sum_i dS[i][j] q_rot[i][d]
  __syncthreads();
  // compute into do_s (dq) and v_s (dk) which are no longer needed after the sync above
  for (int i = threadIdx.x; i < rt * 32; i += blockDim.x) {
    int n = i >> 5, d = i & 31;
    float aq = 0.f, ak = 0.f;
    for (int j = 0; j < rt; ++j) {
      aq = fmaf(ds_s[n * rt + j], k_s[j * 33 + d], aq);
      ak = fmaf(ds_s[j * rt + n], q_s[j * 33 + d], ak);
    }
    do_s[n * 33 + d] = aq * scale;
    v_s[n * 33 + d] = ak * scale;
  }
  __syncthreads();
  rope_rows(do_s, rt, freqs, true);  // the rotation is orthogonal: gradient = inverse rotation
  rope_rows(v_s, rt, freqs, true);
  __syncthreads();
  for (int i = threadIdx.x; i < rt * 32; i += blockDim.x) {
    int n = i >> 5, d = i & 31;
    size_t m = (size_t)s * rt + n;
    float dq = do_s[n * 33 + d];
    dqv[m * 256 + h * 32 + d] = dq;
    if (dqv_bf16) dqv_bf16[m * 256 + h * 32 + d] = __float2bfloat16(dq);
    dk[m * 128 + h * 32 + d] = v_s[n * 33 + d];
  }
}

}  // namespace dq
using namespace dq;

DQ_API int dq_mid_pack(const float* x, void* out_bf16, int b, int rt, int N, int pad, void* stream) {
  if (b <= 0) return 0;
  if (N & 1) return -3;
  if (((size_t)x & 7) || ((size_t)out_bf16 & 3)) return -4;   // float2 loads, bf16x2 stores
  int rows = b * (pad ? rt + 2 : rt);
  mid_pack_kernel<<<(unsigned)rows, 256, 0, (cudaStream_t)stream>>>(x, (__nv_bfloat16*)out_bf16, b, rt, N, pad);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_transpose_bf16(const void* in, void* out, int rows, int cols, long ld_out, int row_shift, void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  if (((rows | cols) & 1) == 0 && (ld_out & 1) == 0 && (((size_t)in | (size_t)out) & 3) == 0) {
    dim3 grid64((unsigned)((cols + 63) / 64), (unsigned)((rows + 63) / 64));
    transpose_bf16_64_kernel<<<grid64, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)in, (__nv_bfloat16*)out, rows, cols, ld_out, row_shift);
    DQ_LAUNCH_CHECK();
    return 0;
  }
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32));
  transpose_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)in, (__nv_bfloat16*)out, rows, cols, ld_out, row_shift);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_cast_transpose(const float* in, void* out_bf16, void* out_t_bf16, int rows, int cols, void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  if (((rows | cols) & 1) == 0 && ((size_t)in & 7) == 0 && ((size_t)out_bf16 & 3) == 0 && ((size_t)out_t_bf16 & 3) == 0) {
    dim3 grid64((unsigned)((cols + 63) / 64), (unsigned)((rows + 63) / 64));
    cast_transpose64_kernel<<<grid64, 256, 0, (cudaStream_t)stream>>>(in, (__nv_bfloat16*)out_bf16, (__nv_bfloat16*)out_t_bf16, rows, cols);
    DQ_LAUNCH_CHECK();
    return 0;
  }
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32));
  cast_transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, (__nv_bfloat16*)out_bf16, (__nv_bfloat16*)out_t_bf16, rows, cols);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_rownorm_fwd(const float* u, int upad, const float* g, const float* ss, int ss_stride, int act,
                          const float* res, float* out_f32, void* out_bf16, int opad, float* inv_out, int b, int rt,
                          int N, void* stream) {
  if (b <= 0) return 0;
  RowNormArgs a{u, g, ss, res, out_f32, (__nv_bfloat16*)out_bf16, inv_out, b, rt, N, upad, opad, ss_stride, act};
  const size_t al = (size_t)u | (size_t)g | (size_t)res | (size_t)out_f32;
  if ((N & 3) == 0 && (al & 15) == 0 && (((size_t)out_bf16 | (size_t)ss) & 7) == 0 && (!ss || (ss_stride & 1) == 0)) {
    rownorm_fwd4_kernel<<<(unsigned)(b * rt), 256, 0, (cudaStream_t)stream>>>(a);
    DQ_LAUNCH_CHECK();
    return 0;
  }
  rownorm_fwd_kernel<<<(unsigned)(b * rt), 256, 0, (cudaStream_t)stream>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_colsum(const float* x, float* out, int rows, int cols, void* stream) {
  if (rows <= 0 || cols <= 0) return 0;
  int rpb = 64;
  dim3 grid((unsigned)((cols + 255) / 256), (unsigned)((rows + rpb - 1) / rpb));
  colsum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, out, rows, cols, rpb);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_rownorm_bwd(const float* dh, int dhpad, const float* u, int upad, const float* g, const float* ss,
                          int ss_stride, int act, const float* inv, float* dot, void* du_bf16, int opad,
                          float* du_f32, int du_acc, float* dg, float* dss, float* dbias, int b, int rt, int N,
                          void* stream) {
  if (b <= 0) return 0;
  RowNormBwdArgs a{dh, u, g, ss, inv, dot, (__nv_bfloat16*)du_bf16, du_f32, du_acc, dg, dss, dbias, b, rt, N, upad, opad, ss_stride, act, dhpad};
  cudaStream_t st = (cudaStream_t)stream;
  if (g) {
    rownorm_rowstats_kernel<<<(unsigned)(b * rt), 256, 0, st>>>(a);
    DQ_LAUNCH_CHECK();
  }
  dim3 grid((unsigned)((N + 255) / 256), (unsigned)b);
  rownorm_colbwd_kernel<<<grid, 256, 0, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}
// opt-in maximum of dynamic shared memory per block on the current device (227 KB on sm_100a)
static size_t attn_smem_limit() {
  int dev = 0, v = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  return (size_t)v;
}
DQ_API int dq_attn_core_fwd(const float* qv, const float* k, const float* freqs, float* P, float* o_f32, void* o_bf16,
                            int b, int rt, void* stream) {
  if (b <= 0) return 0;
  size_t smem = sizeof(float) * (3 * rt * 33 + rt * rt);
  if (smem > attn_smem_limit()) return -2;   // rt too long for one CTA's shared memory
  cudaFuncSetAttribute(attn_core_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  attn_core_fwd_kernel<<<(unsigned)(b * 4), 128, smem, (cudaStream_t)stream>>>(qv, k, freqs, P, o_f32, (__nv_bfloat16*)o_bf16, rt);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_attn_core_bwd(const float* qv, const float* k, const float* freqs, const float* P, const float* dO,
                            float* dqv, void* dqv_bf16, float* dk, int b, int rt, void* stream) {
  if (b <= 0) return 0;
  size_t smem = sizeof(float) * (4 * rt * 33 + 2 * rt * rt);
  if (smem > attn_smem_limit()) return -2;
  cudaFuncSetAttribute(attn_core_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  attn_core_bwd_kernel<<<(unsigned)(b * 4), 128, smem, (cudaStream_t)stream>>>(qv, k, freqs, P, dO, dqv, (__nv_bfloat16*)dqv_bf16, dk, rt);
  DQ_LAUNCH_CHECK();
  return 0;
}
