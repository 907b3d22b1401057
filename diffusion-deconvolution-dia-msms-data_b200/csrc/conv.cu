// Small-channel 1-D convolution family for the down/up path of the denoiser (C in {1..64}, L up to 40000):
// fused forward (dual-source concat read, ConditionalScaleShift on source 1, conv, bias, RMSNorm over channels,
// per-sample scale/shift, SiLU/GELU, residual add), pointwise backward of that epilogue, transposed-conv
// backward-data (dual destination, accumulate), and backward-weight/bias reduction.
//
// Replaces (reference, relative to /root/reference/dquartic/model/unet1d.py): Block.forward 248-268,
// ResnetBlock.forward 302-323, RMSNorm 140, Downsample 110, Upsample 93-96, init_conv 949/1117 with
// ConditionalScaleShift 677-678 and the cat at 1115, the skip cats at 1151/1154/1160, final_conv 1082.
//
// Layout: activations fp32 (R, C, L) channel-planar (the reference's NCL), R = batch*RT rows.  A thread owns
// all output channels of P positions (needed for the channel RMSNorm) that are blockDim apart, so every
// global access is a coalesced 128-byte line per warp; the K taps hit the same lines in L1.
#include "common.cuh"

namespace dq {

struct ConvFwdArgs {
  const float* x1; const float* x2;  // sources (R, c1, Lin), (R, c2, Lin); x2 may be null (c2 = 0)
  const float* in_ss;                // optional (b, in_ss_stride): source-1 channel c gets x*(ss[c]+1)+ss[c1+c]
  const float* w;                    // (cout, c1+c2, K)
  const float* bias;                 // (cout) or null
  const float* g;                    // RMSNorm gain (cout) or null (no norm)
  const float* ss;                   // optional per-sample scale/shift: scale = ss[s*ss_stride + c], shift = [.. + cout + c]
  const float* res;                  // optional residual (R, cout, Lout), added after the activation
  float* u;                          // optional pre-norm output (R, cout, Lout) saved for backward
  float* y;                          // output (R, cout, Lout)
  int c1, c2, R, Lin, Lout, pad, rows_per_sample, ss_stride, in_ss_stride, act;
};

template <int COUT, int K, int STRIDE, int UP, int P>
__global__ void __launch_bounds__(128) conv_fwd_kernel(ConvFwdArgs a) {
  constexpr int COUTP = (COUT + 3) / 4 * 4;
  extern __shared__ float w_s[];  // [(ci*K + k) * COUTP + co]
  const int cin = a.c1 + a.c2;
  for (int i = threadIdx.x; i < cin * K * COUTP; i += blockDim.x) {
    int co = i % COUTP, ck = i / COUTP;
    w_s[i] = (co < COUT) ? a.w[(size_t)co * cin * K + ck] : 0.f;
  }
  __syncthreads();
  const int tiles = (a.Lout + 128 * P - 1) / (128 * P);
  const int r = blockIdx.x / tiles, tile = blockIdx.x % tiles;
  const int l0 = tile * 128 * P + threadIdx.x;
  const int sample = r / a.rows_per_sample;
  const int LinV = a.Lin * UP;

  float acc[P][COUTP];
#pragma unroll
  for (int j = 0; j < P; ++j)
#pragma unroll
    for (int c = 0; c < COUTP; ++c) acc[j][c] = (a.bias && c < COUT) ? a.bias[c] : 0.f;

  for (int ci = 0; ci < cin; ++ci) {
    const float* xr;
    float sc = 1.f, sh = 0.f;
    if (ci < a.c1) {
      xr = a.x1 + ((size_t)r * a.c1 + ci) * a.Lin;
      if (a.in_ss) {
        sc = a.in_ss[(size_t)sample * a.in_ss_stride + ci] + 1.f;
        sh = a.in_ss[(size_t)sample * a.in_ss_stride + a.c1 + ci];
      }
    } else {
      xr = a.x2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.Lin;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float xv[P];
#pragma unroll
      for (int j = 0; j < P; ++j) {
        int lo = l0 + j * 128;
        int i = lo * STRIDE + k - a.pad;
        bool ok = (lo < a.Lout) && (i >= 0) && (i < LinV);
        float v = ok ? __ldg(xr + (UP == 1 ? i : (i / UP))) : 0.f;
        xv[j] = ok ? fmaf(v, sc, sh) : 0.f;
      }
      const float4* wp = reinterpret_cast<const float4*>(w_s + (ci * K + k) * COUTP);
#pragma unroll
      for (int c4 = 0; c4 < COUTP / 4; ++c4) {
        float4 w4 = wp[c4];
#pragma unroll
        for (int j = 0; j < P; ++j) {
          acc[j][c4 * 4 + 0] = fmaf(xv[j], w4.x, acc[j][c4 * 4 + 0]);
          acc[j][c4 * 4 + 1] = fmaf(xv[j], w4.y, acc[j][c4 * 4 + 1]);
          acc[j][c4 * 4 + 2] = fmaf(xv[j], w4.z, acc[j][c4 * 4 + 2]);
          acc[j][c4 * 4 + 3] = fmaf(xv[j], w4.w, acc[j][c4 * 4 + 3]);
        }
      }
    }
  }

  const float sqrtC = sqrtf((float)COUT);
#pragma unroll
  for (int j = 0; j < P; ++j) {
    int lo = l0 + j * 128;
    if (lo >= a.Lout) continue;
    size_t base = (size_t)r * COUT * a.Lout + lo;
    if (a.u) {
#pragma unroll
      for (int c = 0; c < COUT; ++c) a.u[base + (size_t)c * a.Lout] = acc[j][c];
    }
    float inv = 1.f;
    if (a.g) {
      float s2 = 0.f;
#pragma unroll
      for (int c = 0; c < COUT; ++c) s2 = fmaf(acc[j][c], acc[j][c], s2);
      inv = sqrtC / fmaxf(sqrtf(s2), 1e-12f);
    }
#pragma unroll
    for (int c = 0; c < COUT; ++c) {
      float z = acc[j][c];
      if (a.g) z = z * inv * a.g[c];
      if (a.ss) {
        float scale = a.ss[(size_t)sample * a.ss_stride + c];
        float shift = a.ss[(size_t)sample * a.ss_stride + COUT + c];
        z = fmaf(z, scale + 1.f, shift);
      }
      z = act_fwd(z, a.act);
      if (a.res) z += a.res[base + (size_t)c * a.Lout];
      a.y[base + (size_t)c * a.Lout] = z;
    }
  }
}

// ------------------------------------------------------------------ epilogue backward (Block.forward 260-266)
struct BlockBwdArgs {
  const float* dy;  // (R, C, L) gradient of the block output
  const float* u;   // (R, C, L) saved pre-norm conv output
  const float* g;   // (C) or null (no norm)
  const float* ss;  // per-sample scale/shift or null
  float* du;        // (R, C, L) gradient of the conv output
  float* dg;        // (C) accumulated (atomic) or null
  float* dss;       // same layout as ss, accumulated (atomic) or null
  int R, L, rows_per_sample, ss_stride, act, strip;
};

template <int C>
__global__ void __launch_bounds__(128) block_bwd_kernel(BlockBwdArgs a) {
  __shared__ float red[4 * 3 * C];
  const int strips = (a.L + a.strip - 1) / a.strip;
  const int r = blockIdx.x / strips, s0 = (blockIdx.x % strips) * a.strip;
  const int s1 = min(a.L, s0 + a.strip);
  const int sample = r / a.rows_per_sample;
  const float sqrtC = sqrtf((float)C);
  float gl[C], scale1[C], shift[C];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    gl[c] = a.g ? a.g[c] : 1.f;
    scale1[c] = a.ss ? a.ss[(size_t)sample * a.ss_stride + c] + 1.f : 1.f;
    shift[c] = a.ss ? a.ss[(size_t)sample * a.ss_stride + C + c] : 0.f;
  }
  float part[3 * C];
#pragma unroll
  for (int i = 0; i < 3 * C; ++i) part[i] = 0.f;

  for (int l = s0 + threadIdx.x; l < s1; l += blockDim.x) {
    size_t base = (size_t)r * C * a.L + l;
    float uv[C], dz[C];
    float s2 = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      uv[c] = a.u[base + (size_t)c * a.L];
      s2 = fmaf(uv[c], uv[c], s2);
    }
    float nrm = sqrtf(s2);
    float inv = a.g ? 1.f / fmaxf(nrm, 1e-12f) : 1.f;
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      float uh = uv[c] * inv;                                  // u-hat
      float n = a.g ? uh * gl[c] * sqrtC : uv[c];              // normalised
      float z = fmaf(n, scale1[c], shift[c]);
      float d = a.dy[base + (size_t)c * a.L] * act_bwd(z, a.act);
      part[C + c] += d * n;                                    // d scale
      part[2 * C + c] += d;                                    // d shift
      float dn = d * scale1[c];
      part[c] += dn * uh * sqrtC;                              // d g
      float duh = a.g ? dn * gl[c] * sqrtC : dn;               // d u-hat (no norm: plain d u)
      dz[c] = duh;
      dot = fmaf(duh, uh, dot);
      uv[c] = uh;
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
      float d;
      if (!a.g) d = dz[c];
      else if (nrm > 1e-12f) d = (dz[c] - uv[c] * dot) * inv;
      else d = dz[c] * inv;
      a.du[base + (size_t)c * a.L] = d;
    }
  }
  float tot = block_reduce_vec<3 * C>(part, red);
  int i = threadIdx.x;
  if (i < C) {
    if (a.dg && a.g) atomicAdd(a.dg + i, tot);
  } else if (i < 3 * C) {
    if (a.dss && a.ss) atomicAdd(a.dss + (size_t)sample * a.ss_stride + (i - C), tot);
  }
}

// ------------------------------------------------------------------ backward data (transposed conv)
struct ConvBwdDataArgs {
  const float* du;   // (R, cout, Lout)
  const float* w;    // (cout, cin, K)
  float* dx1;        // (R, c1, Lin) or null (skip)
  float* dx2;        // (R, c2, Lin) or null
  int acc1, acc2;    // accumulate into (1) or overwrite (0) each destination
  int c1, c2, cout, R, Lin, Lout, pad;
};

template <int K, int STRIDE, int UP, int P>
__global__ void __launch_bounds__(128) conv_bwd_data_kernel(ConvBwdDataArgs a) {
  constexpr int CT = 4;
  extern __shared__ float w_s[];  // [(co*K + k) * CT + ct]
  const int cin = a.c1 + a.c2;
  const int ci0 = blockIdx.y * CT;
  for (int i = threadIdx.x; i < a.cout * K * CT; i += blockDim.x) {
    int ct = i % CT, k = (i / CT) % K, co = i / (CT * K);
    int ci = ci0 + ct;
    w_s[i] = (ci < cin) ? a.w[((size_t)co * cin + ci) * K + k] : 0.f;
  }
  __syncthreads();
  const int tiles = (a.Lin + 128 * P - 1) / (128 * P);
  const int r = blockIdx.x / tiles, tile = blockIdx.x % tiles;
  const int l0 = tile * 128 * P + threadIdx.x;

  float acc[P][CT];
#pragma unroll
  for (int j = 0; j < P; ++j)
#pragma unroll
    for (int c = 0; c < CT; ++c) acc[j][c] = 0.f;

  for (int co = 0; co < a.cout; ++co) {
    const float* dr = a.du + ((size_t)r * a.cout + co) * a.Lout;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float4 w4 = *reinterpret_cast<const float4*>(w_s + (co * K + k) * CT);
#pragma unroll
      for (int j = 0; j < P; ++j) {
        int l = l0 + j * 128;
        float dsum = 0.f;
#pragma unroll
        for (int iu = 0; iu < UP; ++iu) {
          int num = l * UP + iu + a.pad - k;  // = lo * STRIDE
          bool ok = (l < a.Lin) && (num >= 0) && (num % STRIDE == 0) && (num / STRIDE < a.Lout);
          dsum += ok ? __ldg(dr + num / STRIDE) : 0.f;
        }
        acc[j][0] = fmaf(dsum, w4.x, acc[j][0]);
        acc[j][1] = fmaf(dsum, w4.y, acc[j][1]);
        acc[j][2] = fmaf(dsum, w4.z, acc[j][2]);
        acc[j][3] = fmaf(dsum, w4.w, acc[j][3]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < P; ++j) {
    int l = l0 + j * 128;
    if (l >= a.Lin) continue;
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) {
      int ci = ci0 + ct;
      if (ci >= cin) continue;
      float* dst;
      int accf;
      if (ci < a.c1) {
        dst = a.dx1 ? a.dx1 + ((size_t)r * a.c1 + ci) * a.Lin + l : nullptr;
        accf = a.acc1;
      } else {
        dst = a.dx2 ? a.dx2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.Lin + l : nullptr;
        accf = a.acc2;
      }
      if (dst) *dst = accf ? (*dst + acc[j][ct]) : acc[j][ct];
    }
  }
}

// ------------------------------------------------------------------ backward weight / bias
struct ConvBwdWeightArgs {
  const float* du;   // (R, cout, Lout)
  const float* x1; const float* x2;  // forward sources
  const float* in_ss;  // source-1 affine as in forward (or null)
  float* dw;         // (cout, cin, K) accumulated (atomic)
  float* db;         // (cout) accumulated (atomic) or null
  int c1, c2, cout, R, Lin, Lout, pad, rows_per_block, rows_per_sample, in_ss_stride, strip, strips;
};

template <int K, int STRIDE, int UP>
__global__ void __launch_bounds__(128) conv_bwd_weight_kernel(ConvBwdWeightArgs a) {
  constexpr int T = 4;  // 4 output channels x 4 input channels x K taps per thread
  constexpr int NV = T * T * K + T;
  __shared__ float red[4 * NV];
  const int cin = a.c1 + a.c2;
  const int co0 = blockIdx.y * T, ci0 = blockIdx.z * T;
  const int r0 = (blockIdx.x / a.strips) * a.rows_per_block, r1 = min(a.R, r0 + a.rows_per_block);
  const int lo0 = (blockIdx.x % a.strips) * a.strip, lo1 = min(a.Lout, lo0 + a.strip);
  const int LinV = a.Lin * UP;
  float acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.f;

  for (int r = r0; r < r1; ++r) {
    const int sample = r / a.rows_per_sample;
    const float* xr[T];
    float sc[T], sh[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      int ci = ci0 + t;
      sc[t] = 1.f; sh[t] = 0.f;
      if (ci >= cin) xr[t] = nullptr;
      else if (ci < a.c1) {
        xr[t] = a.x1 + ((size_t)r * a.c1 + ci) * a.Lin;
        if (a.in_ss) {
          sc[t] = a.in_ss[(size_t)sample * a.in_ss_stride + ci] + 1.f;
          sh[t] = a.in_ss[(size_t)sample * a.in_ss_stride + a.c1 + ci];
        }
      } else xr[t] = a.x2 + ((size_t)r * a.c2 + (ci - a.c1)) * a.Lin;
    }
    for (int lo = lo0 + threadIdx.x; lo < lo1; lo += blockDim.x) {
      float d[T];
#pragma unroll
      for (int t = 0; t < T; ++t) {
        int co = co0 + t;
        d[t] = (co < a.cout) ? __ldg(a.du + ((size_t)r * a.cout + co) * a.Lout + lo) : 0.f;
        acc[T * T * K + t] += d[t];
      }
#pragma unroll
      for (int k = 0; k < K; ++k) {
        int i = lo * STRIDE + k - a.pad;
        bool ok = (i >= 0) && (i < LinV);
        int ii = UP == 1 ? i : i / UP;
#pragma unroll
        for (int t = 0; t < T; ++t) {
          float xv = (ok && xr[t]) ? fmaf(__ldg(xr[t] + ii), sc[t], sh[t]) : 0.f;
#pragma unroll
          for (int o = 0; o < T; ++o) acc[(o * T + t) * K + k] = fmaf(d[o], xv, acc[(o * T + t) * K + k]);
        }
      }
    }
  }
  float tot = block_reduce_vec<NV>(acc, red);
  int i = threadIdx.x;
  if (i < T * T * K) {
    int k = i % K, t = (i / K) % T, o = i / (K * T);
    int co = co0 + o, ci = ci0 + t;
    if (co < a.cout && ci < cin) atomicAdd(a.dw + ((size_t)co * cin + ci) * K + k, tot);
  } else if (i < NV) {
    int co = co0 + (i - T * T * K);
    if (a.db && blockIdx.z == 0 && co < a.cout) atomicAdd(a.db + co, tot);
  }
}

// ------------------------------------------------------------------ per-sample reductions for ConditionalScaleShift
// d scale[s] += sum_{rows of s, l} d[r,l] * c[r,l];  d shift[s] += sum d[r,l]      (unet1d.py:677-678 backward)
__global__ void __launch_bounds__(256) sample_dot_kernel(const float* __restrict__ d, const float* __restrict__ c,
                                                         float* dscale, float* dshift, int out_stride, long n_per_sample) {
  __shared__ float red[8 * 2];
  const int s = blockIdx.y;
  const float* dp = d + (size_t)s * n_per_sample;
  const float* cp = c + (size_t)s * n_per_sample;
  float v[2] = {0.f, 0.f};
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n_per_sample; i += (long)gridDim.x * blockDim.x) {
    float dv = dp[i];
    v[0] = fmaf(dv, cp[i], v[0]);
    v[1] += dv;
  }
  float tot = block_reduce_vec<2>(v, red);
  if (threadIdx.x == 0) atomicAdd(dscale + (size_t)s * out_stride, tot);
  if (threadIdx.x == 1) atomicAdd(dshift + (size_t)s * out_stride, tot);
}

template <int COUT, int K, int STRIDE, int UP>
static int launch_fwd(const ConvFwdArgs& a, cudaStream_t st) {
  constexpr int P = (COUT <= 16) ? 4 : 2;
  constexpr int COUTP = (COUT + 3) / 4 * 4;
  size_t smem = (size_t)(a.c1 + a.c2) * K * COUTP * sizeof(float);
  auto kern = conv_fwd_kernel<COUT, K, STRIDE, UP, P>;
  if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  int tiles = (a.Lout + 128 * P - 1) / (128 * P);
  kern<<<(unsigned)(tiles * a.R), 128, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

template <int COUT>
static int dispatch_fwd_mode(const ConvFwdArgs& a, int K, int stride, int up, cudaStream_t st) {
  if (K == 3 && stride == 1 && up == 1) return launch_fwd<COUT, 3, 1, 1>(a, st);
  if (K == 3 && stride == 1 && up == 2) return launch_fwd<COUT, 3, 1, 2>(a, st);
  if (K == 4 && stride == 2 && up == 1) return launch_fwd<COUT, 4, 2, 1>(a, st);
  if (K == 7 && stride == 1 && up == 1) return launch_fwd<COUT, 7, 1, 1>(a, st);
  if (K == 1 && stride == 1 && up == 1) return launch_fwd<COUT, 1, 1, 1>(a, st);
  return -2;
}

template <int K, int STRIDE, int UP>
static int launch_bwd_data(const ConvBwdDataArgs& a, cudaStream_t st) {
  constexpr int P = 4;
  int cin = a.c1 + a.c2;
  size_t smem = (size_t)a.cout * K * 4 * sizeof(float);
  int tiles = (a.Lin + 128 * P - 1) / (128 * P);
  dim3 grid((unsigned)(tiles * a.R), (unsigned)((cin + 3) / 4));
  conv_bwd_data_kernel<K, STRIDE, UP, P><<<grid, 128, smem, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

template <int K, int STRIDE, int UP>
static int launch_bwd_weight(ConvBwdWeightArgs a, cudaStream_t st) {
  int cin = a.c1 + a.c2;
  // ~4096 positions per block: enough work to amortise the block-level reduction, enough blocks to fill 148 SMs
  constexpr int kStrip = 4096;
  int rpb = max(1, kStrip / max(1, a.Lout));
  a.rows_per_block = rpb;
  a.strip = (a.Lout > kStrip) ? kStrip : a.Lout;
  a.strips = (a.Lout + a.strip - 1) / a.strip;
  dim3 grid((unsigned)(((a.R + rpb - 1) / rpb) * a.strips), (unsigned)((a.cout + 3) / 4), (unsigned)((cin + 3) / 4));
  conv_bwd_weight_kernel<K, STRIDE, UP><<<grid, 128, 0, st>>>(a);
  DQ_LAUNCH_CHECK();
  return 0;
}

}  // namespace dq

using namespace dq;

namespace dq {
int conv_fwd_tma_try(const float* x1, int c1, const float* x2, int c2, const float* w, const float* bias, int cout, int K,
                     const float* g, const float* ss, int ss_stride, int act, const float* res, float* u, float* y, int R,
                     int L, int rows_per_sample, int up, cudaStream_t st, const float* in_ss = nullptr, int in_ss_stride = 0);
}

// C-ABI ---------------------------------------------------------------------------------------------------------
DQ_API int dq_conv1d_fwd(const float* x1, int c1, const float* x2, int c2, const float* in_ss, int in_ss_stride,
                         const float* w, const float* bias, int cout, int K, int stride, int pad, int up,
                         const float* g, const float* ss, int ss_stride, int act, const float* res,
                         float* u, float* y, int R, int Lin, int Lout, int rows_per_sample, void* stream) {
  ConvFwdArgs a{x1, x2, in_ss, w, bias, g, ss, res, u, y, c1, c2, R, Lin, Lout, pad, rows_per_sample, ss_stride,
                in_ss_stride, act};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || Lout <= 0) return 0;
  if (stride == 1 && (!in_ss || K == 7) && pad == (K - 1) / 2 && ((up == 1 && Lin == Lout) || (up == 2 && 2 * Lin == Lout))) {
    // bulk-copy pipelined kernel (conv_fused.cu)
    int rc = conv_fwd_tma_try(x1, c1, x2, c2, w, bias, cout, K, g, ss, ss_stride, act, res, u, y, R, Lout, rows_per_sample, up, st,
                              in_ss, in_ss_stride);
    if (rc != 0) return rc < 0 ? rc : 0;
  }
  if (stride == 2 && K == 4 && pad == 1 && up == 1 && !in_ss && !x2 && !res && Lin == 2 * Lout) {
    // Downsample (unet1d.py:110) through the same pipelined kernel (up = -2: stride-2 mode)
    int rc = conv_fwd_tma_try(x1, c1, nullptr, 0, w, bias, cout, K, g, ss, ss_stride, act, nullptr, u, y, R, Lout, rows_per_sample, -2, st);
    if (rc != 0) return rc < 0 ? rc : 0;
  }
  switch (cout) {
    case 1: return dispatch_fwd_mode<1>(a, K, stride, up, st);
    case 4: return dispatch_fwd_mode<4>(a, K, stride, up, st);
    case 8: return dispatch_fwd_mode<8>(a, K, stride, up, st);
    case 12: return dispatch_fwd_mode<12>(a, K, stride, up, st);
    case 16: return dispatch_fwd_mode<16>(a, K, stride, up, st);
    case 24: return dispatch_fwd_mode<24>(a, K, stride, up, st);
    case 32: return dispatch_fwd_mode<32>(a, K, stride, up, st);
    default: return -3;
  }
}

DQ_API int dq_block_bwd(const float* dy, const float* u, const float* g, const float* ss, int ss_stride, int act,
                        float* du, float* dg, float* dss, int C, int R, int L, int rows_per_sample, void* stream) {
  BlockBwdArgs a{dy, u, g, ss, du, dg, dss, R, L, rows_per_sample, ss_stride, act, 4096};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || L <= 0) return 0;
  int strips = (L + a.strip - 1) / a.strip;
  unsigned grid = (unsigned)(strips * R);
  switch (C) {
    case 4: block_bwd_kernel<4><<<grid, 128, 0, st>>>(a); break;
    case 8: block_bwd_kernel<8><<<grid, 128, 0, st>>>(a); break;
    case 12: block_bwd_kernel<12><<<grid, 128, 0, st>>>(a); break;
    case 16: block_bwd_kernel<16><<<grid, 128, 0, st>>>(a); break;
    case 24: block_bwd_kernel<24><<<grid, 128, 0, st>>>(a); break;
    case 32: block_bwd_kernel<32><<<grid, 128, 0, st>>>(a); break;
    default: return -3;
  }
  DQ_LAUNCH_CHECK();
  return 0;
}

DQ_API int dq_conv1d_bwd_data(const float* du, const float* w, float* dx1, int c1, int acc1, float* dx2, int c2,
                              int acc2, int cout, int K, int stride, int pad, int up, int R, int Lin, int Lout,
                              void* stream) {
  ConvBwdDataArgs a{du, w, dx1, dx2, acc1, acc2, c1, c2, cout, R, Lin, Lout, pad};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || Lin <= 0) return 0;
  if (K == 3 && stride == 1 && up == 1) return launch_bwd_data<3, 1, 1>(a, st);
  if (K == 3 && stride == 1 && up == 2) return launch_bwd_data<3, 1, 2>(a, st);
  if (K == 4 && stride == 2 && up == 1) return launch_bwd_data<4, 2, 1>(a, st);
  if (K == 7 && stride == 1 && up == 1) return launch_bwd_data<7, 1, 1>(a, st);
  if (K == 1 && stride == 1 && up == 1) return launch_bwd_data<1, 1, 1>(a, st);
  return -2;
}

DQ_API int dq_conv1d_bwd_weight(const float* du, const float* x1, int c1, const float* x2, int c2,
                                const float* in_ss, int in_ss_stride, float* dw, float* db, int cout, int K,
                                int stride, int pad, int up, int R, int Lin, int Lout, int rows_per_sample,
                                void* stream) {
  ConvBwdWeightArgs a{du, x1, x2, in_ss, dw, db, c1, c2, cout, R, Lin, Lout, pad, 1, rows_per_sample, in_ss_stride, Lout, 1};
  cudaStream_t st = (cudaStream_t)stream;
  if (R <= 0 || Lout <= 0) return 0;
  if (K == 3 && stride == 1 && up == 1) return launch_bwd_weight<3, 1, 1>(a, st);
  if (K == 3 && stride == 1 && up == 2) return launch_bwd_weight<3, 1, 2>(a, st);
  if (K == 4 && stride == 2 && up == 1) return launch_bwd_weight<4, 2, 1>(a, st);
  if (K == 7 && stride == 1 && up == 1) return launch_bwd_weight<7, 1, 1>(a, st);
  if (K == 1 && stride == 1 && up == 1) return launch_bwd_weight<1, 1, 1>(a, st);
  return -2;
}

DQ_API int dq_sample_dot(const float* d, const float* c, float* dscale, float* dshift, int out_stride,
                         long n_per_sample, int n_samples, void* stream) {
  if (n_samples <= 0 || n_per_sample <= 0) return 0;
  int bx = (int)((n_per_sample + 256 * 16 - 1) / (256 * 16));
  if (bx > 1024) bx = 1024;
  dim3 grid((unsigned)bx, (unsigned)n_samples);
  sample_dot_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d, c, dscale, dshift, out_stride, n_per_sample);
  DQ_LAUNCH_CHECK();
  return 0;
}
