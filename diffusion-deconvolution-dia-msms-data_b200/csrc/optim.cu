// Fused optimizer step over the FLAT parameter / gradient buffers: global grad-norm (one reduction), clip
// coefficient on the device (no host sync), AdamW with decoupled weight decay, and the bf16 (+ transposed)
// operand refresh for the tcgen05 GEMMs (mid.cu: cast_transpose).
// Replaces (reference /root/reference/dquartic/model/model_interface.py): clip_grad_norm_(max_norm=10) 1121,
// torch.optim.AdamW(lr) 1011 / optimizer.step() 1122.  Traffic: 4 B/param (norm) + 28 B/param (update; 36 B/param with
// the weight EMA of dq_adamw_ema).
#include "common.cuh"

namespace dq {

__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, long n, double* out) {
  __shared__ double red[8];
  const long stride = (long)gridDim.x * blockDim.x;
  double acc = 0.0;
  const long n4 = ((((size_t)x) & 15) == 0) ? n / 4 : 0;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int cnt = 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = reinterpret_cast<const float4*>(x)[i];
    a0 = fmaf(v.x, v.x, a0); a1 = fmaf(v.y, v.y, a1); a2 = fmaf(v.z, v.z, a2); a3 = fmaf(v.w, v.w, a3);
    if (++cnt == 64) { acc += (double)a0 + (double)a1 + (double)a2 + (double)a3; a0 = a1 = a2 = a3 = 0.f; cnt = 0; }
  }
  acc += (double)a0 + (double)a1 + (double)a2 + (double)a3;
  for (long i = n4 * 4 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) acc += (double)x[i] * (double)x[i];
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    atomicAdd(out, t);
  }
}

// norm = gscale sqrt(sumsq); coef = gscale min(1, max_norm / (norm + 1e-6))   (torch.nn.utils.clip_grad_norm_ applied to
// gscale * g: under data parallelism the buffer holds the SUM over ranks and gscale = 1 / world-size, so the averaging
// costs no pass over the gradient)
__global__ void clip_coef_kernel(const double* sumsq, float max_norm, float gscale, float* out /* [0]=norm, [1]=coef */) {
  float norm = (float)sqrt(*sumsq) * gscale;
  float coef = max_norm / (norm + 1e-6f);
  out[0] = norm;
  out[1] = (coef < 1.f ? coef : 1.f) * gscale;
}

// torch.optim.AdamW single-tensor arithmetic, grads pre-scaled by the clip coefficient read from device memory.
// One AdamW element update (torch.optim.AdamW's op order: p *= 1 - lr wd; exp_avg.lerp_(g, 1 - b1); exp_avg_sq = b2 v +
// (1 - b2) g g; denom = sqrt(v) / sqrt(bc2) + eps; p -= step_size m / denom).  Explicitly rounded intrinsics: the scalar and
// the vector kernel below must agree bit for bit (a replicated parameter range may take either, depending on alignment).
__device__ __forceinline__ void adamw_update(float& pi, float gi, float& mi, float& vi, float coef, float decay, float b1,
                                             float b2, float eps, float step_size, float bc2_sqrt) {
  gi = __fmul_rn(gi, coef);
  pi = __fmul_rn(pi, decay);
  mi = __fmaf_rn(__fsub_rn(gi, mi), 1.f - b1, mi);
  vi = __fmaf_rn(vi, b2, __fmul_rn(__fmul_rn(1.f - b2, gi), gi));
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(vi), bc2_sqrt), eps);
  pi = __fmaf_rn(-step_size, __fdiv_rn(mi, denom), pi);
}

// Exponential moving average of the updated weight, ema += (1 - beta) (p - ema), rounded like adamw_update.
__device__ __forceinline__ void ema_update(float pi, float& ei, float ema_w) { ei = __fmaf_rn(__fsub_rn(pi, ei), ema_w, ei); }

// kEma: the same pass also moves the EMA buffer `ema` towards the updated weights (dq_adamw_ema): one more 4-byte load
// and store per element (36 instead of 28 B/param) instead of a second 12 B/param pass.
template <bool kEma>
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                    float* __restrict__ m, float* __restrict__ v, float* __restrict__ ema,
                                                    long n, const float* __restrict__ coef_ptr, float lr, float b1,
                                                    float b2, float eps, float wd, float step_size, float bc2_sqrt,
                                                    float ema_w) {
  const float coef = coef_ptr ? coef_ptr[1] : 1.f;
  const long stride = (long)gridDim.x * blockDim.x;
  const float decay = 1.f - lr * wd;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float pi = p[i], mi = m[i], vi = v[i];
    adamw_update(pi, g[i], mi, vi, coef, decay, b1, b2, eps, step_size, bc2_sqrt);
    p[i] = pi; m[i] = mi; v[i] = vi;
    if constexpr (kEma) {
      float ei = ema[i];
      ema_update(pi, ei, ema_w);
      ema[i] = ei;
    }
  }
}

// The same update on 16-byte vectors (all arrays 16-byte aligned: the whole flat buffer and the mid-stage ranges):
// 4 (5 with the EMA) x 16-byte loads + 3 (4) x 16-byte stores per thread and iteration instead of 7 (9) four-byte
// accesses; the n % 4 tail elements are handled by the first threads of the grid.  Arithmetic identical to adamw_kernel,
// element by element.
template <bool kEma>
__global__ void __launch_bounds__(256) adamw4_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                     float* __restrict__ m, float* __restrict__ v, float* __restrict__ ema,
                                                     long n, const float* __restrict__ coef_ptr, float lr, float b1,
                                                     float b2, float eps, float wd, float step_size, float bc2_sqrt,
                                                     float ema_w) {
  const float coef = coef_ptr ? coef_ptr[1] : 1.f;
  const long stride = (long)gridDim.x * blockDim.x;
  const float decay = 1.f - lr * wd;
  const long n4 = n >> 2;
  auto upd = [&](float& pi, float gi, float& mi, float& vi) {
    adamw_update(pi, gi, mi, vi, coef, decay, b1, b2, eps, step_size, bc2_sqrt);
  };
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 p4 = reinterpret_cast<float4*>(p)[i], m4 = reinterpret_cast<float4*>(m)[i], v4 = reinterpret_cast<float4*>(v)[i];
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(g) + i);
    upd(p4.x, g4.x, m4.x, v4.x);
    upd(p4.y, g4.y, m4.y, v4.y);
    upd(p4.z, g4.z, m4.z, v4.z);
    upd(p4.w, g4.w, m4.w, v4.w);
    reinterpret_cast<float4*>(p)[i] = p4;
    reinterpret_cast<float4*>(m)[i] = m4;
    reinterpret_cast<float4*>(v)[i] = v4;
    if constexpr (kEma) {
      float4 e4 = reinterpret_cast<float4*>(ema)[i];
      ema_update(p4.x, e4.x, ema_w);
      ema_update(p4.y, e4.y, ema_w);
      ema_update(p4.z, e4.z, ema_w);
      ema_update(p4.w, e4.w, ema_w);
      reinterpret_cast<float4*>(ema)[i] = e4;
    }
  }
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < (n & 3)) {
    const long i = (n4 << 2) + t;
    float pi = p[i], mi = m[i], vi = v[i];
    upd(pi, g[i], mi, vi);
    p[i] = pi; m[i] = mi; v[i] = vi;
    if constexpr (kEma) {
      float ei = ema[i];
      ema_update(pi, ei, ema_w);
      ema[i] = ei;
    }
  }
}

// Exchange two buffers in place (sampling from the EMA weights without a parameter-sized temporary).
__global__ void __launch_bounds__(256) swap_kernel(float* __restrict__ a, float* __restrict__ b, long n) {
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float t = a[i];
    a[i] = b[i];
    b[i] = t;
  }
}

__global__ void __launch_bounds__(256) swap4_kernel(float* __restrict__ a, float* __restrict__ b, long n) {
  const long stride = (long)gridDim.x * blockDim.x;
  const long n4 = n >> 2;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 t = reinterpret_cast<float4*>(a)[i];
    reinterpret_cast<float4*>(a)[i] = reinterpret_cast<float4*>(b)[i];
    reinterpret_cast<float4*>(b)[i] = t;
  }
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < (n & 3)) {
    const long i = (n4 << 2) + t;
    const float x = a[i];
    a[i] = b[i];
    b[i] = x;
  }
}

__global__ void __launch_bounds__(256) fill_kernel(float* __restrict__ p, float v, long n) {
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}

}  // namespace dq
using namespace dq;

DQ_API int dq_sumsq(const float* x, long n, double* out, void* stream) {
  if (n <= 0) return 0;
  long b = (n + 256L * 32 - 1) / (256L * 32);
  if (b > 148L * 8) b = 148L * 8;
  if (b < 1) b = 1;
  sumsq_kernel<<<(unsigned)b, 256, 0, (cudaStream_t)stream>>>(x, n, out);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_clip_coef(const double* sumsq, float max_norm, float gscale, float* out, void* stream) {
  clip_coef_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sumsq, max_norm, gscale, out);
  DQ_LAUNCH_CHECK();
  return 0;
}
// Grid of an elementwise kernel over n elements, `per_thread` of them per thread, at most 16 blocks per SM.
static unsigned ew_blocks(long n, long per_thread) {
  long b = (n + 256L * per_thread - 1) / (256L * per_thread);
  if (b > 148L * 16) b = 148L * 16;
  if (b < 1) b = 1;
  return (unsigned)b;
}

template <bool kEma>
static int launch_adamw(float* p, const float* g, float* m, float* v, float* ema, long n, const float* coef_ptr,
                        float lr, float b1, float b2, float eps, float wd, float step_size, float bc2_sqrt, float ema_w,
                        void* stream) {
  if (n <= 0) return 0;
  if (((((size_t)p) | ((size_t)g) | ((size_t)m) | ((size_t)v) | ((size_t)ema)) & 15) == 0 && n >= 4) {
    adamw4_kernel<kEma><<<ew_blocks(n / 4, 4), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, ema, n, coef_ptr, lr, b1, b2,
                                                                               eps, wd, step_size, bc2_sqrt, ema_w);
    DQ_LAUNCH_CHECK();
    return 0;
  }
  adamw_kernel<kEma><<<ew_blocks(n, 8), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, ema, n, coef_ptr, lr, b1, b2, eps, wd,
                                                                        step_size, bc2_sqrt, ema_w);
  DQ_LAUNCH_CHECK();
  return 0;
}

DQ_API int dq_adamw(float* p, const float* g, float* m, float* v, long n, const float* coef_ptr, float lr, float b1,
                    float b2, float eps, float wd, float step_size, float bc2_sqrt, void* stream) {
  return launch_adamw<false>(p, g, m, v, nullptr, n, coef_ptr, lr, b1, b2, eps, wd, step_size, bc2_sqrt, 0.f, stream);
}
DQ_API int dq_adamw_ema(float* p, const float* g, float* m, float* v, float* ema, long n, const float* coef_ptr,
                        float lr, float b1, float b2, float eps, float wd, float step_size, float bc2_sqrt, float ema_w,
                        void* stream) {
  return launch_adamw<true>(p, g, m, v, ema, n, coef_ptr, lr, b1, b2, eps, wd, step_size, bc2_sqrt, ema_w, stream);
}
DQ_API int dq_swap(float* a, float* b, long n, void* stream) {
  if (n <= 0) return 0;
  if (((((size_t)a) | ((size_t)b)) & 15) == 0 && n >= 4)
    swap4_kernel<<<ew_blocks(n / 4, 4), 256, 0, (cudaStream_t)stream>>>(a, b, n);
  else
    swap_kernel<<<ew_blocks(n, 8), 256, 0, (cudaStream_t)stream>>>(a, b, n);
  DQ_LAUNCH_CHECK();
  return 0;
}
DQ_API int dq_fill(float* p, float v, long n, void* stream) {
  if (n <= 0) return 0;
  long b = (n + 256L * 8 - 1) / (256L * 8);
  if (b > 148L * 16) b = 148L * 16;
  fill_kernel<<<(unsigned)b, 256, 0, (cudaStream_t)stream>>>(p, v, n);
  DQ_LAUNCH_CHECK();
  return 0;
}
