// tcgen05 / TMEM / TMA multi-tap GEMM for the 10 000-channel mid stage of the denoiser (sm_100a only).
//
//   C[M, N] (fp32, row-major, ldc)  (+)=  sum_{tap} A_tap[M, K] . B_tap[N, K]^T   (+ bias[N])
//
// A and B are bf16, K-major (K contiguous).  The taps express the 3-tap Conv1d over the RT axis as an implicit
// GEMM without im2col: tap t reads A shifted by a_row_off[t] rows and/or a_k_off[t] columns and B shifted by
// b_k_off[t] columns (multiples of 8 elements: TMA needs a 16-byte aligned innermost coordinate), from slice
// b_tap[t] of a (taps, N, K) weight tensor.  Out-of-range coordinates are
// zero-filled by TMA, per-sample halo rows are physical zero rows in the padded activation layout
// (see mid.cu), so no masking is needed in the main loop.
//
// Replaces (reference /root/reference/dquartic/model/unet1d.py): the four Conv1d(10000,10000,3,padding=1)
// of mid_block1/2 (243, 1029, 1058) forward / dgrad / wgrad, and Attention.to_qv / to_out 1x1 convs (534, 539).
//
// Structure: a persistent kernel, one CTA per SM, 192 threads = warp 0 TMA producer, warp 1 MMA issuer (+ TMEM
// alloc), warps 2-5 epilogue (TMEM lane quadrant = warp_idx % 4).  STAGES-deep smem ring of 128B-swizzled
// [128|BN] x 64 bf16 tiles filled by cp.async.bulk.tensor, consumed by tcgen05.mma.cta_group::1.kind::f16
// (M=128, N=BN, K=16) with fp32 accumulators in TMEM; tcgen05.commit releases ring slots / signals the epilogue.
//   * each CTA walks a static round-robin list of 128 x BN output tiles; the smem operand ring keeps running across
//     tiles
//   * two TMEM accumulator buffers: the epilogue warps drain tile i while the MMA warp already accumulates tile i+1
//   * tile width BN is a RUN-TIME multiple of 16 (<= 256) picked by the host so that tiles / #SMs has no ragged last wave
//     (M = 1152, N = 10000: 128 x 208 tiles -> 441 tiles = 2.98 waves instead of 360 tiles = 2.43 -> 3 waves at BN 256)
//   * tiles are rasterised in GM x GN super-tiles so that the operands of one wave fit the 126 MB L2 (the K = 9216 weight
//     gradient re-read its operands 26x from DRAM with the plain m-fastest order)
#include <cuda.h>
#include <string.h>
#include "common.cuh"

namespace dq {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle-128B row

struct GemmParams {
  float* C;
  const float* bias;
  long ldc;
  long z_c_stride;
  int M, N, K, taps;
  int a_row_off[4], a_k_off[4], b_k_off[4], b_tap[4];
  int z_b_koff_step, z_b_tap_step;
  int accumulate;
  int m_tiles;
  unsigned long long* err;  // device flag set on pipeline timeout (bring-up safety)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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
// Bounded wait: a descriptor / byte-count mistake must fail loudly instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, unsigned long long* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s
      if (err) atomicExch(err, (unsigned long long)code);
      __threadfence_system();
      __trap();
    }
  }
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// K-major, 128-byte swizzle: 8-row groups 1024 B apart (SBO = 64 x 16 B), LBO unused (=1), version 1, layout 2.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

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
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// the problem (GemmParams) plus the run-time tile width, ring depth and tile-walk geometry
struct GemmParams2 {
  GemmParams g;
  int bn, stages, tiles_m, tiles_n, nz, gm, gn;
};

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void decode_tile(const GemmParams2& p, int t, int& m_tile, int& n_tile, int& z) {
  const int per_z = p.tiles_m * p.tiles_n;
  z = t / per_z;
  int r = t - z * per_z;
  const int band_n = r / (p.gn * p.tiles_m);
  r -= band_n * p.gn * p.tiles_m;
  const int gn = min(p.gn, p.tiles_n - band_n * p.gn);
  const int band_m = r / (p.gm * gn);
  r -= band_m * p.gm * gn;
  const int gm = min(p.gm, p.tiles_m - band_m * p.gm);
  m_tile = band_m * p.gm + r % gm;
  n_tile = band_n * p.gn + r / gm;
}

// 16 consecutive output columns of one row: bias, optional accumulate, 128-bit stores when aligned
__device__ __forceinline__ void store_cols(const GemmParams& p, float* crow, int n, const uint32_t* r, int cnt, bool vec_ok) {
#pragma unroll
  for (int i = 0; i < 16; i += 4) {
    if (i >= cnt) break;
    const int nn = n + i;
    if (nn >= p.N) break;
    float v0 = __uint_as_float(r[i]), v1 = __uint_as_float(r[i + 1]), v2 = __uint_as_float(r[i + 2]), v3 = __uint_as_float(r[i + 3]);
    if (vec_ok && nn + 3 < p.N) {
      if (p.bias) {
        const float4 b4 = *reinterpret_cast<const float4*>(p.bias + nn);
        v0 += b4.x; v1 += b4.y; v2 += b4.z; v3 += b4.w;
      }
      float4* dst = reinterpret_cast<float4*>(crow + nn);
      if (p.accumulate) {
        const float4 o = *dst;
        v0 += o.x; v1 += o.y; v2 += o.z; v3 += o.w;
      }
      *dst = make_float4(v0, v1, v2, v3);
    } else {
      const float vv[4] = {v0, v1, v2, v3};
      for (int t = 0; t < 4 && nn + t < p.N; ++t) {
        float v = vv[t] + (p.bias ? p.bias[nn + t] : 0.f);
        if (p.accumulate) v += crow[nn + t];
        crow[nn + t] = v;
      }
    }
  }
}

__global__ void __launch_bounds__(192, 1)
gemm_tcgen05_persistent_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, GemmParams2 pp) {
  const GemmParams& p = pp.g;
  const int BN = pp.bn, STAGES = pp.stages;
  const uint32_t A_BYTES = BM * BK * 2, B_BYTES = (uint32_t)BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (sbase - smem_u32(smem_raw));
  const uint32_t bars = sbase + STAGES * STAGE_BYTES;   // full[STAGES], empty[STAGES], tfull[2], tempty[2], tmem slot
  const uint32_t full0 = bars, empty0 = bars + 8 * STAGES, tfull0 = bars + 16 * STAGES, tempty0 = tfull0 + 16;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(gen_base + STAGES * STAGE_BYTES + 16 * STAGES + 32);
  const uint32_t tmem_cols = BN > 128 ? 512u : 256u, buf_cols = tmem_cols / 2;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kblocks = (p.K + BK - 1) / BK;
  const int iters = kblocks * p.taps;
  const int total = pp.tiles_m * pp.tiles_n * pp.nz;

  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(full0 + 8 * s, 1);
        mbar_init(empty0 + 8 * s, 1);
      }
      for (int b = 0; b < 2; ++b) {
        mbar_init(tfull0 + 8 * b, 1);
        mbar_init(tempty0 + 8 * b, 4);   // one arrive per epilogue warp
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_d = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        int m_tile, n_tile, z;
        decode_tile(pp, t, m_tile, n_tile, z);
        const int m0 = m_tile * BM, n0 = n_tile * BN;
        for (int it = 0; it < iters; ++it) {
          const int tap = it / kblocks, kb = it - tap * kblocks;
          mbar_wait(empty0 + 8 * s, ph ^ 1, p.err, 1);
          mbar_expect_tx(full0 + 8 * s, STAGE_BYTES);
          const uint32_t sa = sbase + s * STAGE_BYTES, sb = sa + A_BYTES;
          tma_load_2d(sa, &tmA, full0 + 8 * s, kb * BK + p.a_k_off[tap], m0 + p.a_row_off[tap]);
          tma_load_3d(sb, &tmB, full0 + 8 * s, kb * BK + p.b_k_off[tap] + z * p.z_b_koff_step, n0, p.b_tap[tap] + z * p.z_b_tap_step);
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // instruction descriptor: D=f32, A=B=bf16, both K-major, N=BN, M=128
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      int s = 0;
      uint32_t ph = 0;
      int i = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
        const int buf = i & 1;
        mbar_wait(tempty0 + 8 * buf, (uint32_t)(((i >> 1) & 1) ^ 1), p.err, 4);   // epilogue has drained this buffer
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t td = tmem_d + (uint32_t)buf * buf_cols;
        for (int it = 0; it < iters; ++it) {
          mbar_wait(full0 + 8 * s, ph, p.err, 2);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa = sbase + s * STAGE_BYTES, sb = sa + A_BYTES;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_bf16(td, umma_desc_sw128(sa + k * 32), umma_desc_sw128(sb + k * 32), idesc, (it > 0 || k > 0) ? 1u : 0u);
          umma_commit(empty0 + 8 * s);   // frees the smem slot once these MMAs have read it
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit(tfull0 + 8 * buf);   // accumulator of this tile complete
      }
    }
  } else {
    // epilogue: warps 2..5 -> TMEM lane quadrant warp % 4
    const int q = warp & 3;
    int i = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++i) {
      int m_tile, n_tile, z;
      decode_tile(pp, t, m_tile, n_tile, z);
      const int m0 = m_tile * BM, n0 = n_tile * BN;
      const int buf = i & 1;
      mbar_wait(tfull0 + 8 * buf, (uint32_t)((i >> 1) & 1), p.err, 3);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int row = m0 + q * 32 + lane;
      float* crow = p.C + (size_t)z * p.z_c_stride + (size_t)row * p.ldc;
      const bool vec_ok = ((p.ldc & 3) == 0) && ((((size_t)(p.C + (size_t)z * p.z_c_stride)) & 15) == 0);
      const uint32_t tbase = tmem_d + (uint32_t)buf * buf_cols + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        if (c + 32 <= BN) {
          uint32_t r[32];
          tmem_ld32(tbase + (uint32_t)c, r);
          if (row < p.M && n0 + c < p.N) {
            store_cols(p, crow, n0 + c, r, 16, vec_ok);
            store_cols(p, crow, n0 + c + 16, r + 16, 16, vec_ok);
          }
        } else {
          uint32_t r[16];
          tmem_ld16(tbase + (uint32_t)c, r);
          if (row < p.M && n0 + c < p.N) store_cols(p, crow, n0 + c, r, 16, vec_ok);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8 * buf);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"(tmem_cols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

static unsigned long long* g_err_flag = nullptr;
static int g_sm_count = 0;

// tile width that minimises (waves x tile cost): no ragged last wave; ties go to the wider tile (less L2 traffic)
static int pick_bn(int m_tiles, int N, int nz, int sms) {
  if (N <= 128) return 128;
  if (N <= 256) return 256;
  int best = 256;
  double best_cost = 1e30;
  for (int bn = 256; bn >= 128; bn -= 16) {
    const long tiles = (long)m_tiles * ((N + bn - 1) / bn) * nz;
    const long waves = (tiles + sms - 1) / sms;
    const double cost = (double)waves * (bn + 24);
    if (cost < best_cost * 0.995) { best_cost = cost; best = bn; }
  }
  return best;
}

static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, GemmParams p, int nz, int bn, cudaStream_t st) {
  GemmParams2 pp;
  pp.g = p;
  pp.bn = bn;
  const size_t stage = (size_t)BM * BK * 2 + (size_t)bn * BK * 2;
  int stages = (int)((size_t)(225 * 1024) / stage);
  if (stages > 8) stages = 8;
  if (stages < 2) return -9;
  pp.stages = stages;
  pp.tiles_m = p.m_tiles;
  pp.tiles_n = (p.N + bn - 1) / bn;
  pp.nz = nz;
  pp.gm = 12;
  pp.gn = 12;
  const size_t smem = (size_t)stages * stage + 16 * stages + 32 + 16 + 1024;
  auto kern = gemm_tcgen05_persistent_kernel;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int total = pp.tiles_m * pp.tiles_n * nz;
  const int grid = total < g_sm_count ? total : g_sm_count;
  kern<<<(unsigned)grid, 192, smem, st>>>(tmA, tmB, pp);
  DQ_LAUNCH_CHECK();
  return 0;
}

}  // namespace dq

using namespace dq;

// A: bf16 (a_rows, a_cols) with leading dimension a_ld (elements); B: bf16 (b_ntaps, b_rows, b_cols) with
// row stride b_ld and tap stride b_tap_stride (elements).  All strides must be multiples of 8 elements (16 B).
// offs: 16 ints = a_row_off[4], a_k_off[4], b_k_off[4], b_tap[4].  bn: tile width, a multiple of 16 up to 256;
// any other value lets pick_bn choose it.
DQ_API int dq_gemm_bf16_tn(const void* A, long a_rows, long a_cols, long a_ld, const void* B, long b_rows, long b_cols,
                           long b_ld, long b_tap_stride, int b_ntaps, float* C, long ldc, const float* bias,
                           int accumulate, int M, int N, int K, int taps, const int* offs, int nz, int z_b_koff_step,
                           int z_b_tap_step, long z_c_stride, int bn, void* stream) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  if (taps < 1 || taps > 4) return -2;
  if ((a_ld % 8) || (b_ld % 8) || (b_tap_stride % 8) || (((size_t)A) & 15) || (((size_t)B) & 15)) return -4;
  EncodeTiledFn enc = get_encode();
  if (!enc) return -5;
  if (!g_err_flag) {
    if (cudaMalloc(&g_err_flag, sizeof(unsigned long long)) != cudaSuccess) return -6;
    cudaMemset(g_err_flag, 0, sizeof(unsigned long long));
  }
  if (!g_sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev); }
  if (nz < 1) nz = 1;
  if (bn <= 0 || bn % 16 || bn > 256) bn = pick_bn((M + BM - 1) / BM, N, nz, g_sm_count);
  CUtensorMap tmA, tmB;
  {
    cuuint64_t dims[2] = {(cuuint64_t)a_cols, (cuuint64_t)a_rows};
    cuuint64_t strides[1] = {(cuuint64_t)a_ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(A), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return -7;
  }
  {
    cuuint64_t dims[3] = {(cuuint64_t)b_cols, (cuuint64_t)b_rows, (cuuint64_t)b_ntaps};
    cuuint64_t strides[2] = {(cuuint64_t)b_ld * 2, (cuuint64_t)(b_ntaps > 1 ? b_tap_stride : b_ld * b_rows) * 2};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)bn, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(B), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return -8;
  }
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.C = C; p.bias = bias; p.ldc = ldc; p.z_c_stride = z_c_stride; p.M = M; p.N = N; p.K = K; p.taps = taps;
  for (int i = 0; i < 4; ++i) {
    p.a_row_off[i] = offs[i]; p.a_k_off[i] = offs[4 + i]; p.b_k_off[i] = offs[8 + i]; p.b_tap[i] = offs[12 + i];
  }
  for (int i = 0; i < taps; ++i) if ((offs[4 + i] % 8) || (offs[8 + i] % 8)) return -4;
  if (z_b_koff_step % 8) return -4;
  p.z_b_koff_step = z_b_koff_step; p.z_b_tap_step = z_b_tap_step; p.accumulate = accumulate; p.m_tiles = (M + BM - 1) / BM; p.err = g_err_flag;
  cudaStream_t st = (cudaStream_t)stream;
  return launch_gemm(tmA, tmB, p, nz, bn, st);
}

// reads (and clears) the pipeline-timeout flag: 0 = ok, 1 = producer, 2 = MMA, 3 = epilogue wait timed out
DQ_API int dq_gemm_last_error(void) {
  if (!g_err_flag) return 0;
  unsigned long long v = 0;
  if (cudaMemcpy(&v, g_err_flag, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  cudaMemset(g_err_flag, 0, sizeof(v));
  return (int)v;
}
