// Argument block shared by the LinearAttention kernels (linattn.cu: mma.sync TF32 kernels; linattn_tc.cu: tcgen05 kernels).
#pragma once
#include "common.cuh"

namespace dq {

struct LAArgs {
  const float* x;      // (R, C, L) block input
  const float* g_pre;  // (C) PreNorm gain
  const float* wqkv;   // (384, C)
  const float* wout;   // (C, 128)
  const float* bout;   // (C)
  const float* g_out;  // (C)
  float* part;         // (R, nchunk, 128, 2+CP) forward partials [m, s, M[CP]]
  float* msm;          // (R, 128, 2+CP)  [m, s, Ms[CP]]  saved for backward
  float* gmat;         // (R, C, 128)     G[c'][h*32+d]    saved for backward
  float* ypre;         // (R, C, L) to_out output before RMSNorm (saved for backward; may be null)
  float* out;          // (R, C, L)
  // backward
  const float* dres;   // (R, C, L) gradient of the block output
  float* dxnq;         // (R, C, L) scratch: q-path gradient w.r.t. the pre-normed input
  float* dpart;        // (R, nchunk, 128, CP) partial Gq
  float* hmat;         // (R, 128, CP)  H[h*32+d][c]
  float* sd;           // (R, 128)      sum_e dctx*ctx
  float* dx;           // (R, C, L)
  float* dwqkv;        // (384, C) accumulated
  float* dwout;        // (C, 128) accumulated
  float* dbout;        // (C) accumulated
  float* dg_out;       // (C) accumulated
  float* dg_pre;       // (C) accumulated
  int R, L, chunk, nchunk;
};

// tcgen05 / TMEM kernels (linattn_tc.cu).  Return 0 on launch, -3 when the channel count is not covered.
int la_bwd_q_tc(const LAArgs& a, int C, cudaStream_t st);   // C = 4, 8, 12

}  // namespace dq
