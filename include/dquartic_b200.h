/* dquartic_b200.h — C-ABI of the B200-native (sm_100a) dquartic hot path.
 *
 * The reference (Roestlab/diffusion-deconvolution-dia-msms-data, "dquartic") is pure Python/PyTorch and has no
 * FFI seam of its own; its boundary for this path is the Python module API (dquartic.model.unet1d.UNet1d,
 * dquartic.model.model.DDIMDiffusionModel, dquartic.model.model_interface.ModelInterface,
 * dquartic.utils.data_loader.DIAMSDataset).  The replacement modules under
 * diffusion-deconvolution-dia-msms-data_b200/dquartic/ keep that API and call the entry points below through
 * ctypes (diffusion-deconvolution-dia-msms-data_b200/dquartic/_native.py).  INTEGRATION.md shows the binding.
 *
 * Conventions: every pointer is a DEVICE pointer owned by the caller (no allocation inside, except the one-off
 * 8-byte GEMM error flag); every call is asynchronous on `stream` (a cudaStream_t passed as void*); the return
 * value is 0 on success, a positive cudaError_t, or a negative argument error (-2 unsupported mode,
 * -3 unsupported channel count / dtype, -4 misaligned GEMM operand, -5..-8 TMA descriptor failures).
 * Activations are fp32, channel-planar (R, C, L) with R = batch*RT rows ("NCL"), unless stated.
 * `act`: 0 none, 1 SiLU, 2 GELU(erf).  Citations are relative to /root/reference/dquartic/.
 */
#ifndef DQUARTIC_B200_H
#define DQUARTIC_B200_H
#ifdef __cplusplus
extern "C" {
#endif

/* ---- scheduler / loss (model/model.py) ---------------------------------------------------------------- */
/* q_sample with the auto-normalise of x0 fused: model.py:99, 239-242 (train_step 349-352). */
int dq_qsample(const float* x0, const float* noise, const long long* t, const float* alpha_bars, float* xt,
               int b, long n_per_sample, int auto_norm, void* stream);
/* y = (wa*a + wb*b)*m + c : harness mixing model_interface.py:1073-1075 + normalize model.py:99 (b may be NULL). */
int dq_mix_affine(const float* a, const float* b, float wa, float wb, float m, float c, float* y, long n, void* stream);
/* y = (x + c)*m : unnormalize model.py:112. */
int dq_add_mul(const float* x, float c, float m, float* y, long n, void* stream);
/* DDIM reverse step, eta=0, pred_type eps: model.py:273, 283-289. */
int dq_ddim_step(const float* xt, const float* eps, float* xprev, float sa, float s1m, float sap, float s1mp,
                 int last, long n, void* stream);
/* pred_type "x0" reverse step (model.py:275-289): eps = (x_t - sa x0)/s1m, x_prev = last ? x0 : sap x0 + s1mp eps. */
int dq_ddim_step_x0(const float* xt, const float* x0_pred, float* xprev, float* eps_out, float sa, float s1m, float sap,
                    float s1mp, int last, long n, void* stream);
/* ODE sampler step (DDIM / DPM-Solver++(2M)): D = pred_x0 ? out : (x - sigma out)/alpha; last ? x_next = D (eps_out = eps)
 * : x_next = c_x x + c_d (w_cur D + w_prev d_hist), d_hist = D. */
int dq_dpm_step(const float* xt, const float* model_out, float* d_hist, float* x_next, float* eps_out, float alpha,
                float sigma, int pred_x0, float c_x, float c_d, float w_cur, float w_prev, int last, long n,
                void* stream);
/* out[i] = x[i] * scale1[0] (scale read on the device: upstream gradient of the fused MSE node, 1 / world-size). */
int dq_scale_by(const float* x, const float* scale1, float* out, long n, void* stream);
/* evaluation metric (model_interface.py:630-667 consumer): out3[s] += {<a_s, b_s>, |a_s|^2, |b_s|^2} per window s. */
int dq_cosine_sums(const float* a, const float* b, float* out3, long n_per_sample, int n_samples, void* stream);
/* validation scores of predicted maps against clean maps, both (n_windows, rt, mz) fp32: out9[w] = 9 float64 sums
 * {sum (p-g)^2, sum pg, sum p^2, sum g^2, sum_mz PG, sum_mz P^2, sum_mz G^2, sum_mz w r, sum_mz w} with P, G the RT-summed
 * spectra, r the Pearson correlation of a column over RT and w = G (0 for a truth column of zero variance).
 * partial: n_windows * dq_map_scores_nblk(mz) * 9 doubles of scratch.  No atomics: bit-identical per window in any batch. */
int dq_map_scores_nblk(int mz);
int dq_map_scores(const float* pred, const float* truth, double* partial, double* out9, int n_windows, int rt, int mz,
                  void* stream);
/* tail of sample(): model.py:319-322. */
int dq_sample_finalize(const float* x, const float* cond_n, float* xo, float* pn, long n, void* stream);
/* sum (eps-noise)^2 into a double accumulator and d_eps = gscale*(eps-noise): F.mse_loss model.py:361. */
int dq_mse(const float* eps, const float* noise, double* loss_sum, float* deps, float gscale, long n, void* stream);
int dq_add_inplace(float* a, const float* b, long n, void* stream);

/* ---- down/up path (model/unet1d.py) ------------------------------------------------------------------- */
/* Alignment: the tensor pointers of dq_conv1d_fwd, dq_resblock_fwd, dq_block_bwd, dq_conv1d_bwd_data/_weight,
 * dq_conv_bwd_fused, dq_conv_bwd_fused_res, dq_upconv_bwd_fused, dq_downconv_bwd_fused and dq_initconv_bwd need only
 * 4-byte alignment (a view that starts at any float of an allocation is accepted).  Their 16-byte vector / bulk-copy
 * paths are taken only when every pointer such a path touches is 16-byte aligned and the row length allows it; otherwise
 * a 4-byte path runs (or the call returns 1 and the documented composition applies). */
/* Fused Conv1d (+concat of two sources, ConditionalScaleShift on source 1, bias, RMSNorm, scale/shift, act,
 * residual): Block.forward 248-268, ResnetBlock 302-323, init_conv 1107-1117, Downsample 110, Upsample 93-96,
 * skip cats 1151/1154/1160, final_conv 1163, attn_cond_proj 976-978. */
int dq_conv1d_fwd(const float* x1, int c1, const float* x2, int c2, const float* in_ss, int in_ss_stride,
                  const float* w, const float* bias, int cout, int K, int stride, int pad, int up,
                  const float* g, const float* ss, int ss_stride, int act, const float* res,
                  float* u, float* y, int R, int Lin, int Lout, int rows_per_sample, void* stream);
/* Fused ResnetBlock forward (unet1d.py:302-323): Block1 (conv k3, RMSNorm, per-sample scale/shift, SiLU) -> Block2 (conv k3,
 * RMSNorm, SiLU) + skip (1x1 res_conv of the concat input, or identity) in one pass; u1 / h1 / u2 (saved for backward)
 * may be NULL.  Returns 1 (nothing launched) if the shape is not covered: compose from dq_conv1d_fwd instead. */
int dq_resblock_fwd(const float* x1, int c1, const float* x2, int c2, const float* w1, const float* b1, const float* g1,
                    const float* ss, int ss_stride, const float* w2, const float* b2, const float* g2, const float* wres,
                    const float* bres, float* u1, float* h1, float* u2, float* out, int cout, int R, int L,
                    int rows_per_sample, void* stream);
/* backward of the RMSNorm / scale-shift / activation epilogue of Block.forward 260-266. */
int dq_block_bwd(const float* dy, const float* u, const float* g, const float* ss, int ss_stride, int act,
                 float* du, float* dg, float* dss, int C, int R, int L, int rows_per_sample, void* stream);
int dq_conv1d_bwd_data(const float* du, const float* w, float* dx1, int c1, int acc1, float* dx2, int c2, int acc2,
                       int cout, int K, int stride, int pad, int up, int R, int Lin, int Lout, void* stream);
int dq_conv1d_bwd_weight(const float* du, const float* x1, int c1, const float* x2, int c2, const float* in_ss,
                         int in_ss_stride, float* dw, float* db, int cout, int K, int stride, int pad, int up,
                         int R, int Lin, int Lout, int rows_per_sample, void* stream);
/* Fused backward of a stride-1 Conv1d (K = 1 or 3, pad (K-1)/2) and, if u != NULL, of its Block epilogue
 * (unet1d.py:248-268, 302-323): one pass computes du, dx1/dx2 (+dadd, optional accumulate), dW, db, dg, d scale/shift. */
int dq_conv_bwd_fused(const float* dy, const float* u, const float* g, const float* ss, int ss_stride, int act,
                      const float* x1, int c1, const float* x2, int c2, const float* w, const float* dadd,
                      float* dx1, int acc1, float* dx2, int acc2, float* dw, float* db, float* dg, float* dss,
                      int cout, int K, int R, int L, int rows_per_sample, void* stream);
/* The backward of ResnetBlock.block1 (conv k3 + epilogue) AND of ResnetBlock.res_conv (1x1 conv over the same concat
 * input, unet1d.py:299, 322) in one pass: dx1/dx2 = conv3^T du + wres^T dyo, dW, db, dg, d scale/shift, dWres, dbres.
 * dyo = gradient of the block output (R, cout, L); wres (cout, c1+c2).  Returns 1 (nothing launched) if the shape is
 * not covered: run dq_conv_bwd_fused twice (K = 3, then K = 1 with acc) instead. */
int dq_conv_bwd_fused_res(const float* dy, const float* u, const float* g, const float* ss, int ss_stride, int act,
                          const float* x1, int c1, const float* x2, int c2, const float* w, float* dx1, float* dx2,
                          float* dw, float* db, float* dg, float* dss, const float* dyo, const float* wres,
                          float* dwres, float* dbres, int cout, int R, int L, int rows_per_sample, void* stream);
/* Re-indexing glue that lets the backward of Upsample (nearest x2 + Conv1d k3, unet1d.py:93-96) and Downsample
 * (Conv1d k4 s2 p1, unet1d.py:110) run through dq_conv_bwd_fused: y[2j] = y[2j+1] = x[j]; dx[j] (+)= d[2j] + d[2j+1];
 * space-to-depth x (R,C,L) -> (R,2C,L/2) [even samples | odd samples] and back; k4 weights (co,ci,4) <-> k3 weights
 * (co,2ci,3) (dir 0: pack, dir 1: w4 += unpack(w3)). */
int dq_upsample2x(const float* x, float* y, long n, void* stream);
/* Backward of Upsample = nearest x2 + Conv1d(k3, pad 1) (unet1d.py:93-96) in one pass: dy (R, cout, 2 Lh); x and dx
 * (R, cin, Lh) at half rate - the upsampled tensor and its gradient never exist; dw (cout, cin, 3) / db accumulated; dx
 * NULL = not needed, acc = accumulate into dx.  Returns 1 (nothing launched) if the shape is not covered: compose from
 * dq_upsample2x + dq_conv_bwd_fused + dq_fold2x instead. */
int dq_upconv_bwd_fused(const float* dy, const float* x, const float* w, float* dx, int acc, float* dw, float* db,
                        int cout, int cin, int R, int Lh, int rows_per_sample, void* stream);
int dq_fold2x(const float* d, float* dx, long n, int acc, void* stream);
/* Backward of Downsample = Conv1d(k4, stride 2, pad 1) (unet1d.py:110) in one pass: dy (R, cout, L / 2); x and dx
 * (R, cin, L); w / dw (cout, cin, 4); dw / db accumulated; dx NULL = not needed, acc = accumulate into dx.  Returns 1
 * (nothing launched) if the shape is not covered: compose from dq_s2d + dq_down_w + dq_conv_bwd_fused + dq_d2s instead. */
int dq_downconv_bwd_fused(const float* dy, const float* x, const float* w, float* dx, int acc, float* dw, float* db,
                          int cout, int cin, int R, int L, int rows_per_sample, void* stream);
int dq_s2d(const float* x, float* y, int R, int C, int L, void* stream);
int dq_d2s(const float* d, float* dx, int R, int C, int L, int acc, void* stream);
int dq_down_w(float* w4, float* w3, int co, int ci, int dir, void* stream);
/* Backward of init_conv = Conv1d(2 -> cout, k7, pad 3) over cat(ConditionalScaleShift(cond), x) (unet1d.py:1107-1117,
 * 677-678) in one pass: dW, db and the per-sample d scale / d shift (dss[s*ss_stride], [.. + 1]) from raw per-sample
 * correlations; no data gradient tensor.  scratch: (R / rows_per_sample, cout / 4, 88) floats zeroed by the caller.
 * Returns 1 (nothing launched) unless cout % 4 == 0, L % 4 == 0 and 16-byte aligned rows: then use
 * dq_conv1d_bwd_weight + dq_conv1d_bwd_data + dq_sample_dot. */
int dq_initconv_bwd(const float* d, const float* cond, const float* x, const float* ss, int ss_stride, const float* w,
                    float* dw, float* db, float* dss, float* scratch, int cout, int R, int L, int rows_per_sample,
                    void* stream);
/* gradient of ConditionalScaleShift (unet1d.py:677-678): per-sample sum d*c and sum d. */
int dq_sample_dot(const float* d, const float* c, float* dscale, float* dshift, int out_stride, long n_per_sample,
                  int n_samples, void* stream);
/* Residual(PreNorm(LinearAttention)): unet1d.py:473-496, 1017, 1068, restructured so that every per-head 32x32
 * contraction factors through the C input channels (csrc/linattn.cu).  CP = C rounded up to 8,
 * nchunk = dq_la_nchunk(L).  Scratch: part (R,nchunk,128,2+CP), dpart (R,nchunk,128,CP), hmat (R,128,CP),
 * sd (R,128), dxnq (R,C,L).  Saved by forward for backward: msm (R,128,2+CP) = [max, sum, Ms], gmat (R,C,128),
 * ypre (R,C,L). */
int dq_la_nchunk(int L);
/* Pipeline-timeout record of the tcgen05 LinearAttention kernels (csrc/linattn_tc.cu): returns 0 when clean, 1 when an
 * mbarrier wait timed out since the last call (out6 = 0x80000000 | wait code, blockIdx.x, blockIdx.y, threadIdx.x,
 * barrier address, parity); -1 on a CUDA error.  Synchronises with the device; reading clears the record. */
int dq_la_tc_last_error(unsigned int* out6);
int dq_linattn_fwd(const float* x, const float* g_pre, const float* wqkv, const float* wout, const float* bout,
                   const float* g_out, float* part, float* msm, float* gmat, float* ypre, float* out, int C, int R,
                   int L, void* stream);
int dq_linattn_bwd(const float* x, const float* dres, const float* ypre, const float* msm, const float* gmat,
                   const float* g_pre, const float* wqkv, const float* wout, const float* g_out, float* dxnq,
                   float* dpart, float* hmat, float* sd, float* dx, float* dwqkv, float* dwout, float* dbout,
                   float* dg_out, float* dg_pre, int C, int R, int L, void* stream);

/* ---- time embedding and per-sample linears (unet1d.py:211-218, 958-960, 292-296, 664, 535) ------------ */
int dq_time_embed(const long long* t, float* out, int b, int dim, float neg_e, void* stream);
int dq_linear_fwd(const float* x, const float* W, const float* bias, float* y, int rows, int in, int out, void* stream);
int dq_linear_bwd(const float* x, const float* W, const float* dy, float* dx, float* dW, float* db, int rows, int in,
                  int out, void* stream);
int dq_act_fwd(const float* x, float* y, int act, long n, void* stream);
int dq_act_bwd(const float* dy, const float* xpre, float* dx, int act, long n, void* stream);
int dq_ncl_nlc(const float* in, float* out, int B, int C, int L, int reverse, void* stream);

/* ---- mid stage (unet1d.py:1027-1058, 1144-1148; Attention 541-567; Attend 428-443) -------------------- */
/* tcgen05/TMEM/TMA multi-tap GEMM: C[M,N] (+)= sum_tap A_tap[M,K] . B_tap[N,K]^T (+bias); A, B bf16 K-major. */
int dq_gemm_bf16_tn(const void* A, long a_rows, long a_cols, long a_ld, const void* B, long b_rows, long b_cols,
                    long b_ld, long b_tap_stride, int b_ntaps, float* C, long ldc, const float* bias, int accumulate,
                    int M, int N, int K, int taps, const int* offs, int nz, int z_b_koff_step, int z_b_tap_step,
                    long z_c_stride, int bn, void* stream);
int dq_gemm_last_error(void);
/* -3: N odd; -4: x not 8-byte or out_bf16 not 4-byte aligned. */
int dq_mid_pack(const float* x, void* out_bf16, int b, int rt, int N, int pad, void* stream);
int dq_transpose_bf16(const void* in, void* out, int rows, int cols, long ld_out, int row_shift, void* stream);
int dq_cast_transpose(const float* in, void* out_bf16, void* out_t_bf16, int rows, int cols, void* stream);
int dq_rownorm_fwd(const float* u, int upad, const float* g, const float* ss, int ss_stride, int act, const float* res,
                   float* out_f32, void* out_bf16, int opad, float* inv_out, int b, int rt, int N, void* stream);
int dq_rownorm_bwd(const float* dh, int dhpad, const float* u, int upad, const float* g, const float* ss, int ss_stride,
                   int act, const float* inv, float* dot, void* du_bf16, int opad, float* du_f32, int du_acc, float* dg,
                   float* dss, float* dbias, int b, int rt, int N, void* stream);
int dq_colsum(const float* x, float* out, int rows, int cols, void* stream);
/* -2 (before any launch): the rt x rt tiles of one (sample, head) exceed the device's opt-in shared memory (sm_100a: rt > 196 forward, rt > 140 backward). */
int dq_attn_core_fwd(const float* qv, const float* k, const float* freqs, float* P, float* o_f32, void* o_bf16, int b,
                     int rt, void* stream);
int dq_attn_core_bwd(const float* qv, const float* k, const float* freqs, const float* P, const float* dO, float* dqv,
                     void* dqv_bf16, float* dk, int b, int rt, void* stream);

/* ---- optimizer (model/model_interface.py:1011, 1121-1122) --------------------------------------------- */
int dq_sumsq(const float* x, long n, double* out, void* stream);
int dq_clip_coef(const double* sumsq, float max_norm, float gscale, float* out_norm_coef, void* stream);
int dq_adamw(float* p, const float* g, float* m, float* v, long n, const float* coef_ptr, float lr, float b1, float b2,
             float eps, float wd, float step_size, float bc2_sqrt, void* stream);
/* dq_adamw, then ema = ema + ema_w (p_new - ema) in the same pass (ema_w = 1 - EMA decay of this update) */
int dq_adamw_ema(float* p, const float* g, float* m, float* v, float* ema, long n, const float* coef_ptr, float lr,
                 float b1, float b2, float eps, float wd, float step_size, float bc2_sqrt, float ema_w, void* stream);
/* exchange a[0:n) and b[0:n) in place */
int dq_swap(float* a, float* b, long n, void* stream);
int dq_fill(float* p, float v, long n, void* stream);

/* ---- data path (utils/data_loader.py:70-88; model_interface.py:1071-1075) ----------------------------- */
int dq_multiplex(const void* ms2, const void* ms1, int dtype, const long long* pairs, void* stats, float w0, float w1,
                 float* x0, float* other, float* cond, float* ms1_1, float* ms1_2, int items, long n2, int n1,
                 void* stream);

#ifdef __cplusplus
}
#endif
#endif
