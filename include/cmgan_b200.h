/* cmgan_b200 -- C ABI of the B200-native CMGAN hot path (libcmgan_b200.so).
 *
 * The reference (ruizhecao96/CMGAN) has no FFI layer: its boundary for this path is the nn.Module
 * interface (TSCNet.forward generator.py:174-196, Discriminator.forward discriminator.py:62-64,
 * power_compress / power_uncompress utils.py:20-39, torch.stft / torch.istft call sites
 * train.py:81-112).  These entry points are what a binding for that path calls; every function
 *   - takes raw DEVICE pointers, explicit sizes / strides (in elements) and a cudaStream_t (void*),
 *   - allocates nothing and never synchronises (re-entrant per stream, CUDA-graph capturable),
 *   - returns 0 on success, -1 on error with the message available from cmgan_last_error().
 * Activations are channel-last: row index (b*T + t)*F + f, channels contiguous.
 * One declaration per line (cmgan_b200/_lib.py parses this file to build the ctypes prototypes).
 */
#ifndef CMGAN_B200_H
#define CMGAN_B200_H
#include "../cmgan_b200/csrc/gemm_args.h"

#ifdef __cplusplus
extern "C" {
#endif

const char* cmgan_last_error(void);
int cmgan_abi_version(void);
int cmgan_gemm_args_size(void);
int cmgan_set_tf32_rounding(int on);

/* ---- dense contractions (replace nn.Linear / nn.Conv1d(k=1) / nn.Conv2d and their autograd; gemm_args.h) */
int cmgan_gemm_rows_f32(const CmganGemmArgs* a, void* stream);
int cmgan_gemm_wgrad_f32(const CmganGemmArgs* a, void* stream);
int cmgan_pack_weights(const CmganPackDesc* descs, int n, void* stream);
int cmgan_pack_weight(const float* src, float* dst, long long sb_tap, long long sb_k, long long sb_n, int Cin, int ntaps, int N, void* stream);

/* ---- fused macaron feed-forward (conformer.py:54-72,136-148,211-212): LN -> 64x256 -> Swish, dropout -> 256x64 -> dropout, alpha, residual in ONE tcgen05 kernel */
int cmgan_ffn_fwd(const float* x, long long ldx, long long M, const float* ln_g, const float* ln_b, const float* W1p, const float* b1, const float* W2p, const float* b2, float alpha, unsigned long long seed1, unsigned long long seed2, unsigned int thr, float inv_keep, const unsigned long long* seed_dev, float* out, long long ldo, void* stream);

int cmgan_ffn_debug_timeline(long long* buf);
int cmgan_ffn_bwd(const float* x, long long ldx, const float* dz, long long lddz, const float* dout, long long lddo, const float* res2, long long ldr2, long long M, const float* ln_g, const float* ln_b, const float* W1p, const float* b1, const float* W2tp, const float* W1tp, unsigned long long seed1, unsigned int thr, float inv_keep, const unsigned long long* seed_dev, float* dx, long long lddx, float* a_out, float* dh_out, float* xn_out, float* dgamma, float* dbeta, void* stream);

/* ---- LayerNorm (conformer.py:68,161,214), InstanceNorm2d (generator.py:35,55,61,128,148), BatchNorm1d (conformer.py:169) */
int cmgan_ln_stats(const float* x, long long ldx, long long M, float* stats, void* stream);
int cmgan_ln_apply(const float* x, long long ldx, long long M, const float* gamma, const float* beta, const float* res, long long ldr, float* y, long long ldy, float* stats, int round_tf32, void* stream);
int cmgan_ln_bwd(const float* dy, long long lddy, const float* x, long long ldx, const float* stats, const float* gamma, long long M, const float* res, long long ldr, const float* res2, long long ldr2, float* dx, long long lddx, float* dgamma, float* dbeta, void* stream);
int cmgan_ln_bwd_drop(const float* dy, long long lddy, const float* x, long long ldx, const float* stats, const float* gamma, long long M, const float* res, long long ldr, const float* res2, long long ldr2, float* dx, long long lddx, float* dgamma, float* dbeta, float* dz, long long lddz, float alpha, unsigned long long seed, unsigned int thr, float inv_keep, const unsigned long long* seed_dev, void* stream);
int cmgan_norm_stats(const float* x, long long ldx, int G, long long rows_per_group, int C, double* sums, void* stream);
int cmgan_norm_finalize(const double* sums, long long n, int G, int C, int mode, const float* gamma, const float* beta, float* running_mean, float* running_var, float momentum, float* scale, float* shift, float* mean_out, float* rstd_out, long long tstride, void* stream);
int cmgan_norm_stats_varlen(const float* x, long long ldx, int G, long long rows_per_group, int C, const int* frames, long long rows_per_frame, double* sums, void* stream);
int cmgan_norm_finalize_varlen(const double* sums, const int* frames, long long rows_per_frame, int T, int G, int C, const float* gamma, const float* beta, float* scale, float* shift, float* mean_out, float* rstd_out, long long tstride, void* stream);
int cmgan_norm_bwd_reduce(const float* x, long long ldx, const float* dact, long long ldd, int G, long long rows_per_group, int C, int act, const float* scale, const float* shift, const float* mean, const float* rstd, long long tstride, const float* slope, double* S, float* dslope, void* stream);
int cmgan_norm_bwd_apply(const float* x, long long ldx, const float* dact, long long ldd, int G, long long rows_per_group, int C, int act, int use_batch_stats, const float* scale, const float* shift, const float* mean, const float* rstd, long long tstride, const float* slope, const double* S, float* dx, long long lddx, float* dgamma, float* dbeta, void* stream);
int cmgan_norm_apply(const float* x, long long ldx, int G, long long rows_per_group, int C, int act, const float* scale, const float* shift, long long tstride, const float* slope, float* y, long long ldy, void* stream);
int cmgan_fill(float* p, long long n, float v, void* stream);
int cmgan_copy_rows(const float* src, long long lds, float* dst, long long ldd, long long M, int C, void* stream);
int cmgan_copy_rows_operand(const float* src, long long lds, float* dst, long long ldd, long long M, int C, void* stream);
int cmgan_add_rows(const float* src, long long lds, float* dst, long long ldd, long long M, int C, void* stream);

/* ---- attention with Shaw relative positions (conformer.py:100-131); axis 0 = time sequences, 1 = frequency sequences.
 * *_varlen (here and below): ragged batch of B items padded to T frames, frames = device int[B], 1 <= frames[b] <= T; rows of padded frames are
 * never read (they may hold NaN) and their outputs are unspecified. */
int cmgan_attention_fwd(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, void* stream);
int cmgan_attention_fwd_tf32(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, void* stream);
int cmgan_attention_fwd_tf32_nbuf(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, int nbuf, void* stream);
int cmgan_attention_fwd_varlen(const float* qkv, const float* E, int B, int T, int F, int axis, const int* frames, float* ctx, float* lse, void* stream);
int cmgan_attention_fwd_tf32_varlen(const float* qkv, const float* E, int B, int T, int F, int axis, const int* frames, float* ctx, float* lse, void* stream);
int cmgan_attention_fwd_tc(const float* qkv, const float* E, int B, int T, int F, int axis, float* ctx, float* lse, void* stream);
int cmgan_attention_bwd(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B, int T, int F, int axis, float* delta, float* dqkv, float* dE, void* stream);
int cmgan_attention_bwd_tf32_parts(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B, int T, int F, int axis, float* delta, float* dqkv, float* dE, int parts, void* stream);
long long cmgan_attention_bwd_ws_floats(int B, int T, int F, int axis);
int cmgan_attention_bwd_tf32_ws(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B, int T, int F, int axis, float* delta, float* dqkv, float* dE, int parts, float* scratch, long long scratch_floats, void* stream);
int cmgan_attention_bwd_tf32(const float* qkv, const float* E, const float* ctx, const float* dctx, const float* lse, int B, int T, int F, int axis, float* delta, float* dqkv, float* dE, void* stream);

/* ---- GLU + depthwise conv k=31 (conformer.py:30-48,164-168) */
int cmgan_glu_dwconv_fwd(const float* g, const float* w, const float* bias, int B, int T, int F, int axis, float* out, double* bn_sums, void* stream);
int cmgan_glu_dwconv_fwd_varlen(const float* g, const float* w, const float* bias, int B, int T, int F, int axis, const int* frames, float* out, void* stream);
int cmgan_glu_dwconv_bwd(const float* g, const float* dz, const float* w, int B, int T, int F, int axis, float* dg, float* dw, float* dbias, void* stream);

/* ---- signal front / back end (train.py:75-112, evaluation.py:21-51, utils.py:20-39) */
int cmgan_rms_scale(const float* x, long long ldx, int B, int L, float* c, void* stream);
int cmgan_pad_reflect(const float* x, long long ldx, int B, int L, const float* c, float* xp, int Lp, void* stream);
int cmgan_rms_scale_varlen(const float* x, long long ldx, int B, const int* lens, float* c, void* stream);
int cmgan_wrap_pad_reflect_varlen(const float* x, long long ldx, int B, const int* lens, const float* c, float* xp, int Lp, void* stream);
int cmgan_compress(const float* S, int B, int T, float* X, void* stream);
int cmgan_uncompress(const float* re, const float* im, long long sb, long long st, long long sf, int B, int T, float* U, void* stream);
int cmgan_uncompress_bwd(const float* re, const float* im, long long sb, long long st, long long sf, int B, int T, const float* dU, float* dre, float* dim_, int accumulate, void* stream);
int cmgan_power_law(const float* re, const float* im, long long i0, long long i1, long long i2, float* ore, float* oim, long long o0, long long o1, long long o2, int d0, int d1, int d2, float p, void* stream);
int cmgan_power_law_bwd(const float* re, const float* im, long long i0, long long i1, long long i2, const float* gre, const float* gim, long long o0, long long o1, long long o2, float* dre, float* dim_, long long q0, long long q1, long long q2, int d0, int d1, int d2, float p, void* stream);
int cmgan_ola(const float* frames, int B, int T, const float* inv_env, const float* c_div, float* y, long long ldy, void* stream);
int cmgan_ola_varlen(const float* frames, int B, int T, const int* nframes, const double* win_sq, const float* c_div, float* y, long long ldy, void* stream);
int cmgan_ola_bwd(const float* dy, long long lddy, int B, int T, const float* inv_env, float* dframes, void* stream);

/* ---- generator head and tails (generator.py:53,126,136-139,150,175-196) */
int cmgan_head_conv(const float* x, long long sb, long long sc, long long st, long long sf, int B, int T, int F, const float* w, const float* bias, float* out, long long ldo, void* stream);
int cmgan_head_conv_wgrad(const float* x, long long sb, long long sc, long long st, long long sf, int B, int T, int F, const float* draw, long long ldd, float* dw, float* db, void* stream);
int cmgan_rowdot_fwd(const float* in, int B, int T, int Fout, int nout, const float* scale, const float* shift, const float* slope, const float* w, const float* bias, float* out, void* stream);
int cmgan_rowdot_bwd(const float* in, int B, int T, int Fout, int nout, const float* scale, const float* shift, const float* slope, const float* w, const float* dout, float* dact, float* dw, float* dbias, void* stream);
int cmgan_recombine(const float* m1, const float* in_scale, const float* in_shift, const float* a1, const float* fcw, const float* fcb, const float* slope_f, const float* x, long long sb, long long sc, long long st, long long sf, const float* cplx, int B, int T, int F, float* fr, float* fi, void* stream);
int cmgan_recombine_bwd(const float* m1, const float* in_scale, const float* in_shift, const float* a1, const float* fcw, const float* fcb, const float* slope_f, const float* x, long long sb, long long sc, long long st, long long sf, const float* dfr, const float* dfi, long long gb, long long gt, long long gf, int B, int T, int F, float* dcplx, float* dz, float* dslope_f, float* dfcw, float* dfcb, void* stream);

/* ---- discriminator-only pieces (discriminator.py:29-64, utils.py:42-50) and dropout-mask export */
int cmgan_dropout_mask(float* out, long long n, unsigned long long seed, unsigned int thr, void* stream);
int cmgan_stack2(const float* x, long long xb, long long xh, long long xw, const float* y, long long yb, long long yh, long long yw, int B, int H, int W, float* out, void* stream);
int cmgan_unstack2(const float* dxy, long long n, float* dx, float* dy, void* stream);
int cmgan_spectral_norm(const float* W, int R, int Cc, float* u, float* v, int training, float* w_sn, float* sigma, float* uv_out, void* stream);
int cmgan_spectral_norm_bwd(const float* w_sn, const float* dw_sn, int R, int Cc, const float* u, const float* v, const float* sigma, float* dW, void* stream);
int cmgan_norm_maxpool(const float* x, int B, long long rows, int C, const float* scale, const float* shift, const float* slope, float* out, int* arg, void* stream);
int cmgan_maxpool_bwd(const float* dout, const int* arg, int B, long long rows, int C, float* dact, void* stream);
int cmgan_drop_prelu(const float* x, long long n, int C, const float* slope, unsigned long long seed, unsigned int thr, float inv_keep, float* y, const unsigned long long* seed_dev, void* stream);
int cmgan_drop_prelu_bwd(const float* x, const float* dy, long long n, int C, const float* slope, unsigned long long seed, unsigned int thr, float inv_keep, float* dx, float* dslope, const unsigned long long* seed_dev, void* stream);
int cmgan_lsigmoid(const float* x, long long n, const float* slope, float* y, void* stream);
int cmgan_lsigmoid_bwd(const float* x, const float* y, const float* dy, long long n, const float* slope, float* dx, float* dslope, void* stream);

/* ---- losses with fused gradients (train.py:124-174) and flat AdamW (train.py:63-66) */
int cmgan_spec_loss(const float* er, const float* ei, const float* cr, const float* ci, long long per, long long cb, long long n, float w_ri, float w_mag, double* acc, float* d_er, float* d_ei, float* est_mag, float* clean_mag, void* stream);
int cmgan_time_loss(const float* ea, long long lde, const float* clean, long long ldc, int B, int L, float w_t, double* acc, float* d_ea, void* stream);
int cmgan_gen_loss_finalize(const double* acc, double n_spec, double n_time, float w_ri, float w_mag, float w_t, float w_gan, const float* fake, int B, float* loss, float* d_fake, void* stream);
int cmgan_disc_loss(const float* d_max, const float* d_enh, const float* target, int B, float* loss, float* g_max, float* g_enh, void* stream);
int cmgan_mag_bwd_add(const float* er, const float* ei, const float* d_mag, long long gb, long long gt, long long gf, int B, int T, int F, float* d_er, float* d_ei, void* stream);
int cmgan_adamw(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2, float eps, float wd, int step, const unsigned long long* step_dev, const float* lr_dev, void* stream);
int cmgan_counter_add(unsigned long long* p, unsigned long long v, void* stream);

/* ---- PESQ-free scoring on the GPU (src/tools/compute_metrics.py: segmental SNR :350-397, STOI :400-471, LLR :277-347, WSS :80-274), float64 like the numpy reference */
int cmgan_ssnr_f64(const double* clean, const double* proc, long long L, int W, int skip, int nfr, double* out, void* stream);
long long cmgan_stoi_scratch_doubles(long long L);
int cmgan_llr_f64(const double* clean, const double* proc, long long L, int W, int skip, int order, int nfr, double* out, void* stream);
int cmgan_wss_f64(const double* clean, const double* proc, long long L, int W, int skip, int nfft, const double* filt, int nfr, double* out, void* stream);
int cmgan_stoi_f64(const double* clean, const double* proc, long long L, const double* h, const int* band_lo, const int* band_hi, double* scratch, double* out, void* stream);

/* ---- module level: TSCNet.forward, inference mode (generator.py:160-196; eval BatchNorm, no dropout) as one call.
 * params = every floating-point state_dict tensor of the reference TSCNet(64, 201) in state_dict order, each starting at a multiple of 4
 * floats (cmgan_tscnet_param_info enumerates key / offset / numel; cmgan_tscnet_param_floats = size of the block).  x is (B, 2, T, F) with
 * element strides (the reference passes a permuted view, train.py:95); outputs are contiguous (B, 1, T, F).  The workspace is caller-owned,
 * 256-byte aligned, at least cmgan_tscnet_workspace_bytes(B, T, F, precision) bytes; precision 0 = exact fp32, 1 = tf32 tensor cores.
 * cmgan_tscnet_fwd_varlen: ragged batch of utterances padded to T frames, frames = device int[B] with 1 <= frames[b] <= T; rows t < frames[b]
 * equal cmgan_tscnet_fwd on x[b, :, :frames[b]] alone, rows beyond are unspecified; frames == NULL is cmgan_tscnet_fwd; same workspace. */
int cmgan_tscnet_param_count(void);
long long cmgan_tscnet_param_floats(void);
int cmgan_tscnet_param_info(int index, const char** key, long long* offset, long long* numel);
long long cmgan_tscnet_workspace_bytes(int B, int T, int F, int precision);
int cmgan_tscnet_fwd_varlen(const float* params, const float* x, long long sxb, long long sxc, long long sxt, long long sxf, int B, int T, int F, const int* frames, float* final_real, float* final_imag, void* workspace, long long workspace_bytes, int precision, void* stream);
int cmgan_tscnet_fwd(const float* params, const float* x, long long sxb, long long sxc, long long sxt, long long sxf, int B, int T, int F, float* final_real, float* final_imag, void* workspace, long long workspace_bytes, int precision, void* stream);

#ifdef __cplusplus
}
#endif
#endif
