/*
 * adm_b200.h — C ABI of libadm_b200.so: the sm_100a kernels behind the DDM-const training step and sampler.
 *
 * This is the drop-in boundary for the hot path of zacz08/ADM.  The reference has no FFI of its own for this path
 * (every op goes through torch.nn.functional -> ATen); its only native-op precedent is
 * unet/op/upfirdn2d.cpp:8-19 + unet/op/upfirdn2d.py:10-16 (a torch extension taking tensors, launched on the current
 * stream).  We keep that contract — enqueue on the caller's stream, never synchronise, never allocate — but with a plain
 * C signature: raw device pointers, sizes, a cudaStream_t passed as void*.  Each entry point below cites the reference
 * code it replaces.  All functions return 0 on success or a negative ADM_ERR_* code; adm_last_error() returns the
 * message.  There is no CPU path: every pointer must be a CUDA device pointer.
 *
 * Internal activation layout: NHWC bf16 ("pixel-major"): element (n,h,w,c) at ((n*H+h)*W+w)*ld + c, ld >= C, ld % 8 == 0.
 * Reference layout at the API edge: NCHW fp32 contiguous (unet/uncond_unet.py:616).
 */
#ifndef ADM_B200_H
#define ADM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define ADM_OK 0
#define ADM_ERR_SHAPE (-1) /* unsupported / inconsistent shape */
#define ADM_ERR_DTYPE (-2) /* unsupported dtype or architecture */
#define ADM_ERR_CUDA (-3)  /* CUDA runtime / driver error */

/* ---------------------------------------------------------------- library */
const char* adm_last_error(void);      /* message of the last failing call on this thread */
int adm_device_error(void);            /* nonzero if a kernel hit its deadlock guard (device-side flag) */
long long adm_launch_count(void);      /* number of kernels this library has launched in this process */
int adm_version(void);

/* ---------------------------------------------------------------- DDM elementwise (fp32 / fp64, NCHW)
 * K1  q_sample, ddm/ddm_const.py:284-287 with C = -x0 (:319):  x_t = x0 - t*x0 + sqrt(t)*noise
 *     x0, noise, x_t: [B, chw] fp32; t: [B] fp32.                                                        */
int adm_qsample(const float* x0, const float* noise, const float* t, float* x_t, long long batch, long long chw,
                void* stream);

/* K2  C/eps regression loss, forward + backward in one pass.  ddm/ddm_const.py:335-344,358 + ddm/loss.py:300-312
 *     (MSE_Loss reduction='sum' over CHW): loss_b = w1_b*SSE(C_pred, -x0) + w2_b*SSE(eps_pred, noise)
 *     [+ use_l1: w*mean|.| terms and /2, ddm_const.py:345-348],  w1 = (t^2-t+1)/t, w2 = (t^2-t+1)/(1-t+eps) when
 *     weighting != 0 else 1.  Writes per-sample loss [B] (caller sums / B) and, if non-null, the gradients of
 *     (sum_b loss_b)/B * grad_scale w.r.t. C_pred and eps_pred.
 *     use_l1 is a flag word: 1 = + w*mean|.| then /2 (image space, ddm_const.py:345-348); 2 = + w*sum|.| then /2
 *     (latent, ddm_const_2.py:561-564); 4 = + the latent reconstruction term W * sum|x_rec - x0| (ddm_const_2.py:565-568;
 *     the reference's [B] x [B,1] broadcast sums an outer product, i.e. every sample is weighted by
 *     W = sum_j -log(t_j)/2), in which case loss_per_sample has 2*B entries: [total | that term].           */
int adm_ddm_loss(const float* c_pred, const float* eps_pred, const float* x0, const float* noise, const float* t,
                 float eps, int weighting, int use_l1, float grad_scale, float* loss_per_sample, float* d_c_pred,
                 float* d_eps_pred, long long batch, long long chw, void* stream);

/* K3  deterministic sampler update, ddm/ddm_const.py:452-455 (and final :471-476 when last != 0):
 *     x0 = x - C*t_cur - eps*sqrt(t_cur); clamp(+-clip); x' = x0 + C*t_next + eps*sqrt(t_next)
 *     last != 0: x' = (clamp(x', +-clip)/scale_input + 1)/2.   State is fp64 (state_f64 != 0) or fp32.   */
int adm_sampler_step(const void* x, const float* c_pred, const float* eps_pred, void* x_next, double t_cur,
                     double t_next, double clip, int do_clip, int last, double scale_input, int state_f64,
                     long long numel, void* stream);
/*     stochastic variant, ddm/ddm_const.py:404-413 + :296-303: x0 -> clamp -> C=-x0;
 *     mean = x + C*(t-s) - C*t - s/sqrt(t)*eps; x' = mean + sqrt(s*(t-s)/t) * z                            */
int adm_sampler_step_stochastic(const float* x, const float* c_pred, const float* eps_pred, const float* z,
                                float* x_next, double t_cur, double s, double clip, int do_clip, long long numel,
                                void* stream);

/* ---------------------------------------------------------------- EDM preconditioning edges
 * unet/uncond_unet.py:616-628: x_in = c_in(sigma_b) * x, NCHW fp32 -> NHWC bf16 with ld_out channels (zero padded). */
int adm_unet_input(const float* x_nchw, const float* sigma, int sigma_is_scalar, void* x_nhwc, int n, int c, int h,
                   int w, int ld_out, void* stream);
/* unet/uncond_unet.py:621-624,631-632: D1 = c_skip1*x + c_out1*F1, D2 = c_skip2*x + c_out2*F2.
 * F1/F2: NHWC fp32 [pixels][ldf]; x, D1, D2: NCHW fp32.                                                    */
int adm_unet_output(const float* f1, const float* f2, int ldf, const float* x_nchw, const float* sigma,
                    int sigma_is_scalar, float* d1, float* d2, int n, int c, int h, int w, void* stream);
/* backward of the above w.r.t. F: dF = c_out * dD, NCHW fp32 -> NHWC bf16 [pixels][ld_out] (zero padded). */
int adm_unet_output_bwd(const float* dd1, const float* dd2, const float* sigma, void* df1, void* df2, int n, int c,
                        int h, int w, int ld_out, void* stream);

/* ---------------------------------------------------------------- tcgen05 GEMM engine
 * conv3x3 / conv1x1 forward as implicit GEMM (replaces F.conv2d at unet/uncond_unet.py:100,110 and nn.Conv2d in
 * decouple1/2 :500-507).  x1 (and optionally x2: fused channel concat, :570-571) NHWC bf16; wpk = packed weights
 * bf16 [nout][ntaps][pad64(c1)+pad64(c2)] (adm_pack_conv_weight); out [n*h*w][ldc] bf16 (out_mode 0) / fp32 (1);
 * epilogue: out = alpha*acc + bias[col] + residual[row][col].  ntaps = k*k for a square odd kernel with 'same'
 * padding k/2: 1, 9, 25 or 49 (the 7x7 stem of the conditional UNet, unet/cond_unet.py:656); the same values are
 * accepted by adm_conv_dgrad and adm_conv_wgrad.                                                           */
int adm_conv_fprop(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int h, int w,
                   const void* wpk, int nout, int ntaps, void* out, int out_mode, long long ldc, const float* bias,
                   const void* residual, long long ldr, float alpha, void* stream);
/* data gradient: dx[pix][0:n_valid] = alpha * conv^T(dy) + residual, reading the SAME packed weights through a
 * (Cin, tap, Cout) view with reversed taps; kpad = padded input channels of the forward conv.              */
int adm_conv_dgrad(const void* dy, int cout, long long ld_dy, int n, int h, int w, const void* wpk, int kpad,
                   int ntaps, void* dx, int n_valid, long long ldc, const void* residual, long long ldr, float alpha,
                   void* stream);
/* weight gradient, accumulated (atomic fp32) into dw [cout][ntaps][kpad] (packed layout, zero it first). */
int adm_conv_wgrad(const void* dy, int cout, long long ld_dy, const void* x1, int c1, long long ld1, const void* x2,
                   int c2, long long ld2, int n, int h, int w, int ntaps, float* dw, void* stream);
/* same, 1x1 convs only, with an output row map: the gradient of GEMM row r (output channel r of the conv as it is
 * executed) is accumulated into dw row row_map[r] — lets the qkv projection, executed in (q | k | v) x head x d row order,
 * write its weight gradient straight into the reference-ordered gradient (unet/uncond_unet.py:205).           */
int adm_conv_wgrad_mapped(const void* dy, int cout, long long ld_dy, const void* x1, int c1, long long ld1,
                          const void* x2, int c2, long long ld2, int n, int h, int w, int ntaps, const int* row_map,
                          float* dw, void* stream);

/* Generic batched GEMM C[b] = alpha * A[b] * B[b]^T (+bias, +residual) on 3-D bf16 tensor views.  Used for Linear
 * (unet/uncond_unet.py:62-66), and the attention products (:207-208).  An operand is K-major (dim0 = K) or MN-major
 * (dim0 = M or N); batch bt splits into b_hi = bt / bdiv, b_lo = bt % bdiv and each operand's start coordinate is
 * (c0 + b_lo*c0_lo, c1 + b_lo*c1_lo, b_hi*bhi + b_lo*blo).                                                 */
typedef struct adm_operand {
    const void* ptr;
    int mn_major;
    long long dim0, dim1, dim2;  /* extents, innermost first */
    long long stride1, stride2;  /* element strides of dim1, dim2 */
    int c0, c0_lo, c1, c1_lo, bhi, blo;
} adm_operand;
typedef struct adm_gemm_desc {
    adm_operand a, b;
    int m, n, k;        /* per-batch problem */
    int batches, bdiv;
    int splits;         /* split-K factor (needs out_mode 2) */
    void* c;
    int out_mode;       /* 0 bf16, 1 fp32, 2 fp32 atomic accumulate */
    long long ldc, c_bhi, c_blo;
    int c_col_lo;
    const float* bias;
    const void* residual;
    long long ldr;
    float alpha;
} adm_gemm_desc;
int adm_gemm_batched(const adm_gemm_desc* desc, void* stream);

/* ---------------------------------------------------------------- AugmentPipe geometric warp (SURVEY 8 row f-4)
 * ddm/augment.py AugmentPipe.__call__ :153-328 as ddm_const.py:179-180 configures it (flips + one anti-aliased affine
 * warp): x, y fp32 NCHW [n][c][h][w] (c <= 4); flips int [n][2] = (flip x, flip y); theta fp32 [n][6] = the 2 x 3 matrix
 * the reference hands to affine_grid (:265-267, after its margin / upsampling / normalisation compositions); mx0, mx1,
 * my0, my1 = the batch-wide reflect-padding margins (:245-250).  Four CTAs (row bands) per sample; padded and upsampled images are
 * never materialised.  adm_augment_warp_smem: dynamic shared memory the kernel needs (<= 200 KB).             */
long long adm_augment_warp_smem(int c, int h, int w);
int adm_augment_warp(const float* x, float* y, const float* theta, const int* flips, int n, int c, int h, int w,
                     int mx0, int mx1, int my0, int my1, void* stream);

/* ---------------------------------------------------------------- weight packing (derived bf16 caches of the fp32 masters)
 * w fp32 [cout][c1+c2][k][k] (reference layout, unet/uncond_unet.py:85) -> bf16 [cout][k*k][pad64(c1)+pad64(c2)] */
int adm_pack_conv_weight(const float* w, void* wpk, int cout, int c1, int c2, int ksize, const int* row_perm,
                         void* stream);
/*   row_perm (optional, device int[cout]): packed row r holds reference row row_perm[r] — used to store the qkv
 *   projection as (q | k | v) x heads x d instead of the reference's interleaved (head, d, {q,k,v}) order (:205). */
/* inverse for gradients: packed fp32 [cout][k*k][kpad] -> reference layout fp32 [cout][c1+c2][k][k] (overwrite
 * when accumulate == 0, add otherwise)                                                                    */
int adm_unpack_conv_wgrad(const float* dw_packed, float* dw, int cout, int c1, int c2, int ksize, int accumulate,
                          const int* row_perm, void* stream);
int adm_cast_f32_bf16(const float* src, void* dst, long long numel, void* stream);
/* dgrad shadow: batched 64 x 64 tile transpose of packed bf16 weights, [cout][tap][cin] -> [cin][ntaps-1-tap][cout]
 * (the flipped, transposed kernel of conv2d's data gradient — what autograd derives for F.conv2d,
 * unet/uncond_unet.py:100,110), so the data gradient runs through adm_conv_fprop.  tiles: device array of
 * num_tiles x {src offset, dst offset, src row stride, dst row stride} (elements, all multiples of 8); one launch
 * covers every conv of a parameter arena.                                                                    */
int adm_transpose_weight_tiles(const void* src, void* dst, const long long* tiles, int num_tiles, void* stream);
/* batched row gather: for i < n_rows copy row_bytes bytes from src + table[2i] to dst + table[2i+1] (byte offsets,
 * multiples of 4; of 16 when row_bytes is).  One launch per optimizer step re-derives every operand that is a row
 * permutation of arena-resident parameters (the qkv projections in (q | k | v) x head x d row order).        */
int adm_gather_rows(const void* src, void* dst, const long long* table, long long n_rows, int row_bytes,
                    void* stream);

/* ---------------------------------------------------------------- GroupNorm family (NHWC bf16, HBM-bound)
 * Replaces torch.nn.functional.group_norm (unet/uncond_unet.py:128) and the elementwise chain around it in
 * UNetBlock.forward (:191, :193-196, :200): silu, addcmul(shift, norm, scale+1), dropout, plus the depthwise 2x2
 * resample of Conv2d.forward (:105-108) when it directly follows.  x1 (+ optional x2 = fused torch.cat, :570-571).
                                                                                                              */
/* seed_counter (adm_gn_apply / adm_gn_forward / adm_gn_bwd): optional device-resident u64 step counter mixed into the
 * dropout seed, so that a captured CUDA graph draws fresh masks per replay.  It is passed per call (no process-global
 * state), dereferenced only when drop_p > 0, and may be NULL. */
int adm_gn_stats(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int hw,
                 int groups, float eps, const float* gamma, const float* beta, const float* params,
                 long long ld_params, float* work, float* coef, void* stream);
/*   Pass 1: per-(sample, channel) sum / sum of squares, then the coefficient table coef[n][c] = {A, B, mean, rstd}
 *   (fp32 x4) with GN(x)[*(1+scale)+shift] = x*A + B; params = [n][ld_params] holding (scale | shift) or NULL.
 *   work: fp32 scratch of 2*n*C + n elements (zeroed by the call).                                             */
/* y = act(x*A + B); act 1 = SiLU; drop_p > 0 applies Philox dropout keyed by seed; resample 0 none / 1 2x2 average /
 * 2 nearest x2.                                                                                              */
int adm_gn_apply(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int h, int w,
                 const float* coef, int act, float drop_p, unsigned long long seed,
                 const unsigned long long* seed_counter, int resample, void* out, long long ldo, void* stream);
/* Backward of gn_stats + gn_apply.  dy: gradient at the op's output (its resolution).  Accumulates dgamma/dbeta (+=,
 * atomics), writes dparams [n][ld_dparams] = (dscale | dshift), and dx1/dx2 (+ `add`, a skip-path gradient over the
 * full channel range: add_mode 0 same resolution, 1 half resolution spread /4, 2 double resolution summed 2x2).
 * work: fp32 scratch 2*n*C + n; bcoef: fp32 scratch 4*n*C.  dgamma == NULL skips the parameter gradients,
 * dx1 == NULL skips the data gradient.                                                                       */
int adm_gn_bwd(const void* dy, long long ldy, const void* x1, int c1, long long ld1, const void* x2, int c2,
               long long ld2, int n, int h, int w, int groups, const float* coef, const float* gamma,
               const float* beta, const float* params, long long ld_params, int act, float drop_p,
               unsigned long long seed, const unsigned long long* seed_counter, int resample, float* work,
               float* bcoef, float* dgamma, float* dbeta, float* dparams, long long ld_dparams, const void* add,
               long long ldadd, int add_mode, void* dx1, long long ldx1, void* dx2, long long ldx2, float* dbias1,
               float* dbias1b, int dy_scratch, void* stream);
/*   dy_scratch != 0: the caller is done with dy — the kernel may overwrite it (it keeps the gradient at the
 *   pre-activation there between its two passes instead of recomputing SiLU' and the dropout mask).          */
/*   dbias1, dbias1b (optional, fp32 [c1]): += column sums of dx1 — the bias gradient of the conv(s) that produced x1
 *   (conv1 and the 1x1 skip of a UNetBlock share it; unet/uncond_unet.py:111-112 backward), so no separate pass
 *   over dx1 is needed.
 * adm_gn_forward = gn_stats + gn_apply in one call.  When the batch fills the SMs it runs ONE kernel with a
 * thread-block cluster per sample (statistics exchanged through distributed shared memory, apply pass re-reading the
 * sample from L2); adm_gn_bwd does the same for the backward pair.                                            */
int adm_gn_forward(const void* x1, int c1, long long ld1, const void* x2, int c2, long long ld2, int n, int h, int w,
                   int groups, float eps, const float* gamma, const float* beta, const float* params,
                   long long ld_params, float* work, float* coef, int act, float drop_p, unsigned long long seed,
                   const unsigned long long* seed_counter, int resample, void* out, long long ldo, void* stream);
/* out[c] += sum_rows x[row][c] (bias gradients, unet/uncond_unet.py:111-112 backward). */
int adm_col_sums(const void* x, long long ld, long long rows, int c, float* out, void* stream);
/* out[out_map[c]] += sum_rows x[row][c] (out_map: device int[c], or NULL = identity) */
int adm_col_sums_mapped(const void* x, long long ld, long long rows, int c, float* out, const int* out_map,
                        void* stream);
/* out = a + b (+ c): gradient fan-in of the skip connections (torch autograd's implicit adds, unet/uncond_unet.py:563-564) */
int adm_add_bf16(const void* a, long long lda, const void* b, long long ldb, const void* c, long long ldc, void* out,
                 long long ldo, long long rows, int ch, void* stream);
/* skip-path resample of Conv2d(kernel=0, up/down) (unet/uncond_unet.py:181-182,105-108): mode 1 avg 2x2, 2 nearest x2 */
int adm_resample(const void* x, long long ldx, int n, int h, int w, int c, int mode, void* out, long long ldo,
                 void* stream);
/* silu of the embedding MLP (unet/uncond_unet.py:549,556): y fp32 and/or bf16 copies (either may be NULL) */
int adm_silu(const float* x, float* y, void* y_bf16, long long numel, void* stream);
int adm_silu_bwd(const float* x, const float* dy, float* dx, void* dx_bf16, long long numel, void* stream);

/* ---------------------------------------------------------------- attention pieces
 * softmax over the key axis of S = Q^T K / sqrt(d) (unet/uncond_unet.py:207); P bf16 [rows][len].  Forward: any len
 * <= 1024 (one warp per row) or a multiple of 4 up to 65536 (one CTA per row: the autoencoder's single-head mid
 * attention, ddm/encoder_decoder.py:204-209); backward len <= 1024: dS = scale * P * (dP - sum_j dP_j P_j).                                                       */
int adm_softmax_fwd(const float* s, void* p, long long rows, int len, void* stream);
int adm_softmax_bwd(const void* p, const float* dp, void* ds, float scale, long long rows, int len, void* stream);
/* K9 forward, fused (unet/uncond_unet.py:204-208; cond_unet.Attention, unet/cond_unet.py:533-555 with zero-padded heads):
 * persistent CTAs walk (sample, head) units; S = Q K^T lives in TMEM, the softmax runs in registers, P is written back
 * to TMEM as bf16 and consumed from there as the A operand of O = P V.  Neither S nor P ever reaches shared memory or
 * HBM.  qkv [batch][n_pix][3*heads*64] bf16 laid out (q | k | v) x head x 64; n_pix in {16, 64, 256} (small images are
 * packed 2 / 8 samples per 128-row tile); out [batch][n_pix][heads*64] bf16; lse (optional) [batch][heads][n_pix] fp32 =
 * log2-domain log-sum-exp of every query row, the only thing the backward needs besides qkv and out.           */
int adm_attn_fwd_fused(const void* qkv, int batch, int n_pix, int heads, float scale, void* out, float* lse,
                       void* stream);
/* K9 backward, ONE kernel: recomputes P from qkv and lse (nothing N x N is read from HBM), and produces dQ, dK and dV:
 * S^T = K Q^T and dP^T = V dO^T in TMEM, dS^T = scale P^T (dP^T - rowsum(dO o O)), dV += P^T dO and dK += dS^T Q with
 * the A operand read from TMEM, dQ += dS K through a shared-memory tile.  da [batch][n_pix][heads*64] bf16 (gradient
 * of out), out_fwd = the forward output, dqkv [batch][n_pix][3*heads*64] bf16 (dq | dk | dv).                 */
int adm_attn_bwd_fused(const void* da, const void* qkv, const void* out_fwd, const float* lse, int batch, int n_pix,
                       int heads, float scale, void* dqkv, void* stream);
/* The same attention for long sequences, n_pix = nblk * 256 in [512, 4096] (the 32 x 32 level of the CelebAHQ-latent UNet,
 * /root/reference/configs/celebahq/celeb_uncond_ddm_const_uncond_unet_ldm.yaml:55: attn_resolutions [32, 16]): the fused
 * kernels run over (sample, head, query block, key block) units of 256 x 256 and two small merge kernels combine the
 * per-block partials (log-sum-exp weighted sum forward, plain sum backward) — no n_pix x n_pix tensor exists.
 * `work` is caller-owned scratch of at least adm_attn_long_workspace(batch, n_pix, heads, backward) bytes.          */
long long adm_attn_long_workspace(int batch, int n_pix, int heads, int backward);
int adm_attn_fwd_long(const void* qkv, int batch, int n_pix, int heads, float scale, void* out, float* lse, void* work,
                      long long work_bytes, void* stream);
int adm_attn_bwd_long(const void* da, const void* qkv, const void* out_fwd, const float* lse, int batch, int n_pix,
                      int heads, float scale, void* dqkv, void* work, long long work_bytes, void* stream);
/* SpatialAtt + residual of the decouple branches (unet/uncond_unet.py:27-37, :566-567):
 * out = softsign(softmax(q k^T) att) * h + res with att = h . w_map + b; scalars = {b_map, wq, bq, wk, bk}.   */
int adm_spatial_att_fwd(const void* h, long long ldh, const void* res, long long ldr, const float* w_map,
                        const float* scalars, int n, int hw, int c, void* out, long long ldo, float* att_save,
                        float* o_save, void* stream);
int adm_spatial_att_bwd(const void* dy, long long ldy, const void* h, long long ldh, const float* w_map,
                        const float* scalars, const float* att_save, const float* o_save, int n, int hw, int c,
                        void* dh, long long lddh, float* dw_map, float* dscalars, void* stream);

/* ---------------------------------------------------------------- channel LayerNorm (conditional UNet)
 * cond_unet.py LayerNorm (:360-369, used by PreNorm / LinearAttention.to_out :371-379, :516-519):
 * y[p][c] = (x[p][c] - mean_p) * rsqrt(var_p + eps) * g[c] over the C channels of each pixel (biased variance), NHWC bf16.
 * C = 8 * 2^k * {1, 2, 4} with 2^k <= 32 (adm_chan_layernorm_ok).  backward: dx and dg[c] += sum_p dy * xhat (zero dg first);
 * mean / rstd are re-derived from x.                                                                         */
int adm_chan_layernorm_ok(int c);
int adm_chan_layernorm_fwd(const void* x, long long ldx, long long rows, int c, const float* g, float eps, void* y,
                           long long ldy, void* stream);
int adm_chan_layernorm_bwd(const void* dy, long long lddy, const void* x, long long ldx, long long rows, int c,
                           const float* g, float eps, void* dx, long long lddx, float* dg, void* stream);

/* ---------------------------------------------------------------- conditional UNet (unet/cond_unet.py)
 * K11  WeightStandardizedConv2d (:345-358): w_hat = (w - mean_o) * rsqrt(var_o + eps) per output channel (var unbiased =
 *      False), written straight in the GEMM engine's packed order bf16 [cout][k*k][pad64(cin)]; stats [cout][2] =
 *      (mean, rstd) are kept for the backward, which folds the un-pack of the packed weight gradient:
 *      dw = rstd * (g - mean(g) - w_hat * mean(g * w_hat)), g = d loss / d w_hat.                              */
int adm_ws_pack(const float* w, void* wpk, float* stats, int cout, int cin, int ksize, float eps, void* stream);
int adm_ws_pack_bwd(const float* dw_packed, const float* w, const float* stats, float* dw, int cout, int cin, int ksize,
                    int accumulate, void* stream);
/* K12  LinearAttention (:503-531) on qkv [batch][n_pix][ld] bf16 with channel order (q | k | v) x head x 32:
 *      q = softmax_d(q) * scale, k = softmax_n(k), v = v / n_pix, ctx[d][e] = sum_n k v, out[e][n] = sum_d ctx q.
 *      Neither softmax is materialised.  ctx fp32 [batch*heads][32][32] and kstat fp32 [batch*heads][32][2] are saved
 *      for the backward; work: fp32 scratch of adm_linattn_workspace() floats; dctx / r: scratch [batch*heads][32][32]
 *      and [batch*heads][32].  out [batch][n_pix][ldo] holds heads*32 channels; dqkv has the layout of qkv.       */
int adm_linattn_workspace(int batch, int heads, int n_pix, long long* floats);
int adm_linattn_fwd(const void* qkv, long long ld, int batch, int n_pix, int heads, int dim_head, float scale, void* out,
                    long long ldo, float* ctx, float* kstat, float* work, void* stream);
int adm_linattn_bwd(const void* qkv, long long ld, int batch, int n_pix, int heads, int dim_head, float scale,
                    const void* dout, long long ldd, const float* ctx, const float* kstat, float* dctx, float* r,
                    float* work, void* dqkv, long long ldg, void* stream);

/* ---------------------------------------------------------------- relation layers (conditional UNet)
 * BasicAttetnionLayer (unet/cond_unet.py:160-252), the full-resolution tail
 *     out = GroupNorm(x + y) + resize(z),   x = trunk features, y = concat_conv output (:236-240),
 *     z = out_conv applied to the pooled tokens (:248-251; a 1x1 conv commutes with the bilinear resize, whose weights
 *     sum to one), resize = F.interpolate(mode='bilinear', align_corners=True)
 * as one statistics pass + one apply pass over NHWC bf16 x, y [batch][h][w][c] with the sum held in fp32 registers.
 * z fp32 [batch][hq][wq][c]; out bf16 (or fp32 with out_fp32); stats fp32 [batch][groups][2] = (mean, rstd) is written
 * for the backward; work: fp32 scratch of batch * adm_rel_gn_chunks() * max(groups, c) * 2 floats.
 * Shapes: c % 8 == 0, (c / groups) % 8 == 0, c / 8 divides 256 (adm_rel_gn_ok).
 * backward: dpre bf16 = d loss / d (x + y) (the gradient of both addends); work then holds per-(sample, chunk, channel)
 * (sum dout * xhat, sum dout), whose sums over samples and chunks are d gamma / d beta.  d z is adm_bilinear_bwd(dout). */
int adm_rel_gn_ok(int batch, int h, int w, int c, int groups);
int adm_rel_gn_chunks(int batch, int h, int w, int c);
int adm_rel_gn_fwd(const void* x, const void* y, const float* z, int batch, int h, int w, int c, int hq, int wq,
                   int groups, const float* gamma, const float* beta, float eps, void* out, int out_fp32, float* stats,
                   float* work, void* stream);
int adm_rel_gn_bwd(const void* dout, const void* x, const void* y, int batch, int h, int w, int c, int groups,
                   const float* gamma, const float* stats, void* dpre, float* work, void* stream);
/* NHWC bilinear resize with align_corners=True (F.interpolate at unet/cond_unet.py:184, :248): x [batch][hin][win][c]
 * with pixel stride ldx -> y [batch][hout][wout][c] with pixel stride ldy; bf16 or fp32 on either side.  backward:
 * dy bf16 contiguous -> dx fp32 [batch][hin][win][c] as two separable axis reductions (rows into tmp fp32
 * [batch][hin][wout][c], then columns); the weights are re-derived exactly as the forward computes them.        */
int adm_bilinear_fwd(const void* x, long long ldx, int batch, int hin, int win, int c, void* y, long long ldy, int hout,
                     int wout, int in_fp32, int out_fp32, void* stream);
int adm_bilinear_bwd(const void* dy, int batch, int hout, int wout, int c, int hin, int win, float* tmp, float* dx,
                     void* stream);
/* Window average pool of an NHWC bf16 map, zero padded at the far edges to a multiple of the window
 * (F.pad + nn.AvgPool2d(window), unet/cond_unet.py:190-200): out [batch][ceil(h/kh)][ceil(w/kw)][c].           */
int adm_avgpool_fwd(const void* x, int batch, int h, int w, int c, int kh, int kw, void* out, void* stream);
int adm_avgpool_bwd(const void* dy, int batch, int h, int w, int c, int kh, int kw, void* dx, void* stream);

/* ---------------------------------------------------------------- optimizer over the flat parameter arena
 * train_uncond_dpm.py:292 (clip_grad_norm_ 1.0) + :179-180,296 (AdamW).  out += sum g^2.                      */
int adm_sq_norm(const float* g, long long numel, float* out, void* stream);
/* g_eff = g * grad_scale * min(1, max_norm / (sqrt(*sqnorm) * grad_scale + 1e-6)); torch.optim.AdamW update. */
int adm_adamw(float* p, const float* g, float* m, float* v, long long numel, float lr, float beta1, float beta2,
              float eps, float weight_decay, int step, float grad_scale, float max_norm, const float* sqnorm,
              const float* hyper_dev, void* p_bf16, void* stream);
/*   hyper_dev (optional, device fp32[3] = {lr, 1-beta1^step, sqrt(1-beta2^step)}) overrides lr/step so that a captured
 *   CUDA graph of the step can be replayed with fresh values.  p_bf16 (optional, bf16 [numel]): a bf16 shadow of the
 *   updated parameters written in the same pass — the tensor-core operands of the next step, so no separate
 *   weight re-pack is needed for parameters whose arena layout already is the packed [Cout][tap][Cin] order.     */
/* EMA of the weights as one pass over the flat arena (ddm/ema.py:141-156, EMA.update -> update_moving_average:
 * ma.lerp_(current, 1 - decay) per tensor): dst[i] += weight * (src[i] - dst[i]).                              */
int adm_lerp_f32(float* dst, const float* src, long long numel, float weight, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ADM_B200_H */
