/* e4t_b200.h — C-ABI of libe4t_b200.so: the sm_100a (B200) kernels behind the mkshing/e4t-diffusion module API.
 *
 * The reference has no FFI of its own (pure Python over ATen/cuBLAS/cuDNN/SDPA); these entry points are what its
 * Python operator layer binds for the E4T pre-training hot path (SURVEY.md §8b).  Each function cites the reference
 * call it replaces.  Conventions:
 *   - plain pointers + sizes only (no torch types); all pointers are DEVICE pointers unless stated otherwise
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous and stream-ordered, never allocates,
 *     never synchronises, holds no state between calls (thread-safe by construction)
 *   - returns 0 on success; non-zero -> e4t_last_error() describes the failure (the Python side raises)
 *   - activations are bf16, channels-last: images [B][H][W][C], tokens [B][N][C]; parameters/statistics are fp32
 */
#ifndef E4T_B200_H
#define E4T_B200_H
#ifdef __cplusplus
extern "C" {
#endif

/* ---- plumbing ---------------------------------------------------------------------------------------------- */
const char* e4t_last_error(void);              /* message of the last failing call on this thread               */
int e4t_version(void);                         /* 100 = 0.1.0                                                    */
unsigned long long e4t_launch_count(void);     /* kernels launched by this library since the last reset          */
void e4t_reset_launch_count(void);

/* ---- tcgen05 GEMM engine ------------------------------------------------------------------------------------ */
/* out[b] = alpha * op(A[b]) op(B[b])^T (+bias[n]) (+rowgroup[m / rows_per_group][n]) (+residual[m][n]).
 * Replaces F.linear at e4t/models/cross_attention.py:506,516,518,534, attention.py:429 (GEGLU proj), the 1x1
 * proj_in/proj_out convs of transformer_2d.py:153,209 and every autograd-generated dX / dW GEMM behind them.
 * a_mn / b_mn = 0: operand stored [rows][K] (K contiguous); = 1: stored [K][rows] (rows contiguous).
 * lda/ldb: row stride in elements (multiple of 8); a_bstride/b_bstride: batch stride, 0 = shared across the batch.
 * out_mode 0: bf16 store, 1: fp32 store, 2: fp32 atomic accumulate (required when splits > 1: split-K).
 * ldo / out_bstride: output row / batch stride in elements; ldr / res_bstride: the same for the bf16 residual.
 * splits: split-K factor; 0 with out_mode 2 = chosen by the library's tile cost model (weight gradients).
 * force_bn: N-tile override for tuning (0 = heuristic).
 * Alignment (also for the convolutions below, whose epilogue this is):
 *   - refused (non-zero return, nothing launched): A or B not 16-byte aligned, lda or ldb not a multiple of 8, bias or
 *     rowgroup not 16-byte aligned.  The rowgroup's row stride is N.  Also refused: splits > 1 with a bias, rowgroup or
 *     residual, and a force_bn outside [32, 256] or not a multiple of 32 (of 64 with b_mn).
 *   - any other pointer, ldo, ldr or batch stride is accepted; it only selects the epilogue.  A bf16 output goes
 *     through the TMA store when N, ldo (and out_bstride if batch > 1) are multiples of 8, out is 16-byte aligned and
 *     the residual is vectorisable (below).  Otherwise each thread stores 8 columns per 16-byte access if out is
 *     16-byte aligned and ldo / out_bstride are multiples of 16 bytes in the output type, the residual is vectorisable
 *     and (with a rowgroup) N % 4 == 0, and one element at a time if not.  The residual is vectorisable when it is
 *     16-byte aligned and ldr (and res_bstride if batch > 1) are multiples of 8. */
int e4t_gemm_bf16(const void* A, const void* B, void* out, int M, int N, int K, int batch, int a_mn, int b_mn,
                  long long lda, long long ldb, long long a_bstride, long long b_bstride, int out_mode,
                  long long ldo, long long out_bstride, const float* bias, const float* rowgroup,
                  int rows_per_group, const void* residual, long long ldr, long long res_bstride, float alpha,
                  int splits, int force_bn, void* stream);

/* 3x3 / stride 1 / pad 1 convolution as implicit GEMM (9 taps x Cin/64 K-chunks, halo by TMA zero fill).
 * Replaces nn.Conv2d inside diffusers ResnetBlock2D.conv1/conv2, Upsample2D.conv, Downsample2D.conv
 * (constructed at e4t/models/unet_2d_blocks.py:481-492,760-771,801-808,1732-1743,1773-1774) and their dgrad.
 * x [B][H][W][Cin] bf16 (Cin % 64 == 0, W | 128); w [9][Cout][Cin] bf16 (tap = ky*3+kx); out [B][H][W][Cout];
 * bias fp32 [Cout]; rowgroup fp32 [B][Cout] (time-embedding projection added per image); residual bf16 like out. */
int e4t_conv3x3_bf16(const void* x, const void* w, void* out, int B, int H, int W, int Cin, int Cout, int out_mode,
                     const float* bias, const float* rowgroup, const void* residual, int force_bn, void* stream);

/* 3x3 / stride 2 / pad 1 (diffusers Downsample2D.conv, built at e4t/models/unet_2d_blocks.py:801-808): computed at the
 * OUTPUT resolution — the implicit-GEMM A operand is gathered with TMA element strides.  x [B][H][W][Cin] ->
 * out [B][H/2][W/2][Cout]. */
int e4t_conv3x3_s2_bf16(const void* x, const void* w, void* out, int B, int H, int W, int Cin, int Cout,
                        const float* bias, int force_bn, void* stream);
/* General forward 3x3 convolution for the VAE (diffusers AutoencoderKL Encoder/Decoder): stride 1 or 2; top/left
 * padding `pad` 1, or 0 with stride 2 (Downsample2D(padding=0) == F.pad(x, (0,1,0,1)) + pad-0 conv; the bottom/right
 * zeros come from the TMA out-of-bounds fill).  Output width W/stride divides 128 or is a multiple of 128 (wide images:
 * one M tile = 128 pixels of one row).  x [B][H][W][Cin] -> out [B][H/stride][W/stride][Cout] bf16; bias fp32 [Cout];
 * residual bf16 like out or null. */
int e4t_conv3x3_ex(const void* x, const void* w, void* out, int B, int H, int W, int Cin, int Cout, int stride, int pad,
                   const float* bias, const void* residual, int force_bn, void* stream);
/* Weight gradient of the 3x3 / stride 1 / pad 1 convolution: dw9[tap][co][ci] += sum dy[b][y][x][co] * x[b][y+ky-1][x+kx-1][ci]
 * (fp32 atomic accumulation; implicit GEMM with 9 taps as the batch dimension, split-K over pixels).  Replaces autograd's
 * conv2d weight gradient when the base UNet is trainable (tuning_e4t.py:139-146; every requires_grad parameter under
 * accelerate's DDP, pretrain_e4t.py:410). */
int e4t_conv3x3_wgrad(const void* x, const void* dy, float* dw9, int B, int H, int W, int Cin, int Cout, void* stream);

/* ---- attention core ------------------------------------------------------------------------------------------ */
/* O = softmax(Q K^T * scale) V, LSE = logsumexp rows.  Replaces F.scaled_dot_product_attention at
 * e4t/models/cross_attention.py:527-529 (== get_attention_scores + bmm, :222-251,313-315).
 * Q [B][N][H*dh], K/V [B][M][H*dh] with row strides ld* and batch strides *_bs (elements), dh % 8 == 0, <= 192.
 * LSE fp32 [B][H][N]. */
int e4t_attn_fwd(const void* Q, const void* K, const void* V, void* O, float* LSE, int B, int H, int N, int M, int dh,
                 long long ldq, long long q_bs, long long ldk, long long k_bs, long long ldv, long long v_bs,
                 long long ldo, long long o_bs, float scale, void* stream);
/* Backward of the above (autograd of SDPA in the reference).  Dv: fp32 scratch [B][H][N]. */
int e4t_attn_bwd(const void* Q, const void* K, const void* V, const void* O, const void* dO, const float* LSE,
                 float* Dv, void* dQ, void* dK, void* dV, int B, int H, int N, int M, int dh, long long ldq,
                 long long q_bs, long long ldk, long long k_bs, long long ldv, long long v_bs, long long ldo,
                 long long o_bs, long long lddo, long long do_bs, long long lddq, long long dq_bs, long long lddk,
                 long long dk_bs, long long lddv, long long dv_bs, float scale, void* stream);

/* Single-pass backward: S and dP are computed once per (query block, key tile) pair and dQ is reduced into the fp32
 * scratch dQacc [B][N][H*dh] (zeroed by the call) before being written to dQ as bf16.  Falls back to e4t_attn_bwd
 * when 256 + 3*round16(dh) TMEM columns do not fit (dh > 80) or N < 128. */
int e4t_attn_bwd_fused(const void* Q, const void* K, const void* V, const void* O, const void* dO, const float* LSE,
                       float* Dv, float* dQacc, void* dQ, void* dK, void* dV, int B, int H, int N, int M, int dh,
                       long long ldq, long long q_bs, long long ldk, long long k_bs, long long ldv, long long v_bs,
                       long long ldo, long long o_bs, long long lddo, long long do_bs, long long lddq, long long dq_bs,
                       long long lddk, long long dk_bs, long long lddv, long long dv_bs, float scale, void* stream);
/* The same with a causal mask (key j contributes to query i only if j <= i; N == M, dh <= 80, any N): backward of the CLIP
 * text tower's masked self-attention, e4t/models/modeling_clip.py:45-51.  O / LSE from e4t_attn_small_fwd(causal = 1). */
int e4t_attn_bwd_fused_causal(const void* Q, const void* K, const void* V, const void* O, const void* dO, const float* LSE,
                       float* Dv, float* dQacc, void* dQ, void* dK, void* dV, int B, int H, int N, int M, int dh,
                       long long ldq, long long q_bs, long long ldk, long long k_bs, long long ldv, long long v_bs,
                       long long ldo, long long o_bs, long long lddo, long long do_bs, long long lddq, long long dq_bs,
                       long long lddk, long long dk_bs, long long lddv, long long dv_bs, float scale, void* stream);

/* Short-sequence attention (N, M <= 128, dh <= 64) with optional causal mask: the CLIP text tower's 77-token causal
 * self-attention (e4t/models/modeling_clip.py:45-51, HF CLIPAttention) and its backward.  Same layout as e4t_attn_fwd. */
int e4t_attn_small_fwd(const void* Q, const void* K, const void* V, void* O, float* LSE, int B, int H, int N, int M,
                       int dh, long long ldq, long long q_bs, long long ldk, long long k_bs, long long ldv,
                       long long v_bs, long long ldo, long long o_bs, float scale, int causal, void* stream);
int e4t_attn_small_bwd(const void* Q, const void* K, const void* V, const void* O, const void* dO, const float* LSE,
                       void* dQ, void* dK, void* dV, int B, int H, int N, int M, int dh, long long ldq, long long q_bs,
                       long long ldk, long long k_bs, long long ldv, long long v_bs, long long ldo, long long o_bs,
                       long long lddo, long long do_bs, long long lddq, long long dq_bs, long long lddk, long long dk_bs,
                       long long lddv, long long dv_bs, float scale, int causal, void* stream);

/* Row softmax P[r][:M] = softmax(S[r][:M]) (fp32 in, bf16 out, row stride ld for both; M, ld % 4 == 0): the middle of
 * the three launches of the VAE mid-block AttentionBlock (diffusers attention.py AttentionBlock.forward),
 * S = alpha Q K^T and O = P V being e4t_gemm_bf16 calls.  No length limit on M.  Entries may be -inf (masked) as long
 * as a row keeps one finite entry; P's columns M..ld-1 are not written.  S 16-byte and P 8-byte aligned. */
int e4t_softmax_rows(const float* S, void* P, long long rows, int M, long long ld, void* stream);

/* ---- normalisation ------------------------------------------------------------------------------------------- */
/* GroupNorm (+ optional fused SiLU).  Replaces nn.GroupNorm + F.silu in diffusers ResnetBlock2D, Transformer2DModel
 * .norm (transformer_2d.py:149,253) and conv_norm_out/conv_act (unet_2d_condition.py:554-556).
 * x,y [B][HW][C] bf16; stats fp32 [B][G][2] = (Σ(x - p), Σ(x - p)²) over the group, taken about its first element
 * p = x[b][0][g * C/G] (mean = p + Σ(x - p)/n, var = Σ(x - p)²/n - (Σ(x - p)/n)², free of the cancellation of
 * Σx²/n - mean² for groups whose mean is large against their spread); written by fwd and consumed by bwd with the same x. */
int e4t_groupnorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* stats, int B, int HW,
                      int C, int G, float eps, int act_silu, void* stream);
int e4t_groupnorm_bwd(const void* x, const void* dy, const float* gamma, const float* beta, const float* stats,
                      void* dx, float* scratch /* [B][G][2] */, int B, int HW, int C, int G, float eps, int act_silu,
                      void* stream);
/* LayerNorm over the last dim.  Replaces nn.LayerNorm at attention.py:258-273.  stats fp32 [rows][2] = (mean, rstd). */
int e4t_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* stats, long long rows,
                      int C, float eps, void* stream);
int e4t_layernorm_bwd(const void* x, const void* dy, const float* gamma, const float* stats, void* dx, long long rows,
                      int C, float eps, void* stream);

/* Affine-parameter gradients (accumulating into fp32 dgamma / dbeta), needed when the norms are trainable
 * (tuning_e4t.py:139-146, --unfreeze_clip_vision).  LayerNorm: stats as written by e4t_layernorm_fwd.  GroupNorm(+SiLU):
 * mean_c / rstd_c fp32 [B][C] = the group statistics expanded per channel. */
int e4t_layernorm_param_grad(const void* x, const void* dy, const float* stats, const float* gamma, float* dgamma,
                             float* dbeta, long long rows, int C, void* stream);
int e4t_groupnorm_param_grad(const void* x, const void* dy, const float* mean_c, const float* rstd_c, const float* gamma,
                             const float* beta, float* dgamma, float* dbeta, int B, int HW, int C, int act_silu,
                             void* stream);

/* ---- elementwise --------------------------------------------------------------------------------------------- */
/* Activations on bf16: mode 0 exact erf GELU (open_clip ViT MLP, e4t/encoder.py:91-96), 1 quick GELU (HF CLIP text MLP
 * behind e4t/models/modeling_clip.py:10-82), 2 LeakyReLU(0.01) (E4TEncoder head, e4t/encoder.py:101-105,163-166). */
int e4t_act_fwd(const void* x, void* y, long long n, int mode, void* stream);
int e4t_act_bwd(const void* x, const void* dy, void* dx, long long n, int mode, void* stream);
/* out[g][n] += sum over the rows of group g (rows_per_group consecutive rows; <= 0: one group) of X[m][n]: bias gradients
 * and the per-image time-embedding-row gradient of ResnetBlock2D. */
int e4t_colsum_acc(const void* X, float* out, long long M, int N, long long ld, long long rows_per_group, void* stream);
/* Weight gradients of the UNet's two narrow 3x3 convolutions (conv_in 4->C, unet_2d_condition.py:481; conv_out C->4, :557):
 * acc[w][n][tap] += sum wide[b][y][x][w] * narrow[b][n][y+sgn*(ky-1)][x+sgn*(kx-1)]; wide bf16 NHWC, narrow fp32 NCHW (<= 4 ch). */
int e4t_narrow_conv_wgrad(const void* wide, const float* narrow, float* acc, int B, int H, int W, int Cw, int Cn, int sgn,
                          void* stream);
/* GEGLU: out = h[:, :F] * gelu(h[:, F:]) (attention.py:409-430). */
int e4t_geglu_fwd(const void* h, void* out, long long rows, int F, void* stream);
int e4t_geglu_bwd(const void* h, const void* dout, void* dh, long long rows, int F, void* stream);
/* 2x spatial resampling on NHWC (H, W = the SMALL resolution): mode 0 nearest upsample (diffusers Upsample2D),
 * 1 its adjoint, 2 stride-2 pick (Downsample2D = stride-1 conv sampled at even positions), 3 zero insertion. */
int e4t_resample2x(const void* x, void* y, int B, int H, int W, int C, int mode, void* stream);
/* UNet conv_in (unet_2d_condition.py:481): NCHW fp32 -> NHWC bf16; w fp32 [Cout][Cin][3][3]. */
int e4t_conv_in_fwd(const float* x, const float* w, const float* bias, void* y, int B, int Cin, int H, int W,
                    int Cout, void* stream);
/* 1x1 convolution on NCHW fp32 (Cin, Cout <= 8): the VAE's post_quant_conv on the latents before Decoder.conv_in.
 * w fp32 [Cout][Cin]; bias fp32 [Cout] or null. */
int e4t_pointwise_nchw(const float* x, const float* w, const float* bias, float* y, int B, int Cin, int Cout,
                       long long HW, void* stream);
/* UNet conv_out (unet_2d_condition.py:557): NHWC bf16 -> NCHW fp32, and its input gradient. */
int e4t_conv_out_fwd(const void* x, const float* w, const float* bias, float* y, int B, int H, int W, int C, int Cout,
                     void* stream);
int e4t_conv_out_bwd(const float* dy, const float* w, void* dx, int B, int H, int W, int C, int Cout, void* stream);
/* E4TEncoder feature pooling (e4t/encoder.py:147-148): out[b][c_off + c] = mean over HW, and its adjoint. */
int e4t_meanpool_fwd(const void* x, float* out, int B, int HW, int C, int ldo, int c_off, void* stream);
int e4t_meanpool_bwd(const float* dout, void* dx, int B, int HW, int C, int ldo, int c_off, void* stream);

/* ---- WeightOffsets (e4t/weightoffsets.py:14-23, applied at cross_attention.py:506,516,518) -------------------- */
/* Closed form: vx = w1 v + b1, vy = w2 v + b2, a = Wc vx, b = Wr vy, s = Wr 1; Delta = b a^T + s bc^T + br 1^T. */
int e4t_wo_factors_fwd(const float* v, const float* w1, const float* b1, const float* w2, const float* b2,
                       const float* Wc, const float* Wr, float* vx, float* vy, float* a, float* b, float* s, int R,
                       int C, void* stream);
/* W_eff[c][r] = bf16(W[c][r] * (1 + Delta[c][r])) — `attn.to_q.weight * (1 + attn.wo_q())`. */
int e4t_wo_weff_fwd(const float* W, const float* a, const float* bc, const float* b, const float* s, const float* br,
                    void* w_eff, int C, int R, void* stream);
/* All nine parameter gradients from the accumulated dW_eff (fp32 [C][R]); scratch fp32 [4C + 3R]. */
int e4t_wo_bwd(const float* dWeff, const float* W, const float* v, const float* w1, const float* w2, const float* Wc,
               const float* Wr, const float* bc, const float* vx, const float* vy, const float* a, const float* b,
               const float* s, float* scratch, float* dv, float* dw1, float* db1, float* dw2, float* db2, float* dWc,
               float* dbc, float* dWr, float* dbr, int R, int C, void* stream);

/* Batched variants over ALL WeightOffsets projections of a model: `tab` is a device array of n WOProj records
 * (csrc/elementwise.cu; mirrored by e4t_b200/wobank.py) holding parameter, scratch, W_eff, dW_eff and gradient
 * pointers.  fwd = 2 launches (factors, W_eff); bwd = 4 launches + one memset of the backward scratch. */
int e4t_wo_bank_fwd(const void* tab, int n, int max_r, int max_c, void* stream);
int e4t_wo_bank_bwd(const void* tab, int n, int max_r, int max_c, float* bw_base, long long bw_floats, void* stream);
/* The same in two phases, for data-parallel runs: _reduce leaves the five G reductions of every projection in bw
 * (contiguous, ~2 MB for SD-v1.4); the caller all-reduces bw; _apply expands them into the parameter gradients
 * (every later step is linear in them with rank-identical coefficients, SURVEY.md App. A). */
int e4t_wo_bank_bwd_reduce(const void* tab, int n, int max_r, int max_c, float* bw_base, long long bw_floats, void* stream);
int e4t_wo_bank_bwd_apply(const void* tab, int n, int max_r, int max_c, void* stream);
int e4t_wo_bank_record_size(void);

/* ---- optimiser (torch.optim.AdamW at pretrain_e4t.py:389-392,652) ---------------------------------------------- */
int e4t_adamw_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, int step, float grad_scale, void* stream);
/* Same with the step counter in device memory (*step_dev is incremented, then used): CUDA-graph replayable. */
int e4t_adamw_step_dev(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
                       float eps, float weight_decay, int* step_dev, float grad_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* E4T_B200_H */
