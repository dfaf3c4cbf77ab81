/* mos_sm100.h — C ABI of libmos_sm100.so, the B200 (sm_100a) ED-LoRA diffusion hot path.
 *
 * Conventions (SURVEY.md §8b): every entry point returns int (0 = ok, negative = MOS_E*); the message of the
 * last failure on the calling thread is available from mos_last_error(). All pointers are raw device pointers
 * owned by the caller (PyTorch allocates everything); the library never allocates per call, never retains a
 * pointer after return and never synchronises: work is enqueued on the cudaStream_t passed as `stream`.
 * Activations and packed weights are 16-bit, NHWC / token-major resp. K-major: bf16 (training) or fp16 (sampling: the
 * reference's own sampling precision; its three extra mantissa bits keep the classifier-free-guidance difference accurate,
 * DESIGN.md "numerics"); `act_dtype` / MOS_DT_* selects the type.  tcgen05 kind::f16 takes ONE operand format per MMA, so
 * the operands of a GEMM share the type.  Accumulation, statistics and softmax are fp32.
 *
 * Each entry point cites the reference call site it replaces (paths relative to TencentARC/Mix-of-Show).
 */
#ifndef MOS_SM100_H
#define MOS_SM100_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOS_OK 0
#define MOS_EINVAL (-1)   /* bad argument (shape / alignment / null pointer) */
#define MOS_ECUDA (-2)    /* CUDA runtime / driver error */
#define MOS_EUNSUPPORTED (-3)

int mos_version(void);
const char* mos_last_error(void);

/* ------------------------------------------------------------------------------------------------------------
 * Fused GEMM (+ implicit-GEMM 3x3 convolution) with LoRA / bias / temb / GEGLU / residual epilogue.
 *   out[m, n] = epi( sum_k A[m, k] * W[n, k]  +  sum_r (sum_k A[m,k] * lora_down[r,k]) * lora_up[n, r] )
 * Replaces, in one tcgen05 kernel:
 *   - LoRALinearLayer.forward                     mixofshow/models/edlora.py:244-246
 *   - attn.to_q / to_k / to_v / to_out[0]         mixofshow/models/edlora.py:143-145,161 (and :69-71,88)
 *   - region to_k / to_v                          mixofshow/pipelines/pipeline_regionally_t2iadapter.py:122-126
 *   - diffusers ResnetBlock2D conv1/conv2, Transformer2DModel proj_in/proj_out, FeedForward GEGLU
 *     (called through unet(...) at mixofshow/pipelines/pipeline_edlora.py:277)
 * ---------------------------------------------------------------------------------------------------------- */
enum { MOS_DT_BF16 = 0, MOS_DT_F16 = 1 };   /* 16-bit storage type of activations (`act_dtype` arguments) */
enum { MOS_OUT_BF16 = 0 /* 16-bit rows of type a_dtype */, MOS_OUT_HEADS = 1, MOS_OUT_F32 = 2 };
enum { MOS_SEG_ROWS = 0 /* [b,h,row,dpad] (Q, K) */, MOS_SEG_TRANSPOSED = 1 /* [b,h,d,row] (V^T) */ };
enum { MOS_ACT_NONE = 0, MOS_ACT_RELU = 1 };   /* epilogue activation (`act`) */

typedef struct mos_gemm_args {
  const void* A;          /* bf16 [M, lda]; conv: NHWC activation [B, H, Wd, C] */
  const void* W;          /* bf16 [N, Kw], K contiguous; conv: [N, 9*C] with k = (kh*3+kw)*C + c */
  int64_t M, N, K;        /* K = C for conv (reduction per tap) */
  int64_t lda;            /* row pitch of A in elements (conv: pixel pitch, >= C) */
  int32_t conv;           /* 0 = plain GEMM, 1 = 3x3 / stride 1 / pad 1 convolution */
  int32_t B, H, Wd, C;    /* conv geometry */
  int32_t splits;         /* split-K factor, >= 1; > 1 requires `partial` and forbids lora / geglu / heads */
  int32_t stages;         /* smem pipeline depth, 0 = default */
  float* partial;         /* fp32 workspace [splits, M, N] */
  const float* bias;      /* [N] or NULL */
  const float* bias_batch;/* [nbatch, N] or NULL; row m uses batch m / rows_per_batch (resnet temb add) */
  int64_t rows_per_batch;
  int64_t bias_batch_ld;  /* row pitch of bias_batch in elements (0 = N) */
  const void* residual;   /* bf16 [M, ldr] or NULL, added last */
  int64_t ldr;
  int32_t geglu;          /* 1: tile columns are [80 x a | 80 x gate]; writes a*gelu(gate), N_out = N/2 */
  const void* lora_down;  /* bf16 [16, K], rows >= rank zero; NULL = no LoRA */
  const float* lora_up;   /* fp32 [N, 4], pre-multiplied by alpha */
  int64_t lora_seg;       /* columns per LoRA segment (N, or C for fused q|k|v: segment s uses down rows 4s..4s+3) */
  int32_t out_mode;       /* MOS_OUT_* */
  void* out;              /* bf16 / fp32 [M, ldc] for MOS_OUT_BF16 / MOS_OUT_F32 */
  int64_t ldc;
  /* MOS_OUT_HEADS: columns are `nseg` segments of seg_len = heads*head_dim; segment s goes to seg_ptr[s] */
  void* seg_ptr[3];
  int32_t seg_kind[3];
  int64_t seg_rows_pad[3];   /* padded row count of the destination (tokens or keys) */
  int32_t heads, head_dim, dpad, dv_pad;
  int64_t tokens_per_batch;
  int32_t accumulate;     /* MOS_OUT_F32 only: out += result (Gram accumulation, gradient fusion) */
  int32_t w_static;       /* reserved, ignored (round 1 requested the first W tiles ahead of griddepcontrol.wait when set; the
                           * measurement was neutral and the path was removed) */
  int32_t a_dtype;        /* MOS_DT_*: type of A, of the 16-bit outputs (rows, head-split) and of `residual` */
  int32_t w_dtype;        /* MOS_DT_*: type of W and lora_down; must equal a_dtype (one operand format per tcgen05 MMA) */
  int32_t pair_mode;      /* 0 = library heuristic, 1 = force 2-CTA pair tiles (needs an even number of 128-row tiles),
                           * 2 = force the 1-CTA kernel (benchmarking) */
  int32_t* tile_counters; /* split-K only, optional: int32 [tile_counters_len] device counters, ZERO on entry (the kernel
                           * leaves them zero).  When given, the launch also finalizes: the `splits` CTAs of an output tile
                           * sum the partials in split order and write bias / bias_batch / residual -> `out` themselves
                           * (no mos_splitk_finalize launch).  One buffer per stream: launches that may overlap must not
                           * share it. */
  int32_t tile_counters_len;   /* >= (M tiles) x (N / 160) */
  const void* prefetch_ptr;    /* optional: [prefetch_bytes] of STATIC device data (normally the next layer's weights) that the
                                * launch pulls into L2 with cp.async.bulk.prefetch.L2 while it runs; semantically a no-op */
  int64_t prefetch_bytes;
  int32_t act;            /* MOS_ACT_*: out = act(acc + bias) (+ residual), in fp32 before rounding (T2I-Adapter resnet
                           * block1).  Needs 16-bit row output without split-K / geglu / LoRA. */
} mos_gemm_args;

int mos_gemm_bf16(const mos_gemm_args* args, void* stream);

/* Profiling aid: register a device buffer of 64 uint64 (or NULL to disable); the first 8 CTAs of every subsequent
 * mos_gemm_bf16 launch store %globaltimer stamps [start, setup done, pdl wait done, first TMA landed, epilogue
 * prefetch done, accumulators ready, accumulators drained, tile written]. */
int mos_debug_set_timeline(void* buf);

/* Profiling aid for mos_attention_fwd: register a device buffer of 256 uint64 (or NULL to disable); CTA (0,0) of every
 * subsequent launch stores clock64 stamps for its first 32 kv tiles: softmax warp 0 at [j*4 + k] (k: before s_full wait,
 * S visible, softmax pass done, P published) and the MMA thread at [128 + j*4 + k] (k: K/V landed, S buffer free and
 * S_j issued next, before p_full wait, P visible and PV_j issued next). */
int mos_debug_set_attn_timeline(void* buf);

/* Sum split-K partials and apply bias / bias_batch / residual -> bf16 [M, ldc]. */
int mos_splitk_finalize(const float* partial, int32_t splits, int64_t M, int64_t N, const float* bias,
                        const float* bias_batch, int64_t rows_per_batch, int64_t bias_batch_ld,
                        const void* residual, int64_t ldr, void* out, int64_t ldc, int32_t act_dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Flash attention (tcgen05 S = QK^T and PV in TMEM, online softmax in registers), head_dim in {40, 80, 160}.
 *   Q, K : bf16 [batch*heads, nq|nk, DP]   DP = head_dim rounded up to 64, pad columns zero
 *   Vt   : bf16 [batch*heads, DV, nk8]     DV = head_dim rounded up to 16, nk8 = nk rounded up to 8, pads zero
 *   out  : bf16 [batch, nq, ldo], head h at columns [h*head_dim, (h+1)*head_dim)
 *   probs: optional fp32 [batch*heads, nq, nk] (cross-attention maps for the controller; single kv tile only)
 * Replaces xformers.ops.memory_efficient_attention and attn.get_attention_scores + torch.bmm at
 *   mixofshow/models/edlora.py:77-83,151-156; mixofshow/pipelines/pipeline_regionally_t2iadapter.py:111-116
 * and the per-region einsum/softmax/einsum at pipeline_regionally_t2iadapter.py:71-78 (one call per region).
 * ---------------------------------------------------------------------------------------------------------- */
int mos_attention_fwd(const void* Q, const void* K, const void* Vt, void* out, int64_t ldo, float* probs,
                      int32_t batch, int32_t heads, int32_t head_dim, int32_t nq, int32_t nk, int32_t nk8,
                      float scale, int32_t act_dtype, void* stream);

/* GroupNorm(32)(+SiLU) over NHWC bf16 rows: x [B, HW, ldx] -> y [B, HW, ldy]; partial = fp32 workspace of
 * partial_capacity_floats floats (>= B * 592 * 64 is always enough). The LAST 64 words of the workspace hold the grid-barrier
 * state of the single-launch path and must be zero-initialised once by the caller (never touched afterwards). diffusers ResnetBlock2D.norm1/norm2,
 * Transformer2DModel.norm, conv_norm_out (reached from mixofshow/pipelines/pipeline_edlora.py:277). */
int mos_groupnorm_fwd(const void* x, int64_t ldx, int32_t B, int32_t HW, int32_t C, const float* gamma,
                      const float* beta, float eps, int32_t silu_act, float* partial,
                      int32_t partial_capacity_floats, void* y, int64_t ldy, int32_t act_dtype, void* stream);

/* Debug / benchmarking switch: 1 forces the two-launch GroupNorm (statistics kernel + apply kernel), 0 the one-pass cluster
 * kernel (default; environment MOS_GN_TWOPASS=1 has the same effect). */
int mos_debug_set_gn_twopass(int32_t on);

/* LayerNorm over rows of bf16 [M, ldx] -> [M, ldy], C <= 1280 (BasicTransformerBlock.norm1/2/3). */
int mos_layernorm_fwd(const void* x, int64_t ldx, int64_t M, int32_t C, const float* gamma, const float* beta,
                      float eps, void* y, int64_t ldy, int32_t act_dtype, void* stream);

/* Sinusoidal timestep embedding [B, dim] fp32 = [cos | sin] (diffusers Timesteps, flip_sin_to_cos, shift 0). */
int mos_timestep_embedding(const float* t, int32_t B, int32_t dim, float* out, void* stream);

/* Small-batch GEMV: out[b, n] = act_out(bias[n] + sum_k act_in(x[b,k]) W[n,k]); x fp32 [nb<=8, K], W bf16 [N, K];
 * act: 0 = identity, 1 = SiLU. Time-embedding MLP and all ResnetBlock2D.time_emb_proj in one launch. */
int mos_gemv_bf16(const float* x, int32_t nb, int32_t K, const void* W, const float* bias, int32_t N,
                  int32_t act_in, int32_t act_out, float* out, int64_t ldo, void* stream);

/* conv_in: NCHW fp32 latents [B, Cin, H, W] -> NHWC bf16 [B, H, W, ldy]; w fp32 [9*Cin, Cout] tap-major. */
int mos_conv_in(const float* x, int32_t B, int32_t Cin, int32_t H, int32_t W, const float* w, const float* bias,
                int32_t Cout, void* y, int64_t ldy, int32_t act_dtype, void* stream);
/* conv_out: NHWC bf16 [B, H, W, C] -> NCHW fp32 [B, Cout<=4, H, W]; w fp32 [Cout, 9, C]. */
int mos_conv_out(const void* x, int32_t B, int32_t H, int32_t W, int32_t C, const float* w, const float* bias,
                 int32_t Cout, float* y, int32_t act_dtype, void* stream);

/* Upsample2D nearest x2: NHWC bf16 [B, H, W, ldx] -> contiguous [B, 2H, 2W, C]. */
int mos_upsample2x(const void* x, int64_t ldx, int32_t B, int32_t H, int32_t W, int32_t C, void* y, void* stream);
/* Downsample2D (3x3, stride 2) im2col: NHWC 16-bit -> [B*H/2*W/2, 9*C] for mos_gemm_bf16.  pad = 1: symmetric padding 1
 * (UNet Downsample2D); pad = 0: the VAE encoder's variant (F.pad (0,1,0,1) then no padding: taps start at 2*ho). */
int mos_im2col_s2(const void* x, int64_t ldx, int32_t B, int32_t H, int32_t W, int32_t C, int32_t pad, void* col,
                  void* stream);
/* x[m, :C] += r[m, :C] (T2I-Adapter residuals, pipeline_regionally_t2iadapter.py:565). */
int mos_add_rows(void* x, int64_t ldx, const void* r, int64_t ldr, int64_t M, int32_t C, int32_t act_dtype,
                 void* stream);

/* ---- T2I-Adapter (diffusers T2IAdapter, adapter_type 'full_adapter', run once per condition image at
 * pipeline_regionally_t2iadapter.py:474-482).  Its 3x3 / 1x1 convolutions reuse mos_gemm_bf16 (conv / plain, MOS_ACT_RELU). */
/* PixelUnshuffle(r): fp32 NCHW [B, C, H, W] -> 16-bit NHWC rows [B*(H/r)*(W/r), ldy], column c*r*r + i*r + j =
 * x[b, c, ho*r + i, wo*r + j] (torch's channel order).  H, W multiples of r; C*r*r a multiple of 8. */
int mos_pixel_unshuffle(const float* x, int32_t B, int32_t C, int32_t H, int32_t W, int32_t r, void* y, int64_t ldy,
                        int32_t act_dtype, void* stream);
/* AvgPool2d(2, 2, ceil_mode=True): 16-bit NHWC [B, H, W, ldx] -> [B, ceil(H/2), ceil(W/2), ldy]; fp32 sum divided by the
 * number of taps inside the input (odd H / W: the last row / column averages 2 or 1 taps). */
int mos_avgpool2x2(const void* x, int64_t ldx, int32_t B, int32_t H, int32_t W, int32_t C, void* y, int64_t ldy,
                   int32_t act_dtype, void* stream);

/* ---- CLIP text encoder (SURVEY.md 8f rank 1; transformers CLIPTextModel called at pipeline_edlora.py:133-145,
 * trainer_edlora.py:220-234, gradient_fusion.py:182-199).  The linears and LayerNorms reuse mos_gemm_bf16 / mos_layernorm_fwd. */
/* x[m, :C] = token_embedding[ids[m]] + position_embedding[m % T] -> bf16 [M, ld]; columns C..ld-1 are zeroed. */
int mos_clip_embed(const int32_t* ids, const float* token_embedding, const float* position_embedding, int64_t M, int32_t T,
                   int32_t C, int32_t vocab, void* x, int64_t ld, void* stream);
/* x[m, :C] <- x * sigmoid(1.702 x) in place (quick-GELU of the CLIP MLP). */
int mos_quick_gelu(void* x, int64_t ld, int64_t M, int32_t C, void* stream);
/* Causal self-attention over one key tile (n <= 128): layouts as mos_attention_fwd; head_dim 80 only (CLIP's 64-dim heads
 * run zero-padded to 80 with scale = 64^-0.5). */
int mos_attention_fwd_causal(const void* Q, const void* K, const void* Vt, void* out, int64_t ldo, int32_t batch,
                             int32_t heads, int32_t head_dim, int32_t n, int32_t n8, float scale, float* lse2,
                             void* stream);   /* lse2 (optional) [batch*heads, n]: saved for mos_attention_bwd (causal) */
/* Training pieces of the CLIP text encoder (trainer_edlora.py:220-234 reached through loss.backward(), train_edlora.py:120):
 * out-of-place quick-GELU (the pre-activation is kept) and its backward; the gradient of the new-concept rows of the
 * token-embedding table: out[r, :C] (+)= sum_{m: ids[m] == rows[r]} dx[m, :C]  (fp32 [n_rows, C], fixed summation order). */
int mos_quick_gelu_fwd(const void* x, int64_t ldx, int64_t M, int32_t C, void* y, int64_t ldy, void* stream);
int mos_quick_gelu_bwd(const void* x, int64_t ldx, const void* dy, int64_t lddy, int64_t M, int32_t C, void* dx,
                       int64_t lddx, void* stream);
int mos_clip_embed_bwd(const int32_t* ids, const void* dx, int64_t ld, int64_t M, int32_t C, const int32_t* rows,
                       int32_t n_rows, int32_t accumulate, float* out, void* stream);

/* ---- VAE (AutoencoderKL; SURVEY.md 8f rank 2: `vae.encode(images).latent_dist.sample() * 0.18215` trainer_edlora.py:203-204,
 * `vae.decode(latents / 0.18215)` pipeline_edlora.py:303-313).  Convolutions / projections / GroupNorm reuse mos_gemm_bf16,
 * mos_groupnorm_fwd, mos_conv_in / mos_conv_out, mos_upsample2x, mos_im2col_s2(pad = 0); the single-head d = 512 attention
 * of the mid block is two GEMMs around mos_softmax_rows. */
/* out[r, :cols] = softmax(scale * S[r, :cols]) as 16-bit; S fp32 [rows, lds]. */
int mos_softmax_rows(const float* S, int64_t lds, int64_t rows, int32_t cols, float scale, void* out, int64_t ldo,
                     int32_t act_dtype, void* stream);
/* fp32 NCHW 1x1 convolution with <= 8 channels (post_quant_conv): y[b,o,p] = bias[o] + sum_c w[o,c] x[b,c,p]. */
int mos_conv1x1_nchw(const float* x, int32_t B, int32_t Cin, int64_t HW, const float* w, const float* bias, int32_t Cout,
                     float* y, void* stream);
/* encoder tail: h 16-bit NHWC [B*HW, ldh] (2L moment channels) -> quant_conv (w [2L,2L], bias) -> mean, logvar (clamped to
 * [-30, 20]) fp32 NCHW [B, L, HW]; with `noise` (standard normal, same layout): latents = scaling (mean + exp(logvar/2) noise). */
int mos_vae_moments(const void* h, int64_t ldh, int32_t B, int64_t HW, int32_t L, const float* w, const float* bias,
                    float* mean, float* logvar, const float* noise, float scaling, float* latents, int32_t act_dtype,
                    void* stream);

/* One fused kernel for mixofshow/pipelines/pipeline_edlora.py:273-290: classifier-free-guidance combine,
 * DPM-Solver++(2M) data-prediction update and re-duplication of the latents for the next UNet call.
 * noise_pred fp32 [2n] (uncond | cond) when cfg else [n]; coefficients from the host-side schedule.
 * t_out (optional): t_count floats set to t_next, the timestep input of the next UNet call. */
int mos_cfg_dpmpp_step(const float* noise_pred, float* latents, float* x0_prev, float* unet_in, int64_t n,
                       int32_t cfg, float guidance, float c_x, float c_m0, float c_m1, float alpha_s, float sigma_s,
                       float* t_out, int32_t t_count, float t_next, void* stream);

/* Region combine (pipeline_regionally_t2iadapter.py:54-83, replace_ratio = 1): out = global where no region
 * covers the feature pixel, else the mean of the covering regions' attention outputs. boxes_host: int32
 * [nregions, 4] = (start_h, start_w, end_h, end_w) feature-pixel indices computed by the host in float64 exactly
 * as the reference does (ceil / floor); region_ptrs_dev: device array of nregions bf16 pointers. */
int mos_region_combine(const void* glob, const void* const* region_ptrs_dev, int32_t nregions,
                       const int32_t* boxes_host, int32_t B, int32_t FH, int32_t FW, int32_t C, int64_t ld, void* out,
                       int32_t act_dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Gradient fusion in Gram form (gradient_fusion.py:22-96 update_quasi_newton / chunk_compute_mse, :99-143 merge,
 * :146-167 feature hooks).  Features are reduced on the fly to G_c = X_c^T X_c (mos_transpose_bf16 + mos_gemm_bf16
 * with MOS_OUT_F32 / accumulate, or mos_gram_small for the handful of text-token rows); a closure of the L-BFGS
 * driver is mos_sgemm_nn (Y = W G) + mos_ls_grad_loss; the driver's vector algebra uses the mos_vec_* primitives
 * (fixed reduction order -> reproducible scalars).  `scratch` >= 256 floats, `out`/`loss` 1 float, all on device.
 * ---------------------------------------------------------------------------------------------------------- */
int mos_transpose_bf16(const void* x, int64_t ldx, int32_t rows, int32_t C, void* out, int64_t ldo, void* stream);
int mos_gram_small(const float* X, int32_t n, int32_t d, float* G, int32_t accumulate, void* stream);
int mos_atb_small(const float* X, const float* Y, int32_t n, int32_t dx, int32_t dy, float* out, int32_t accumulate,
                  void* stream);
int mos_sgemm_nn(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K, float alpha, float beta,
                 void* stream);
/* closure: Y (fp64) = D (fp32) * G (fp64); grad (fp32) = 2 s (Y - R), loss (fp64) = s <D, Y - 2R> + f0 */
int mos_dgemm_mixed(const float* A, const double* B, double* C, int32_t M, int32_t N, int32_t K, void* stream);
int mos_ls_grad_loss(const float* W, const double* Y, const double* Cm, int64_t n, double s, double f0, float* grad,
                     double* loss, double* scratch, void* stream);
int mos_vec_dot(const float* a, const float* b, int64_t n, float* out, float* scratch, void* stream);
int mos_vec_asum(const float* a, int64_t n, float* out, float* scratch, void* stream);
int mos_vec_absmax(const float* a, int64_t n, float scale, float* out, float* scratch, void* stream);
int mos_vec_axpby(float* y, const float* x, float alpha, float beta, int64_t n, void* stream);
/* L-BFGS direction d = -H g by the two-loop recursion (torch.optim.LBFGS as driven by gradient_fusion.py:76-85) over k
 * curvature pairs, and gtd[0] = <g, d>, without host round trips: 2k + 1 launches, every coefficient stays in device memory.
 * S, Y: HOST arrays of k device pointers (fp32 [n], oldest pair first); rho[i] = 1 / <y_i, s_i> and h_diag = <y, s> / <y, y>
 * of the newest pair: host values.  Bit-identical to the same recursion driven from the host with mos_vec_dot /
 * mos_vec_axpby.  work: >= k + 1 doubles; partial: >= 257 floats with partial[256] == 0 on entry (left zero). */
int mos_lbfgs_direction(const void* const* S, const void* const* Y, const double* rho, int32_t k, const float* g,
                        float h_diag, int64_t n, float* d, double* work, float* partial, float* gtd, void* stream);

/* The same recursion with the history in two rings of `slots` vectors (logical pair i = physical slot (*head_dev + i) % slots
 * of S_ring / Y_ring [slots, n]); rho_dev [slots] (physical order) and hdiag_dev [1] live in device memory.  No launch
 * parameter changes between iterations with the same k: the launches can be captured once in a CUDA graph (csrc/lbfgs.cu). */
int mos_lbfgs_direction_ring(const float* S_ring, const float* Y_ring, int32_t slots, const int32_t* head_dev,
                             const double* rho_dev, const float* hdiag_dev, int32_t k, const float* g, int64_t n, float* d,
                             double* work, float* partial, float* gtd, void* stream);

/* Native driver of one per-layer fusion solve: ONE torch.optim.LBFGS.step(closure) (strong-Wolfe line search, `history` pairs,
 * at most `max_iter` iterations and max_iter * 5 / 4 closure evaluations, tolerances 1e-16 / 1e-16, lr 1: gradient_fusion.py:76-85)
 * on f(D) = s <D, D G - 2 R> + f0 from D = 0; best_D receives the iterate with the lowest loss over all evaluations
 * (gradient_fusion.py:72-74).  The loop runs on the host inside the library and issues the mos_vec_* / mos_lbfgs_direction /
 * mos_dgemm_mixed / mos_ls_grad_loss launches on `stream` (results identical to driving the same launches from the caller).
 * workspace: device memory of mos_lbfgs_workspace_bytes(out_f, in_f, history) bytes.  Blocking. */
typedef struct mos_lbfgs_problem {
  const double* G;      /* [in_f, in_f]  fp64, device */
  const double* R;      /* [out_f, in_f] fp64, device: C - W0 G */
  int32_t out_f, in_f;
  double s, f0;
  int32_t max_iter;
  int32_t history;      /* 0 = 25 */
  float* best_D;        /* out, device fp32 [out_f * in_f] */
  double* best_loss;    /* out, host (may be NULL) */
  int32_t* n_evals;     /* out, host (may be NULL) */
} mos_lbfgs_problem;
int64_t mos_lbfgs_workspace_bytes(int32_t out_f, int32_t in_f, int32_t history);
int mos_lbfgs_solve(const mos_lbfgs_problem* problem, void* workspace, void* stream);
/* The independent layers of a fusion stage: `workers` host threads, each with its own CUDA stream and workspace, take the
 * problems largest first.  Synchronises the device on entry and exit. */
int mos_lbfgs_solve_batch(const mos_lbfgs_problem* problems, int32_t n_problems, int32_t workers);
/* Batched W_l += alpha * up_l @ down_l (convert_edlora_to_diffusers.py:33-76, gradient_fusion.py:99-143).
 * table_dev: int64 [n_layers, 6] = {W fp32 ptr, down fp32 ptr, up fp32 ptr, out, in, rank}. */
int mos_lora_merge(const int64_t* table_dev, int32_t n_layers, float alpha, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fused optimiser step of ED-LoRA training (train_edlora.py:57 AdamW param groups, :129 optimizer.step, :138-140
 * Norm_mean): one flat fp32 state [concept rows | text-encoder LoRA | UNet LoRA]; group_end = exclusive end offsets
 * (host int64[3]), group_lr = host float[3]; grad_scale = 1/world after the single all-reduce (SURVEY.md §8e);
 * norm_mean_out (optional) = mean L2 norm of the first emb_rows rows of width emb_dim after the update.
 * ---------------------------------------------------------------------------------------------------------- */
int mos_flat_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                        const int64_t* group_end, const float* group_lr, float beta1, float beta2, float eps,
                        float weight_decay, int64_t step, float grad_scale, int32_t emb_rows, int32_t emb_dim,
                        float* norm_mean_out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training step (EDLoRATrainer.forward, trainer_edlora.py:202-261, + loss.backward(), train_edlora.py:120-123).
 * All base weights are frozen (trainer_edlora.py:88-90), so the backward pass only produces activation gradients
 * and the rank-4 LoRA gradients.  Linear / conv activation gradients reuse mos_gemm_bf16 on transposed weight packs.
 * ---------------------------------------------------------------------------------------------------------- */
/* forward attention that also saves lse2 [B*H, nq] (log2-domain log-sum-exp of scale*S) and, for cross-attention,
 * the per-head probabilities at key columns pos[b][0..1] -> pcols [B*H, nq, 2] (attention regulariser :263-313). */
int mos_attention_fwd_train(const void* Q, const void* K, const void* Vt, void* out, int64_t ldo, float* lse2,
                            float* pcols, const int32_t* pos, int32_t batch, int32_t heads, int32_t head_dim,
                            int32_t nq, int32_t nk, int32_t nk8, float scale, void* stream);
/* flash-attention backward.  Q, K, V, dO: head-split rows [B*H, n, DP]; Qt, Kt, dOt: transposed copies [B*H, DV, n8]
 * (mos_heads_transpose); delta from mos_attn_delta; gcols/pos (optional): gradient on the probabilities at the two
 * key columns pos[b][0..1], [B, nq, 2].  dq/dk/dv: token-major bf16 [B*n, ld] (head h in columns h*d..). */
int mos_attention_bwd(const void* Q, const void* K, const void* V, const void* dO, const void* Qt, const void* Kt,
                      const void* dOt, const float* lse2, const float* delta, const float* gcols, const int32_t* pos,
                      void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, int32_t batch,
                      int32_t heads, int32_t head_dim, int32_t nq, int32_t nk, int32_t nq8, int32_t nk8, float scale,
                      int32_t causal /* 1: keys <= query only (nq == nk; CLIP text encoder) */, void* stream);
/* dst[bh, j, r] = src[bh, r, j]: rows [BH, R, DP] -> transposed [BH, DV, R8] (dst zero-initialised by the caller). */
int mos_heads_transpose(const void* src, int32_t BH, int32_t R, int32_t DP, int32_t DV, int32_t R8, void* dst,
                        void* stream);
/* delta[bh, q] = sum_j dO[bh, q, j] O[b*N + q, h*d + j]  (+ sum_c pcols[bh, q, c] gcols[b, q, c]) */
int mos_attn_delta(const void* dO, int32_t DP, const void* O, int64_t ldo, int32_t batch, int32_t heads,
                   int32_t head_dim, int32_t N, const float* pcols, const float* gcols, float* delta, void* stream);
/* GroupNorm(32)(+SiLU) / LayerNorm backward with frozen affine: dx = J^T dy (+ add); statistics recomputed from x.
 * workspace (GroupNorm): fp32, >= B * 128 floats (more = more parallel chunks). */
int mos_groupnorm_bwd(const void* x, int64_t ldx, const void* dy, int64_t lddy, int32_t B, int32_t HW, int32_t C,
                      const float* gamma, const float* beta, float eps, int32_t silu_act, float* workspace,
                      int32_t workspace_floats, const void* add, int64_t ldadd, void* dx, int64_t lddx, void* stream);
int mos_layernorm_bwd(const void* x, int64_t ldx, const void* dy, int64_t lddy, int64_t M, int32_t C,
                      const float* gamma, float eps, const void* add, int64_t ldadd, void* dx, int64_t lddx,
                      void* stream);
/* GEGLU in un-fused form: z [M, 2H] in 160-column tiles [80 a | 80 gate] (the fused GEMM's weight-row interleave),
 * y = a * gelu(gate) [M, H]; backward writes dz in the same interleaved layout. */
int mos_geglu_fwd(const void* z, int64_t ldz, int64_t M, int32_t H, void* y, int64_t ldy, void* stream);
int mos_geglu_bwd(const void* z, int64_t ldz, const void* dy, int64_t lddy, int64_t M, int32_t H, void* dz,
                  int64_t lddz, void* stream);
/* backward of nearest x2 (sum of each 2x2 block), of the stride-2 im2col (col2im gather, optional + add) and of
 * conv_out (dy fp32 NCHW -> dx bf16 NHWC; w fp32 [Cout][9][C]). */
int mos_upsample2x_bwd(const void* dy, int64_t lddy, int32_t B, int32_t H, int32_t W, int32_t C, void* dx,
                       int64_t lddx, void* stream);
int mos_col2im_s2(const void* dcol, int32_t B, int32_t H, int32_t W, int32_t C, const void* add, int64_t ldadd,
                  void* dx, int64_t lddx, void* stream);
int mos_conv_out_bwd(const float* dy, int32_t B, int32_t H, int32_t W, int32_t C, const float* w, int32_t Cout,
                     void* dx, void* stream);
/* masked MSE (trainer_edlora.py:251-252): loss = mean_b sum_{c,hw}((pred-target)^2 mask_b) / sum_hw mask_b ;
 * dpred = grad_scale * dloss/dpred.  pred/target fp32 [B, Cc, HW], mask fp32 [B, HW]; ws >= 2B floats. */
int mos_masked_mse(const float* pred, const float* target, const float* mask, int32_t B, int32_t Cc, int32_t HW,
                   float grad_scale, float* ws, float* loss, float* dpred, void* stream);
/* DDPMScheduler.add_noise (trainer_edlora.py:218): out = sqrt(ac[t_b]) x0 + sqrt(1 - ac[t_b]) noise */
int mos_add_noise(const float* x0, const float* noise, const int32_t* timesteps, const float* alphas_cumprod,
                  int32_t B, int64_t per_sample, float* out, void* stream);
/* LoRA gradients of y = x W^T + alpha (x D^T) U^T (edlora.py:244-246):  d_up [N, 4] (+)= alpha dY^T (x D^T),
 * d_down [4, K] (+)= alpha (dY U)^T x.  x bf16 [M, K], dy bf16 [M, N], down fp32 [4, K], up fp32 [N, 4];
 * workspace >= 128 * 4 * (K + N) floats (at most 128 row slabs, one partial each); fixed-order reduction (bitwise
 * reproducible). */
int mos_lora_grad(const void* x, int64_t ldx, const void* dy, int64_t lddy, int64_t M, int32_t K, int32_t N,
                  const float* down, const float* up, float alpha, float* workspace, int64_t workspace_floats,
                  int32_t accumulate, float* d_down, float* d_up, void* stream);

/* Attention regulariser (cal_attn_reg, trainer_edlora.py:263-313) restricted to the two concept-token columns.
 * One resolution group per call: pcols_host_ptrs = host array of L device pointers [B*heads, res*res, 2] (the
 * mos_attention_fwd_train outputs of the group's layers); mask fp32 [B, 1, MH, MW]; cm [B, res*res, 2] and
 * stats[8] = {max0, max1, argmax0, argmax1, n_zero, weighted loss, S0, S1} are outputs.  mos_attn_reg_grad turns them
 * into gcols [B, res*res, 2] (the gradient on every layer/head's probabilities of the group; zero if any group of
 * stats_all [ngroups][8] is NaN, the reference's skip rule :257); mos_attn_reg_total: out[0] = mse + valid attention
 * loss, out[1] = attention loss (NaN when skipped). */
int mos_attn_reg_group(const float* const* pcols_host_ptrs, int32_t L, int32_t B, int32_t heads, int32_t res,
                       const float* mask, int32_t MH, int32_t MW, int32_t full_identity, float weight, float* cm,
                       float* stats, void* stream);
int mos_attn_reg_grad(const float* cm, const float* mask, int32_t B, int32_t res, int32_t MH, int32_t MW,
                      int32_t full_identity, float weight, const float* stats_all, int32_t ngroups, int32_t group,
                      int32_t L, int32_t heads, float grad_scale, float* gcols, void* stream);
int mos_attn_reg_total(const float* mse, const float* stats_all, int32_t ngroups, float* out, void* stream);

/* Re-pack all LoRA pairs of the flat training state into the forward / backward GEMM operand layouts after an
 * optimiser step.  table_dev: int64 [n_modules, 8] = {D fp32 [4,K] ptr, U fp32 [N,4] ptr, K, N, forward down rows
 * (bf16, 4 rows of pitch K), forward up rows (fp32 [N,4], scaled by alpha), backward "down" (bf16 [16,N], rows
 * 0..3 = U^T; may be 0), backward "up" (fp32 [K,4] = alpha D^T; may be 0)}. */
int mos_lora_pack(const int64_t* table_dev, int32_t n_modules, float alpha, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOS_SM100_H */
