/* fdx.h -- C-ABI of libfdx.so, the B200 (sm_100a) kernel library under the
 * flaxdiff_b200 Python surface.
 *
 * The reference (AshishKumar4/FlaxDiff) has no FFI / plugin interface: every device
 * op on its UNet hot path is a flax.linen / jax.numpy call lowered by XLA.  Each entry
 * point below names the reference call site (file:line under /root/reference) whose
 * XLA lowering it replaces.  Conventions:
 *   - plain pointers + sizes, caller-owned DEVICE buffers, no hidden allocation;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it;
 *   - return 0 on success, <0 on error (fdx_last_error() gives the message);
 *   - activations are NHWC bf16 unless stated, described by fdx_act (a pixel stride
 *     larger than c lets producers write straight into channel slots of a concat
 *     buffer: jnp.concatenate at flaxdiff/models/simple_unet.py:145,196 is free);
 *   - conv kernels are HWIO [3][3][Cin][Cout] exactly as flax stores them.
 */
#ifndef FDX_H_
#define FDX_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDX_OK 0
#define FDX_ERR_INVALID_ARG (-1)
#define FDX_ERR_UNSUPPORTED (-2)
#define FDX_ERR_CUDA (-3)
#define FDX_ERR_NO_DEVICE (-4)

typedef struct fdx_act {
  void* ptr;            /* device pointer to element (n=0,y=0,x=0,c=0) */
  int n, h, w, c;       /* logical dims */
  long long pix_stride; /* elements between consecutive pixels (>= c, multiple of 8) */
} fdx_act;

/* ---- library ---------------------------------------------------------------- */
const char* fdx_last_error(void);
int fdx_version(void);
int fdx_device_sm_count(void);
/* number of libfdx kernels launched (or captured into a CUDA graph) by this process so far */
unsigned long long fdx_launch_count(void);
/* tensor-core kernel family of the most recent launch (-1 = none yet) and its SASS-visible kernel name: lets a
 * profiler attribute a CUDA-event interval around one C-ABI call to the kernel that ran (bench.py roofline). */
#define FDX_KERNEL_TC 0       /* fdx_tc_kernel: pixels-as-M tap-GEMM engine */
#define FDX_KERNEL_TCT 1      /* fdx_tct_kernel: transposed (weights-as-M) engine */
#define FDX_KERNEL_WGRAD9K 2  /* fdx_wgrad9k_kernel: nine-tap weight gradient, ky pairs in M / kx in N */
#define FDX_KERNEL_WGRAD9 3   /* fdx_wgrad9_kernel: round-1 nine-tap weight gradient */
#define FDX_KERNEL_CONV3 4    /* fdx_conv3_kernel: halo-sharing forward (opt-in) */
#define FDX_KERNEL_ATTN_FWD 5 /* fdx_attn_fwd_kernel: fused attention forward */
#define FDX_KERNEL_ATTN_BWD 6 /* fdx_attn_bwd_kernel: fused attention backward */
int fdx_last_kernel_kind(void);
const char* fdx_kernel_kind_name(int kind);

/* ---- tensor-core contractions (tcgen05 + TMA + TMEM) ------------------------- */
/* flax nn.Conv 3x3 SAME, stride 1 or 2 (models/common.py:166-172, 237-244).
 * y = conv(x, w) + bias + rowvec[n] + res ; bias [Cout] f32, rowvec [N][Cout] f32 (the
 * ResidualBlock's `out + temb` add, common.py:300-308), res = residual add (common.py:334).
 * w_hwio is bf16.  Cin, Cout multiples of 64. */
int fdx_conv3x3_fwd(const fdx_act* x, const void* w_hwio, const float* bias, const float* rowvec,
                    const fdx_act* res, const fdx_act* y, int stride, void* stream);
/* Same convolution, additionally accumulating per (image, output channel) the sum and the sum of
 * squares of the stored bf16 values - the statistics of the GroupNorm that consumes y
 * (models/common.py:273-288), so that norm needs no pass of its own over y.
 * cs->ws = f32 [slots][N][2][ld], zeroed by the caller, pre-offset to y's first channel inside the
 * destination buffer (ld = that buffer's channel count).  FDX_ERR_UNSUPPORTED when an image of y has
 * fewer than 128 pixels.  fdx_groupnorm_stats_from_cols turns the sums into fdx_groupnorm_stats' output. */
typedef struct fdx_colstats {
  float* ws;
  int slots;
  int ld;
} fdx_colstats;
int fdx_conv3x3_fwd_stats(const fdx_act* x, const void* w_hwio, const float* bias, const float* rowvec,
                          const fdx_act* res, const fdx_act* y, int stride, const fdx_colstats* cs,
                          void* stream);
int fdx_groupnorm_stats_from_cols(const float* cols, int slots, int N, int ld, int c0, int C, int groups,
                                  float* stats, void* stream);   /* channels [c0, c0+C) of the ld-wide rows */
/* d(loss)/dx of the conv above (jax.value_and_grad, trainer/general_diffusion_trainer.py:321). */
int fdx_conv3x3_dgrad(const fdx_act* dy, const void* w_hwio, const fdx_act* dx, int stride,
                      int accumulate, void* stream);
/* d(loss)/dw, f32 HWIO, ACCUMULATED into dw_hwio (caller zeroes it). */
int fdx_conv3x3_wgrad(const fdx_act* x, const fdx_act* dy, float* dw_hwio, int stride,
                      void* stream);

/* 1x1 convolution in convolution geometry (ResidualBlock.residual_conv, models/common.py:324-333):
 * y = x W + bias + res with W = [Cin][Cout] bf16 (flax (1,1,Cin,Cout) kernel), and its data gradient
 * dx (+)= dy W^T.  Same arithmetic as fdx_gemm on the flattened pixels, but eligible for the transposed
 * engine (few output columns, one or two K chunks: epilogue / bandwidth bound layers). */
int fdx_conv1x1_fwd(const fdx_act* x, const void* w_io, const float* bias, const fdx_act* res, const fdx_act* y,
                    void* stream);
int fdx_conv1x1_dgrad(const fdx_act* dy, const void* w_io, const fdx_act* dx, int accumulate, void* stream);

#define FDX_GEMM_KK 0   /* D[m][n] = sum_k A[m][k] * B[n][k]   (both k-contiguous)   */
#define FDX_GEMM_KMN 1  /* D[m][n] = sum_k A[m][k] * B[k][n]                          */
#define FDX_GEMM_MNMN 2 /* D[m][n] = sum_k A[k][m] * B[k][n]   (weight-gradient type) */
typedef struct {
  int mode;
  int M, N, K;
  int batch1, batch2;      /* two batch dims (e.g. heads, images); 0/1 = none */
  const void* A; long long a_ld, a_s1, a_s2; /* bf16; leading dim and batch strides, elements */
  const void* B; long long b_ld, b_s1, b_s2; /* bf16; b_s1 = b_s2 = 0 -> B shared by the batch */
  void* D; long long d_ld, d_s1, d_s2;
  int d_f32;               /* output dtype: 0 bf16, 1 f32 */
  int d_atomic;            /* f32 atomicAdd into D (split-K allowed) */
  int reduce_batch;        /* MNMN only: also reduce over the batch dims (dense weight grads) */
  float alpha;
  const float* bias;       /* [N] or NULL */
  const void* res; long long r_ld, r_s1, r_s2; /* bf16 residual added to D, or NULL */
} fdx_gemm_desc;
/* 1x1 conv (common.py:324-333), nn.DenseGeneral (attention.py:132-154, common.py:300-305),
 * and the QK^T / PV / backward products of nn.dot_product_attention (attention.py:170-174). */
int fdx_gemm(const fdx_gemm_desc* g, void* stream);

/* Upsample = jax.image.resize(nearest, x2) + ConvLayer 3x3 (models/common.py:210-226) without materialising
 * the upsampled tensor: four output parities, each a 2x2 convolution of the LOW-resolution input with
 * summed taps (4/9 of the FLOPs).  x / dx are the low-resolution tensors, y / dy the full-resolution ones.
 *   fdx_upconv3x3_pack  : weff bf16 [4 parities][2][2][Cin][Cout] from the f32 HWIO master weights
 *   fdx_upconv3x3_fwd   : y = conv3x3(nearest2x(x)) + bias
 *   fdx_upconv3x3_dgrad : dx (+)= d/dx, one 16-tap launch
 *   fdx_upconv3x3_wgrad : dw_hwio += d/dw; dweff_ws = f32 scratch of 16*Cin*Cout floats */
int fdx_upconv3x3_pack(const float* w_hwio, int cin, int cout, void* weff_bf16, void* stream);
int fdx_upconv3x3_fwd(const fdx_act* x, const void* weff_bf16, const float* bias, const fdx_act* y,
                      void* stream);
int fdx_upconv3x3_fwd_stats(const fdx_act* x, const void* weff_bf16, const float* bias, const fdx_act* y,
                            const fdx_colstats* cs, void* stream);   /* cs as in fdx_conv3x3_fwd_stats */
int fdx_upconv3x3_dgrad(const fdx_act* dy, const void* weff_bf16, const fdx_act* dx, int accumulate,
                        void* stream);
int fdx_upconv3x3_wgrad(const fdx_act* x, const fdx_act* dy, float* dweff_ws, float* dw_hwio,
                        void* stream);

/* ---- normalisation (HBM-bound; warp-shuffle + shared/global atomics reductions) ---- */
/* nn.GroupNorm(groups, eps) statistics (models/common.py:273-281): stats[n][g] = (sum, sumsq), f32. */
int fdx_groupnorm_stats(const fdx_act* x, int groups, float* stats, void* stream);
/* y = silu?((x-mean)*rstd*gamma+beta) (models/common.py:286-288,310-312; simple_unet.py:209-210). */
int fdx_groupnorm_apply(const fdx_act* x, int groups, const float* stats, const float* gamma,
                        const float* beta, float eps, int silu, const fdx_act* y, void* stream);
/* fdx_groupnorm_apply with the statistics taken straight from the producers' epilogue column sums
 * (cols = [slots][N][2][ld] as written by fdx_conv3x3_fwd_stats / fdx_upconv3x3_fwd_stats, channels c0 .. c0+C of
 * the buffer): no fdx_groupnorm_stats_from_cols launch; stats_out[N][groups][2] receives the statistics for the
 * backward. */
int fdx_groupnorm_apply_cols(const fdx_act* x, int groups, const float* cols, int slots, int ld, int c0,
                             const float* gamma, const float* beta, float eps, int silu, const fdx_act* y,
                             float* stats_out, void* stream);
/* Backward of the pair above.  ws: f32 scratch of at least 2*N*groups floats (a larger buffer is fine; only
 * the first 2*N*groups are used).  dgamma/dbeta ACCUMULATED.
 * csum_img [n][c] / csum_tot [c] (NULL allowed; csum_tot needs csum_img): column sums over pixels of the
 * dx this call produces, written (not accumulated) - the timestep row-vector and conv-bias gradients. */
int fdx_groupnorm_bwd(const fdx_act* x, const fdx_act* dy, int groups, const float* stats,
                      const float* gamma, const float* beta, float eps, int silu, float* ws,
                      float* dgamma, float* dbeta, const fdx_act* dx, int accumulate,
                      float* csum_img, float* csum_tot, void* stream);
/* Same, with the result ADDED to another tensor: dx = d/dx + addend (addend may be dx itself = accumulate).  The
 * ResidualBlock's skip gradient (common.py:334-336: out + residual) joins here instead of in a separate pass. */
int fdx_groupnorm_bwd_add(const fdx_act* x, const fdx_act* dy, int groups, const float* stats,
                          const float* gamma, const float* beta, float eps, int silu, float* ws,
                          float* dgamma, float* dbeta, const fdx_act* dx, const fdx_act* addend,
                          float* csum_img, float* csum_tot, void* stream);
/* Fused variant of the backward above: the data-gradient convolution that PRODUCES dy applies
 * silu'(z) in its epilogue and accumulates the first-pass sums, so x and dy are read once less.
 *   fdx_groupnorm_coeffs : ab[n][0][c] = rstd*gamma_c, ab[n][1][c] = beta_c - mean*rstd*gamma_c
 *   fdx_conv3x3_dgrad_gn : stride-1 3x3 data gradient (as fdx_conv3x3_dgrad) writing
 *                          dz = dgrad * silu'(a x + b) and ws_slots[slot][n][{0,1}][c] += (sum dz, sum dz*x);
 *                          zeroes ws_slots (slots*N*2*C floats) itself; FDX_ERR_UNSUPPORTED when an image
 *                          has fewer than 128 pixels (caller then uses the two-pass path)
 *   fdx_groupnorm_bwd_dz : second pass from dz, one launch; ws is not read (NULL allowed, kept for
 *                          signature compatibility). */
int fdx_groupnorm_coeffs(const float* stats, const float* gamma, const float* beta, int N, int HW, int C,
                         int groups, float eps, float* ab, void* stream);
int fdx_conv3x3_dgrad_gn(const fdx_act* dy, const void* w_hwio, const fdx_act* dz, const fdx_act* x,
                         const float* ab, float* ws_slots, int slots, void* stream);
int fdx_groupnorm_bwd_dz(const fdx_act* x, const fdx_act* dz, int groups, const float* stats,
                         const float* gamma, float eps, const float* ws_slots, int slots, float* ws,
                         float* dgamma, float* dbeta, const fdx_act* dx, int accumulate, float* csum_img,
                         float* csum_tot, void* stream);
/* fdx_groupnorm_bwd_dz with dx = GroupNorm backward + addend (the identity-residual gradient of the
 * ResidualBlock, flaxdiff/models/common.py:334-336), as fdx_groupnorm_bwd_add. */
int fdx_groupnorm_bwd_dz_add(const fdx_act* x, const fdx_act* dz, int groups, const float* stats,
                             const float* gamma, float eps, const float* ws_slots, int slots, float* ws,
                             float* dgamma, float* dbeta, const fdx_act* dx, const fdx_act* addend,
                             float* csum_img, float* csum_tot, void* stream);
/* nn.RMSNorm(eps) over channels (models/attention.py:325-326). C a multiple of 8, <= 1024. */
int fdx_rmsnorm_fwd(const fdx_act* x, const float* scale, float eps, const fdx_act* y,
                    void* stream);
int fdx_rmsnorm_bwd(const fdx_act* x, const fdx_act* dy, const float* scale, float eps,
                    const fdx_act* dx, int accumulate, float* dscale, void* stream);

/* ---- diffusion step streaming kernels ------------------------------------------------ */
/* (x-127.5)/127.5, x_t = alpha*x0 + sigma*eps, target, model input bf16(x_t*c_in)
 * (trainer/general_diffusion_trainer.py:258,285-291; predictors/__init__.py:19-24).
 * target_kind: 0 = x0, 1 = eps, 2 = v.  E = elements per sample. */
int fdx_diffuse_forward(const void* x0, int x0_is_u8, const float* eps, const float* alpha,
                        const float* sigma, const float* c_in, int B, long long E, int normalize,
                        int target_kind, float* x_t, float* target, void* model_in_bf16,
                        void* stream);
/* pred = c_out*F + c_skip*x_t; loss = mean(0.5*(pred-target)^2*w); dF = dloss/dF
 * (general_diffusion_trainer.py:295-302; predictors/__init__.py:84-91). */
int fdx_loss_fwd_bwd(const float* F, const float* x_t, const float* target, const float* c_out,
                     const float* c_skip, const float* weight, int B, long long E,
                     float* loss_sum, float* dF, void* stream);
/* out1 = sum_i coef1[i][b]*in_i ; out2 = sum_i coef2[i][b]*in_i ; out_bf16 = bf16(out1*scale[b]).
 * One pass for x0/eps recovery, CFG mixing (samplers/common.py:93-96) and every sampler update
 * (samplers/euler.py:8-18,39-56; heun_sampler.py:7-27; ddim.py:30-47; ddpm.py:6-15). */
int fdx_affine_combine(int n_in, const float* const* inputs, const float* coef1, const float* coef2,
                       const float* bf16_scale, int B, long long E, float* out1, float* out2,
                       void* out_bf16, int clip, float clip_lo, float clip_hi, void* stream);
/* ---- optimiser / EMA / loss scaling over ONE flat f32 buffer (fdx_optim.cu) -------------------- */
/* optax.adam / adamw / lamb (+ optax.clip_by_global_norm) as flax TrainState.apply_gradients does them
 * (training.py:263-267,594-608; trainer/general_diffusion_trainer.py:311,327), fused with
 * TrainState.apply_ema (trainer/diffusion_trainer.py:31-37) and the refresh of the bf16 weight shadow the
 * tensor-core kernels read.  `ema` NULL = apply_gradients only.  The gradient the update sees is
 *   g * grad_scale [/ dynscale[0]] * min(1, clip_norm / ||.||)          (||.|| from gstats[0])
 * and with `dynscale` set the parameter / moment update is SKIPPED when gstats[1] > 0 (non-finite gradients,
 * general_diffusion_trainer.py:313-318) while the EMA still runs on the unchanged parameters.
 * lamb: seg_offsets = the nseg tensor start offsets (elements, ascending, first = 0, multiples of 4),
 * seg_norms = f32 [nseg][2] scratch, u_ws = f32 [n] scratch (optax.scale_by_trust_ratio is per tensor). */
#define FDX_OPT_ADAM 0 /* adam (weight_decay = 0) and adamw */
#define FDX_OPT_LAMB 1
typedef struct fdx_opt_desc {
  int kind;
  float* p; const float* g; float* m; float* v;
  float* ema;               /* or NULL */
  void* shadow_bf16;        /* or NULL */
  long long n;              /* multiple of 4 */
  float lr, b1, b2, eps, weight_decay;
  int step;                 /* optimiser count after this step (>= 1): bias corrections */
  float ema_decay;
  float grad_scale;         /* e.g. 1/world after a sum all-reduce; 1 otherwise */
  const float* gstats;      /* device f32[2] from fdx_grad_stats, or NULL */
  float clip_norm;          /* 0 = no clipping */
  const float* dyn_lr_bc;   /* device {lr, 1-b1^t, 1-b2^t} overriding lr/step (CUDA-graph replay), or NULL */
  const float* dynscale;    /* device DynamicScale state {scale, fin_steps, last_finite}, or NULL */
  const long long* seg_offsets; int nseg; float* seg_norms; float* u_ws;   /* lamb only */
} fdx_opt_desc;
int fdx_optimizer_step(const fdx_opt_desc* d, void* stream);
/* adamw + EMA + shadow, the common case, without the descriptor (gnorm_sq = fdx_grad_stats output). */
int fdx_adamw_ema_step(float* p, const float* g, float* m, float* v, float* ema, void* shadow_bf16,
                       long long n, float lr, float b1, float b2, float eps, float weight_decay,
                       int step, float ema_decay, float grad_scale, const float* gnorm_sq,
                       float clip_norm, const float* dyn_lr_bc /* device {lr,1-b1^t,1-b2^t} or NULL */,
                       void* stream);
/* TrainState.apply_ema on its own: ema = decay*ema + (1-decay)*p (trainer/diffusion_trainer.py:31-37). */
int fdx_ema_update(float* ema, const float* p, long long n, float decay, void* stream);
/* out2[0] = sum g^2 (optax.clip_by_global_norm), out2[1] = number of non-finite elements (DynamicScale's
 * is_finite, flax/training/dynamic_scale.py via general_diffusion_trainer.py:308).  fdx_sumsq = same call. */
int fdx_grad_stats(const float* g, long long n, float* out2, void* stream);
int fdx_sumsq(const float* g, long long n, float* out2, void* stream);
/* DynamicScale state update after a step: state3 = {scale, fin_steps, last_finite}; finite: after
 * growth_interval finite steps scale *= growth_factor; non-finite: scale = max(scale*backoff, minimum). */
int fdx_dynscale_update(float* state3, const float* gstats, float growth_factor, float backoff_factor,
                        int growth_interval, float minimum_scale, void* stream);

/* ---- data-parallel exchange (fdx_comm.cu): jax.lax.pmean of the gradients and the loss ---------------
 * (trainer/general_diffusion_trainer.py:325,334,340-345).  NCCL is bound at run time (dlopen); one
 * communicator per process, one process per GPU.  fdx_comm_allreduce_avg is asynchronous on `stream` and
 * may be called on sub-ranges ("buckets") of the flat gradient buffer while the backward pass still runs. */
typedef struct fdx_comm fdx_comm;
int fdx_comm_unique_id(void* id128 /* 128 bytes out; rank 0 creates it, every rank passes it to init */);
int fdx_comm_init(fdx_comm** out, int rank, int world, const void* id128);
int fdx_comm_allreduce_avg(fdx_comm* c, float* buf, long long n, void* stream);   /* in place, mean over ranks */
int fdx_comm_world(const fdx_comm* c, int* rank, int* world);
int fdx_comm_nccl_version(void);      /* 0 when NCCL cannot be bound */
int fdx_comm_destroy(fdx_comm* c);
int fdx_cast_f32_bf16(const float* src, void* dst, long long n, void* stream);
/* jax.image.resize(nearest) x2 (models/common.py:214-215) and its adjoint. */
int fdx_upsample2x(const fdx_act* x, const fdx_act* y, void* stream);
int fdx_upsample2x_bwd(const fdx_act* dy, const fdx_act* dx, int accumulate, void* stream);
int fdx_act_add(const fdx_act* a, const fdx_act* b, const fdx_act* out, void* stream);
/* column sums over pixels: out[c] or out[n][c] (bias / timestep-vector gradients). */
int fdx_colsum(const fdx_act* x, float* out, int per_image, void* stream);

/* ---- 3-channel convolutions (CUDA cores) ----------------------------------------------- */
/* conv_in 3->Cout (models/simple_unet.py:47-54): x bf16 [N,H,W,3] dense, w f32 HWIO. */
int fdx_conv_in_fwd(const void* x_bf16, int N, int H, int W, const float* w_hwio,
                    const float* bias, const fdx_act* y, void* stream);
int fdx_conv_in_wgrad(const void* x_bf16, const fdx_act* dy, float* dw_hwio, float* dbias,
                      void* stream);
/* im2col of a 3-channel tensor for the two weight gradients above/below as tensor-core GEMMs:
 * col[p][t*3+k] = src[p + sgn*d(t)][k] (zero outside the image), bf16 [N*H*W][32]; column 27 = 1 if
 * ones_col (bias row).  dW_in = col^T dY ; dW_out = x^T col (via fdx_gemm MNMN). */
int fdx_im2col3x3_c3(const void* src, int src_is_f32, int sgn, int N, int H, int W, int ones_col,
                     void* col_bf16, void* stream);
/* Scatter step of the tensor-core conv_out (models/simple_unet.py:212-221): col f32 [N*H*W][32] holds
 * <x[p], w[t][:][k]> at column t*3+k; y[p][k] = bias[k] + sum_t col[p + d(t)][t*3+k], SAME padding. */
int fdx_col2im3x3_c3(const float* col_f32, const float* bias, int N, int H, int W, float* y_f32,
                     void* stream);
/* conv_out Cin->3 (models/simple_unet.py:212-221): y f32 [N,H,W,3] dense. */
int fdx_conv_out_fwd(const fdx_act* x, const float* w_hwio, const float* bias, float* y_f32,
                     void* stream);
int fdx_conv_out_dgrad(const float* dF, const float* w_hwio, const fdx_act* dx, void* stream);
int fdx_conv_out_wgrad(const fdx_act* x, const float* dF, float* dw_hwio, float* dbias,
                       void* stream);

/* ---- timestep embedding + softmax ------------------------------------------------------ */
/* FourierEmbedding + TimeProjection (models/common.py:97-124), f32; saves four/h1/h2 for bwd. */
int fdx_time_embed_fwd(const float* t, const float* freqs, const float* W1, const float* b1,
                       const float* W2, const float* b2, int B, int D, float* four, float* h1,
                       float* h2, float* emb, void* emb_bf16, void* stream);
int fdx_time_embed_bwd(const float* demb, const float* four, const float* h1, const float* h2,
                       const float* W2, int B, int D, float* dh1_ws, float* dh2_ws, float* dW1,
                       float* db1, float* dW2, float* db2, void* stream);
/* softmax of nn.dot_product_attention (models/attention.py:170-174): S f32 -> P bf16.  Rows hold Lp
 * columns of which the first L are real keys (cross-attention to 77 text tokens is padded to 96). */
int fdx_softmax_fwd(const float* S, long long rows, int L, int Lp, void* P_bf16, void* stream);
int fdx_softmax_bwd(const void* P_bf16, const float* dP, long long rows, int L, int Lp, float scale,
                    void* dS_bf16, void* stream);

/* FlaxGEGLU of the full transformer block (models/attention.py:179-205): u bf16 [rows][2*inner] =
 * [hidden_linear | hidden_gelu] -> g = hidden_linear * gelu_tanh(hidden_gelu) bf16 [rows][inner], and its
 * backward du [rows][2*inner] from dg.  inner a multiple of 8. */
int fdx_geglu_fwd(const void* u_bf16, long long rows, int inner, void* g_bf16, void* stream);
int fdx_geglu_bwd(const void* u_bf16, const void* dg_bf16, long long rows, int inner, void* du_bf16,
                  void* stream);

/* ---- fused attention (fdx_attn.cu) ------------------------------------------------------------------
 * nn.dot_product_attention inside NormalAttention (models/attention.py:156-177): o = softmax(q k^T * scale) v
 * per (image, head), self-attention (Lk = L) or cross-attention to the text context (Lk = 77), and its
 * backward under jax.value_and_grad (trainer/general_diffusion_trainer.py:321).  The logits and probabilities
 * never reach HBM: flash-style tcgen05 kernels with S / P in TMEM / shared memory; the backward recomputes
 * them from `lse` (two kernels: dQ per query tile, dK + dV per key block; deterministic, no atomics).
 * Tensors: bf16 [B][rows][heads*dh], `*_ld` = elements between rows, `*_bs` = elements between images;
 * dh (as STORED) is 32 or 64 - narrower heads are zero-padded by the caller, `scale` = 1/sqrt(true width).
 * lse: f32 [B][heads][L] (written by fwd, read by bwd); dvec_ws: f32 [B][heads][L] scratch (bwd). */
typedef struct fdx_attn_desc {
  int B, heads, L, Lk, dh;
  float scale;
  const void* q; long long q_ld, q_bs;
  const void* k; long long k_ld, k_bs;
  const void* v; long long v_ld, v_bs;
  void* o; long long o_ld, o_bs;          /* fwd: output; bwd: the saved forward output (input) */
  float* lse;
  /* backward only */
  const void* d_o; long long do_ld, do_bs;
  float* dvec_ws;
  void* dq; long long dq_ld, dq_bs;
  void* dk; long long dk_ld, dk_bs;
  void* dv; long long dv_ld, dv_bs;
} fdx_attn_desc;
int fdx_attention_fwd(const fdx_attn_desc* a, void* stream);
int fdx_attention_bwd(const fdx_attn_desc* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FDX_H_ */
