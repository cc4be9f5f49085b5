/* phendiff_b200 — C ABI of the B200-native DDIM inversion + regeneration hot path.
 *
 * The reference (thethomasboyer/PhenDiff) is pure Python and has no FFI of its own; its boundary for this path is
 * the Python object protocol of SURVEY.md §8(b).  This header is the C-ABI a reference maintainer would bind
 * with ctypes from those Python objects (see INTEGRATION.md).  Every entry point cites the reference interface
 * it replaces.
 *
 * Conventions
 *   - plain C types only; all tensors are raw DEVICE pointers unless the name says "host".
 *   - the caller (PyTorch) allocates every buffer including the workspace; the library keeps no caller pointer
 *     beyond a call, except the workspace registered with pd_unet_bind_workspace and the weights, which are
 *     COPIED into library-owned, re-laid-out device buffers by pd_unet_load_weight / pd_unet_finalize.
 *   - every compute call is asynchronous on the given cudaStream_t; no hidden synchronisation.
 *   - return value: 0 = ok, non-zero = error; pd_last_error() gives the thread-local message.
 *   - a handle is bound to the CUDA device that was current at pd_unet_create and is not thread-safe
 *     (one process per GPU, like the reference).
 *   - boundary tensors are NCHW fp32 contiguous (the reference's layout); inside, activations are NHWC
 *     16-bit (PD_PREC_BF16, or PD_PREC_FP16 — the reference's own autocast type) feeding the tensor cores with fp32
 *     accumulation, or NHWC fp32 on CUDA cores (PD_PREC_FP32 validation mode).
 */
#ifndef PHENDIFF_B200_H
#define PHENDIFF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pd_unet pd_unet_t;
typedef struct pd_train pd_train_t;
typedef void* pd_stream_t; /* cudaStream_t */

enum { PD_PREC_FP32 = 0, PD_PREC_BF16 = 1, PD_PREC_FP16 = 2 };
enum { PD_PRED_EPSILON = 0, PD_PRED_SAMPLE = 1, PD_PRED_V = 2 };
#define PD_MAX_BLOCKS 8

/* Constructor arguments of CustomCondUNet2DModel (reference: src/cond_unet_2d/cond_unet_2d.py:73-107), i.e. the
 * keys of models_configs/denoiser/*.json.  Only the shipped option set is implemented natively
 * (positional time embedding, class_embed_type None, act "silu", resnet_time_scale_shift "default"). */
typedef struct pd_unet_config {
    int32_t in_channels;
    int32_t out_channels;
    int32_t n_blocks;
    int32_t block_out_channels[PD_MAX_BLOCKS];
    int32_t down_attn[PD_MAX_BLOCKS]; /* 1: AttnDownBlock2D, 0: DownBlock2D */
    int32_t up_attn[PD_MAX_BLOCKS];   /* 1: AttnUpBlock2D,   0: UpBlock2D   */
    int32_t layers_per_block;
    int32_t attention_head_dim; /* <= 0: the JSON's null = ONE head of dim C (cond_unet_2d.py:176-178) */
    int32_t norm_num_groups;
    float norm_eps;
    int32_t num_class_embeds; /* 0: no class embedding table */
    int32_t flip_sin_to_cos;
    float freq_shift;
    int32_t downsample_padding;
    float mid_block_scale_factor;
    int32_t add_attention;
    int32_t precision;       /* PD_PREC_* */
    int32_t max_microbatch;  /* images processed per pass through the layer graph (0: library default) */
    int32_t conv_impl;       /* 0: tcgen05 implicit GEMM where the shape allows (16-bit modes), 1: force SIMT kernels */
    int32_t attn_impl;       /* 0: tensor-core flash kernel (16-bit modes), 1: force SIMT kernel */
} pd_unet_config_t;

/* One scheduler update, host-computed scalars (reference: diffusers DDIMScheduler.step /
 * DDIMInverseScheduler.step as called at pipeline_conditionial_ddim.py:340-347 and utils_Img2Img.py:794-798;
 * SURVEY.md Appendix A.3-A.5):
 *   x0  = by prediction type from (x, m, sqrt_alpha, sqrt_beta);  eps likewise
 *   x0  = clamp(x0, +-clip_range) if clip;   eps = (x - sqrt_alpha*x0)/sqrt_beta if use_clipped_model_output
 *   out = sqrt_alpha_next * x0 + dir_coef * eps  (+ sigma * noise when noise != NULL)
 * where dir_coef = sqrt(1 - alpha_next - sigma^2).  IEEE semantics are kept at alpha = 0 (x0 = +-inf/NaN -> clamp). */
typedef struct pd_step_coeffs {
    int32_t pred_type; /* PD_PRED_* */
    int32_t clip;
    int32_t use_clipped_model_output;
    float clip_range;
    float sqrt_alpha;
    float sqrt_beta;
    float sqrt_alpha_next;
    float dir_coef;
    float sigma;
    float timestep; /* value fed to the UNet for this step (whole-path entry point only) */
} pd_step_coeffs_t;

const char* pd_last_error(void);
int pd_version(void);
/* launches of the opt-in cta_group::2 kernel for 1x1 layers (PHENDIFF_B200_LIN2CTA=1) since load: test support */
long long pd_debug_pair_kernel_launches(void);

/* ---- lifetime (replaces CustomCondUNet2DModel.__init__ / from_config / load_state_dict, cond_unet_2d.py:73-242,
 *      utils_models.py:158-182) ---- */
int pd_unet_create(const pd_unet_config_t* cfg, pd_unet_t** out);
int pd_unet_destroy(pd_unet_t* h);
/* parameter table in diffusers checkpoint naming (SURVEY.md Appendix A.7) */
int pd_unet_num_params(pd_unet_t* h, int32_t* n);
int pd_unet_param_info(pd_unet_t* h, int32_t idx, const char** name, int32_t* ndim, int64_t shape[4]);
/* copy one fp32 tensor (host or device pointer, contiguous, OIHW / (out,in) as in the checkpoint) */
int pd_unet_load_weight(pd_unet_t* h, const char* name, const float* data, const int64_t* shape, int32_t ndim);
/* re-layout weights for the kernels; fails if a parameter was never loaded */
int pd_unet_finalize(pd_unet_t* h, pd_stream_t stream);
int pd_unet_time_embed_dim(pd_unet_t* h, int32_t* dim);

/* ---- planning: static buffer plan for (batch, H, W); the caller then provides the workspace.
 *      The batch runs in micro-batches of `microbatch` images (pd_unet_plan_info): the largest divisor of the batch within
 *      max_microbatch (default 64) when one exists within a factor 2 of it, else even micro-batches whose ragged last one runs
 *      on padded scratch copies inside the workspace (the padding images are copies of a real image; only real outputs are
 *      written back). ---- */
int pd_unet_plan(pd_unet_t* h, int32_t batch, int32_t height, int32_t width, size_t* workspace_bytes);
int pd_unet_bind_workspace(pd_unet_t* h, void* workspace, size_t bytes);

/* ---- CustomCondUNet2DModel.forward(sample, timestep, class_labels, class_emb) (cond_unet_2d.py:244-362) ----
 * sample, out: (B,C,H,W) fp32 NCHW.  timesteps: (B,) fp32 (already broadcast, cond_unet_2d.py:276-287).
 * Exactly one of class_labels (B,) int64 / class_emb (B, time_embed_dim) fp32 is non-NULL when the model has a
 * class table; both NULL otherwise. */
int pd_unet_forward(pd_unet_t* h, const float* sample, const float* timesteps, const int64_t* class_labels,
                    const float* class_emb, float* out, pd_stream_t stream);

/* ---- DDIMScheduler.step / DDIMInverseScheduler.step on (n) elements (SURVEY A.3/A.4) ----
 * x_out and x0_out may be NULL; x_out may alias x.  noise is NULL when eta == 0. */
int pd_ddim_step(const pd_step_coeffs_t* c, const float* x, const float* model_output, const float* noise,
                 float* x_out, float* x0_out, int64_t n, pd_stream_t stream);

/* DDIMScheduler.add_noise / get_velocity (SURVEY A.3): out = ca[b]*a + cb[b]*b per sample (per_sample elements each) */
int pd_axpby_per_sample(const float* a, const float* b, const float* ca, const float* cb, float* out, int32_t batch,
                        int64_t per_sample, pd_stream_t stream);

/* classifier-free guidance combine (pipeline_conditionial_ddim.py:323-332): out = base + w[b]*(cond - uncond),
 * base = uncond ("imagen", eqn 0) or cond ("CFG", eqn 1); w is a (B,) device vector */
int pd_cfg_combine(const float* cond, const float* uncond, const float* w, int32_t eqn, float* out, int32_t batch,
                   int64_t per_sample, pd_stream_t stream);

/* pipeline post-processing (pipeline_conditionial_ddim.py:349-350): NCHW [-1,1] -> NHWC [0,1] */
int pd_denorm_nhwc(const float* x, float* out, int32_t batch, int32_t channels, int32_t height, int32_t width,
                   pd_stream_t stream);

/* ---- whole path: _ddib (utils_Img2Img.py:566-612) = _inversion (utils_Img2Img.py:763-800) + the pipeline loop
 *      (pipeline_conditionial_ddim.py:286-347) with w = 0.  steps_host: n_inv inversion steps followed by n_gen
 *      generation steps, in execution order.  x: (B,C,H,W) fp32, updated IN PLACE to the regenerated x_0'.
 *      The scheduler update of every step is fused into the conv_out kernel, so x_t is read and written once. */
int pd_ddib_transfer(pd_unet_t* h, float* x, const int64_t* src_labels, const int64_t* tgt_labels,
                     const pd_step_coeffs_t* steps_host, int32_t n_inv, int32_t n_gen, pd_stream_t stream);

/* ---- classifier-free-guided generation (SURVEY §8 row f1): the pipeline loop of pipeline_conditionial_ddim.py:286-347
 *      with guidance on, as driven by _classifier_free_guidance_forward_start (utils_Img2Img.py:615-648).  Per step ONE pass
 *      of the UNet over 2P images — P conditional samples and their P unconditional copies (class embedding = zeros,
 *      :308-317; the reference's own TODO at :287 asks for this batching) — whose conv_out epilogue combines
 *      m = (eqn == 0 ? m_u : m_c) + w (m_c - m_u) (:323-332) and applies the scheduler update to x_t in place: the guided
 *      score never exists in HBM.  Plan with pd_unet_plan_guided(h, B, H, W) (B = samples; the pass holds 2 x as many
 *      images), bind the workspace, then call.  x (B,C,H,W) fp32 updated in place; labels (B) int64; w (B) fp32 guidance
 *      scale per sample (device); eqn 0 = "imagen", 1 = "CFG"; steps_host: n_steps generation steps in execution order. */
int pd_unet_plan_guided(pd_unet_t* h, int32_t batch, int32_t height, int32_t width, size_t* workspace_bytes);
int pd_cfg_transfer(pd_unet_t* h, float* x, const int64_t* labels, const float* w, int32_t eqn,
                    const pd_step_coeffs_t* steps_host, int32_t n_steps, pd_stream_t stream);

/* ---- training step (SURVEY §8 row f2; BASELINE.json configs[3]): the inner step of perform_training_epoch for the DDIM model type
 *      (src/utils_training.py:244-456).  The caller (Python mirror phendiff_b200/training.py) samples noise and timesteps, forms the
 *      noisy images with DDIMScheduler.add_noise and the regression target by prediction type (:415-433: noise / clean images /
 *      velocity; per-sample SNR weights for "sample"); this entry point runs forward + backward of the UNet and ACCUMULATES
 *      the gradients of mean_b,chw( weight[b] * (model_out - target)^2 ).  Parameters and gradients are flat fp32 vectors in
 *      parameter-table order (pd_unet_param_info; PyTorch layouts), owned by the caller: offsets from pd_train_param_offset.
 *      labels NULL = the unconditional pass of classifier-free-guidance training (class_emb = zeros, :508-516).
 *      fp32 path: every operator of the backward pass as a CUDA-core kernel (validated against torch.autograd on the oracle). */
int pd_train_create(pd_unet_t* h, int32_t batch, int32_t height, int32_t width, pd_train_t** out);
int pd_train_destroy(pd_train_t* t);
/* precision PD_PREC_FP32 (default): fp32 on CUDA cores, the validation path.  PD_PREC_BF16: "bf16" mixed precision as accelerate runs
 * the reference (mixed_precision="bf16", train.py:57-61): convolutions (forward, dgrad, wgrad) take bf16 operands on the tcgen05 kernels
 * and attention its operands on mma.sync, with fp32 accumulation, for every shape those kernels support (the PHENDIFF_B200_TRAIN_TC
 * mask selects the pieces); everything else (GroupNorm statistics, embeddings, loss, optimizer, master weights, gradients) stays fp32.
 * PD_PREC_FP16: the same pieces with fp16 operands, as the reference's launch scripts train (accelerate --mixed_precision=fp16).  fp16
 * gradients need a loss scale (pd_train_set_loss_scale, pd_adamw_step_scaled) to stay above fp16's subnormal range.
 * Changes the workspace plan: call before pd_train_workspace_bytes / pd_train_bind. */
int pd_train_set_precision(pd_train_t* t, int32_t precision);
/* loss scale S of every following pd_train_step_grad on this handle: the backward starts from S * d(loss), so the gradients come out
 * multiplied by S (torch GradScaler.scale(loss).backward()); loss_out stays unscaled.  scale_dev: ONE fp32 on the device, read on the
 * stream when the step runs (typically &state->scale of a pd_grad_scaler_state_t); NULL (the default): 1. */
int pd_train_set_loss_scale(pd_train_t* t, const float* scale_dev);
/* convolution forward passes / weight gradients that took the tensor-core path since creation */
int pd_train_tc_counts(pd_train_t* t, int64_t* convs, int64_t* wgrads);
int pd_train_num_params_flat(pd_train_t* t, int64_t* numel);
int pd_train_param_offset(pd_train_t* t, int32_t idx, int64_t* offset);
int pd_train_workspace_bytes(pd_train_t* t, size_t* bytes);
int pd_train_bind(pd_train_t* t, void* workspace, size_t bytes);   /* 256-byte aligned, caller-owned */
/* noisy, target, model_out (optional): (B,C,H,W) fp32; timesteps (B) fp32; labels (B) int64 or NULL; sample_weight (B) fp32 or NULL;
 * loss_out: one fp32 on the device */
int pd_train_step_grad(pd_train_t* t, const float* params, float* grads, const float* noisy, const float* timesteps,
                       const int64_t* labels, const float* target, const float* sample_weight, float* loss_out, float* model_out,
                       pd_stream_t stream);
int pd_train_launch_count(pd_train_t* t, int64_t* n);

/* ---- gradient-guided generation (SURVEY §8 row f4): _custom_guided_generation (src/utils_Img2Img.py:701-760).  Per step the reference
 *      runs the UNet on images.requires_grad_(), takes x0 = scheduler.step(...).pred_original_sample, losses = Lp_loss(x0, input_images, p)
 *      (:245-270) and torch.autograd.grad(losses, images) (:741).  Here: pd_train_forward keeps the activations, pd_guidance_lp_grad
 *      turns (x_t, model output, reference images) into the per-image losses and their gradients w.r.t. the model output and (directly)
 *      w.r.t. x_t, pd_train_backward_input plays the backward pass WITHOUT parameter gradients down to the input of conv_in:
 *      grad = d_x (direct) + d_input (through the UNet).  All tensors (B,C,H,W) fp32; scratch / losses: B floats on the device. */
int pd_train_forward(pd_train_t* t, const float* params, const float* x, const float* timesteps, const int64_t* labels, float* model_out,
                     pd_stream_t stream);
int pd_train_backward_input(pd_train_t* t, const float* d_model_out, float* d_input, pd_stream_t stream);
int pd_guidance_lp_grad(const pd_step_coeffs_t* step, const float* x, const float* model_out, const float* ref, int32_t batch, int64_t per,
                        float p, float* scratch, float* losses, float* d_model_out, float* d_x, pd_stream_t stream);
/* accelerator.clip_grad_norm_(params, max_grad_norm) (utils_training.py:439; <= 0: no clipping) + torch.optim.AdamW.step
 * (train.py:279-285; `step` counts from 1) + diffusers EMAModel.step with the given decay (utils_training.py:224-241; ema NULL:
 * none) over flat fp32 vectors, in place.  scratch: PD_ADAMW_SCRATCH_FLOATS fp32 on the device (per-block partials of the gradient norm,
 * summed in a fixed order: data-parallel replicas get bit-identical clip coefficients); grad_norm_out (optional): the pre-clip global norm. */
#define PD_ADAMW_SCRATCH_FLOATS 1185
int pd_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* ema, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int32_t step, float max_grad_norm, float ema_decay, float* scratch,
                  float* grad_norm_out, pd_stream_t stream);

/* Dynamic loss scaling (torch.amp.GradScaler, what accelerate builds for mixed_precision="fp16"), kept on the device so that the training
 * step never waits for the host.  Initialise on the host (scale = init_scale, everything else 0) and copy to the device once. */
typedef struct pd_grad_scaler_state {
    float scale;              /* S: the loss scale the next backward multiplies by (GradScaler._scale) */
    int32_t growth_tracker;   /* consecutive applied steps since the last scale change (GradScaler._growth_tracker) */
    int32_t optimizer_steps;  /* AdamW steps applied: AdamW's step count (bias correction) and what LambdaLR counts */
    int32_t found_inf;        /* 1 when the last pass found an inf / NaN gradient and skipped the step */
    int32_t skipped_steps;    /* passes skipped since initialisation */
} pd_grad_scaler_state_t;
/* pd_adamw_step on loss-scaled gradients, one optimizer step of accelerate's fp16 loop: GradScaler.unscale_ (inv = 1 / S, found_inf =
 * any gradient inf or NaN, g *= inv), clip_grad_norm_ on the unscaled gradients, GradScaler.step (AdamW runs only when no gradient was
 * inf / NaN: otherwise parameters and moments stay bit-identical and the AdamW step count does not advance), GradScaler.update (found_inf:
 * S *= backoff_factor, tracker = 0; else tracker + 1, and at growth_interval S *= growth_factor if finite, tracker = 0), then the EMA
 * step, which runs on skipped steps too (toward the unchanged parameters).  grads are read, not modified.  The bias correction uses
 * state->optimizer_steps; lr applies to the step when it is not skipped.  scratch: PD_ADAMW_SCALED_SCRATCH_FLOATS fp32 on the device;
 * grad_norm_out (optional): the norm of the unscaled gradients (non-finite on a skipped step).  Deterministic: data-parallel replicas
 * with the same gradients keep bit-identical parameters and scaler state. */
#define PD_ADAMW_SCALED_SCRATCH_FLOATS 2376
int pd_adamw_step_scaled(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* ema, int64_t n, float lr,
                         float beta1, float beta2, float eps, float weight_decay, float max_grad_norm, float ema_decay,
                         pd_grad_scaler_state_t* state, float growth_factor, float backoff_factor, int32_t growth_interval,
                         float* scratch, float* grad_norm_out, pd_stream_t stream);

/* number of kernels launched by this handle since creation (bench.py's gpu_launches) */
int pd_unet_launch_count(pd_unet_t* h, int64_t* n);
/* current plan: images per pass, layers on the tcgen05 kernel / on the SIMT kernel, recorded ops per forward */
int pd_unet_plan_info(pd_unet_t* h, int32_t* microbatch, int32_t* tc_layers, int32_t* simt_layers, int32_t* ops);

/* ---- measurement support (bench.py roofline): sampled per-op device timing with CUDA events on the launch stream.
 *      Every `every_n`-th forward is bracketed op by op (at most max_samples forwards); _end synchronises those events
 *      (call it after the timed region) and accumulates per kernel class:
 *      0 conv_tcgen05, 1 conv_simt, 2 groupnorm, 3 attention, 4 embedding, 5 conv_in, 6 conv_out(+DDIM), 7 upsample. */
enum { PD_CLS_CONV_TC = 0, PD_CLS_CONV_SIMT, PD_CLS_GN, PD_CLS_ATTN, PD_CLS_EMBED, PD_CLS_CONV_IN, PD_CLS_CONV_OUT,
       PD_CLS_UPSAMPLE, PD_CLS_COUNT };
int pd_unet_profile_begin(pd_unet_t* h, int32_t every_n, int32_t max_samples);
int pd_unet_profile_end(pd_unet_t* h, int32_t* samples);
int pd_unet_profile_query(pd_unet_t* h, int32_t cls, double* ms, int64_t* launches, double* flops);
/* per recorded op (0 <= idx < ops of pd_unet_plan_info) after pd_unet_profile_end: label, class, summed ms over `samples` forwards, algorithmic FLOPs per run */
int pd_unet_profile_op(pd_unet_t* h, int32_t idx, const char** name, int32_t* cls, double* ms, int32_t* samples, double* flops);

/* ---- unit-test entry points for individual kernels (used by tests/, not by the product path) ---- */
/* generic NHWC convolution through the SIMT fp32 kernel or the tcgen05 kernel; dtype: 0 fp32, 1 bf16, 2 fp16.
 * x1 (N,H,W,C1) and optional x2 (N,H,W,C2) are channel-concatenated; w is OIHW fp32 (O, C1+C2, k, k);
 * optional sc_w (O, Csc1+Csc2) 1x1 shortcut over (sc1|sc2) accumulated into the same output;
 * addvec (N,O) fp32, residual (N,Ho,Wo,O) optional.  out (N,Ho,Wo,O). */
int pd_test_conv(int32_t use_tc, int32_t dtype, int32_t n, int32_t h, int32_t w, int32_t c1, int32_t c2,
                 int32_t cout, int32_t ksize, int32_t stride, int32_t pad, const void* x1, const void* x2,
                 const float* weight, const float* bias, const float* addvec, const void* residual,
                 const void* sc1, const void* sc2, int32_t csc1, int32_t csc2, const float* sc_w, float out_scale,
                 void* out, pd_stream_t stream);
/* extended form: impl 0 = SIMT, 1 = tcgen05 per-tap kernel, 2 = tcgen05 halo kernel.  upsample: nearest-2x + 3x3 conv run as
 * four sub-pixel phase convs (impl 2).  mode 1: conv_out epilogue (cout <= 16) writing NCHW fp32 model_out and / or updating
 * x_t in place with `step`.  stats_out (N, cout/stats_cw, 2) fp64, zero on entry, receives the GroupNorm chunk
 * statistics (sum, sum of squares over H*W of every stats_cw-channel chunk) of the stored output.  addvec_row (N) int32 or NULL. */
typedef struct pd_test_conv_args {
    int32_t impl, dtype, n, h, w, c1, c2, cout, ksize, stride, pad, upsample, mode, stats_cw, csc1, csc2;
    const void *x1, *x2;
    const float *weight, *bias, *addvec;
    const int32_t* addvec_row;
    const void* residual;
    const void *sc1, *sc2;
    const float* sc_w;
    float out_scale;
    void* out;
    double* stats_out;
    float* model_out;
    float* x_t;
    const pd_step_coeffs_t* step;
} pd_test_conv_args_t;
int pd_test_conv_ex(const pd_test_conv_args_t* args, pd_stream_t stream);
/* GroupNorm + SiLU of concat(x1, x2) fused INTO the 3x3 stride-1 convolution that consumes it (tcgen05 halo kernel, GN variant:
 * the normalised tensor exists only as shared-memory tiles).  Same optional epilogue inputs as pd_test_conv_ex; dtype 1 / 2.
 * Replaces the norm1/nonlinearity/conv1 and norm2/nonlinearity/conv2 pairs of diffusers ResnetBlock2D (SURVEY A.1). */
int pd_test_gn_conv(int32_t dtype, int32_t n, int32_t h, int32_t w, int32_t c1, int32_t c2, int32_t cout, int32_t groups, float eps,
                    const void* x1, const void* x2, const float* gamma, const float* beta, const float* weight, const float* bias,
                    const float* addvec, const void* residual, const void* sc1, const void* sc2, int32_t csc1, int32_t csc2,
                    const float* sc_w, float out_scale, void* out, double* stats_out, pd_stream_t stream);
/* GroupNorm(+SiLU) over NHWC, two concatenated sources */
int pd_test_groupnorm(int32_t dtype, int32_t n, int32_t hw, int32_t c1, int32_t c2, int32_t groups, float eps,
                      int32_t do_silu, const void* x1, const void* x2, const float* gamma, const float* beta,
                      void* out, pd_stream_t stream);
/* self-attention core on packed qkv (N, S, 3C) -> (N, S, C), head_dim d.  use_mma: 0 = SIMT kernel, 1 = tensor-core kernel on
   raw q, 2 = tensor-core kernel on q already multiplied by log2(e)/sqrt(d) (what pd_unet_finalize folds into the q rows of
   the fused qkv projection, so that scores leave the MMA in log2 units); 3 / 4 / 5 = as 2 but forcing the chunked warp-level /
   head-resident warp-level / tcgen05 kernel */
int pd_test_attention(int32_t use_mma, int32_t dtype, int32_t n, int32_t s, int32_t c, int32_t d, const void* qkv,
                      void* out, pd_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PHENDIFF_B200_H */
