// phendiff_b200 — launch interface of the training-step kernels (pd_train_kernels.cu), used by the driver in pd_train.cu.
#pragma once
#include "pd_common.cuh"
#include <string>

namespace pd {

struct WgradArgs {
    const float *x1, *x2;     // NHWC fp32 sources of the conv input (channel concat), x2 may be null
    int C1, C2, N, H, W, Cout, ksize, stride, pad, Ho, Wo;
    const float* dy;          // (N, Ho, Wo, Cout)
    float* dw;                // OIHW (Cout, C1 + C2, k, k), accumulated
    float scale;
    int Iw;                   // I dimension of dw (input channels >= Iw are padding and skipped); 0: C1 + C2
    int dy_pitch;             // row pitch of dy in floats; 0: Cout
    int chunk;                // pixels per CTA (set by the launcher)
};
int launch_conv_wgrad(const WgradArgs& a, cudaStream_t s);
int launch_relayout_dgrad(const float* w, int O, int I, int k, int i0, int Isub, float* out, cudaStream_t s);
int launch_colsum(const float* dy, int M, int C, int rows_per_seg, float scale, float* out, cudaStream_t s, int Cvalid = 0);
int launch_add_bias_rows(float* x, const float* bias, int B, int D, cudaStream_t s);
int launch_conv_dgrad_gather(const float* dy, int dy_pitch, const float* w, int N, int H, int W, int C, int Ho, int Wo, int Cout, int pad,
                             int stride, float* dx, cudaStream_t s);
int launch_upsample2x_bwd(const float* dy, int N, int H, int W, int C, float* dx, cudaStream_t s);

struct GNBwdArgs {
    const float *x1, *x2;     // GroupNorm input (concat), NHWC fp32
    float *dx1, *dx2;         // accumulated
    const void* dy;           // (N, HW, C1 + C2) gradient w.r.t. the (activated) output: fp32, or 16-bit when dy_dt says so
    int C1, C2, N, HW, groups, silu, stats_cw;
    float eps, scale;
    const float *gamma, *beta;
    float *dgamma, *dbeta;    // accumulated
    const double *stats1, *stats2;   // chunk statistics of the inputs (forward)
    float* gsum;              // scratch (N, groups, 2)
    int dy_dt;                // DT_F32 (0, default) or the 16-bit type `dy` is stored in (written by a tensor-core dgrad)
};
int launch_gn_bwd(const GNBwdArgs& a, cudaStream_t s);
// forward of the mixed-precision path: fp32 sources -> 16-bit output only (uses x1/x2, C1/C2, N, HW, groups, silu, eps, gamma, beta, stats)
int launch_gn_apply16(int dt, const GNBwdArgs& a, void* out, cudaStream_t s);
int launch_nchw_to_nhwc16_pad(int dt, const float* x, int N, int C, int HW, int Cp, void* out, cudaStream_t s);

// q, k, v: (N, S, pitch)-strided rows with the head's 8 values at head * 8 (packed qkv: pitch 3C, k = q + C, v = q + 2C)
int launch_attn8_fwd(const float* q, const float* k, const float* v, int pitch, int N, int S, int C, float* out, float* lse, cudaStream_t s);
int launch_attn8_bwd(const float* q, const float* k, const float* v, int pitch, const float* o, const float* dout, const float* lse, int N,
                     int S, int C, float* dq, float* dk, float* dv, float* delta, cudaStream_t s);

// C[M, N] (+)= alpha * op(A) op(B); ta: A is stored (K, M); tb: B is stored (N, K)
int launch_sgemm(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                 int accumulate, cudaStream_t s);
int launch_sinusoid(const float* t, int B, int C0, int flip, float shift, float* out, cudaStream_t s);
int launch_bias_silu_fwd(float* pre, const float* bias, const float* table, const int64_t* labels, int B, int D, float* act, cudaStream_t s);
int launch_silu_bwd(const float* pre, const float* dact, size_t total, float* dpre, cudaStream_t s);
int launch_scatter_rows(const float* d, const int64_t* labels, int B, int D, float scale, float* table_grad, cudaStream_t s);
int launch_nchw_to_nhwc_pad(const float* x, int N, int C, int HW, int Cp, float* out, cudaStream_t s);
int launch_add_inplace(float* y, const float* x, float alpha, size_t n, cudaStream_t s);
// dm is the gradient of the loss times *loss_scale (NULL: 1); the loss itself is never scaled
int launch_mse_loss(const float* m, const float* target, const float* weight, int B, size_t per, const float* loss_scale, float* loss, float* dm,
                    cudaStream_t s);
int launch_adamw(float* p, const float* g, float* m, float* v, float* ema, size_t n, float lr, float b1, float b2, float eps, float wd,
                 int step, float max_norm, float ema_decay, float* scratch_sumsq, float* norm_out, cudaStream_t s);
// the same on loss-scaled gradients with torch.amp.GradScaler's unscale / skip-on-inf / scale update; scaler state on the device
int launch_adamw_scaled(float* p, const float* g, float* m, float* v, float* ema, size_t n, float lr, float b1, float b2, float eps, float wd,
                        float max_norm, float ema_decay, pd_grad_scaler_state_t* state, float growth, float backoff, int interval,
                        float* scratch, float* norm_out, cudaStream_t s);

// gradient-guided generation (f4): loss_i = || pred_original_sample(x, m) - ref ||_p per image and its gradients w.r.t. m and (directly) x
int launch_guidance_lp_grad(const pd_step_coeffs_t& c, const float* x, const float* m, const float* ref, int B, size_t per, float p, float* sums,
                            float* losses, float* dm, float* dx, cudaStream_t s);
int launch_nhwc_to_nchw_f32(int dt, const void* x, int N, int C, int HW, int Cp, float* out, cudaStream_t s);

// ---- mixed-precision path (bf16 tensor-core convolutions; pd_train_wgrad_tc.cu) -------------------------------------------------
int launch_relayout_tc_dgrad(int dt, const float* w, int O, int I, int k, int i0, int Isub, void* out, cudaStream_t s, int ktot = 0, int koff = 0,
                             int ostride = 0);
int launch_f2h(int dt, const float* x, void* out, size_t n, cudaStream_t s);
int launch_h2f_epilogue(int dt, const void* y16, const float* addvec, const float* residual, float scale, float* out, int B, int HW, int C,
                        cudaStream_t s);
// the same fused with the chunk statistics (N, C/cw, 2) of the fp32 result (zeroed by the caller)
int launch_h2f_epilogue_stats(int dt, const void* y16, const float* addvec, const float* residual, float scale, float* out, int B, int HW, int C,
                              int cw, double* stats, cudaStream_t s);
int launch_h2f_accumulate(int dt, const void* y16, float* out, size_t n, cudaStream_t s);
int launch_relayout_tc_dgrad_s2(int dt, const float* w, int O, int I, void* out, cudaStream_t s);
// one pass over dY: column sums per tensor (out_all) and / or per image (out_img), optional 16-bit copy (dt: DT_BF16 / DT_F16)
int launch_colsum_cast(int dt, const float* dy, int B, int rows_per_img, int C, float* out_all, float* out_img, void* out16, cudaStream_t s);
int launch_wgrad_unstage(const float* stage, int O, int I, int kk, float* dw, cudaStream_t s, int Opad = 0, int Ipad = 0);

// softmax attention (head_dim 8) on the warp-level tensor cores, 16-bit operands (dt: DT_BF16 / DT_F16) staged from the fp32 activations
// (pd_train_attn_mma.cu); otherwise the interface of launch_attn8_fwd / launch_attn8_bwd
bool attn8_mma_supported(int S, int C, int pitch);
int launch_attn8_mma_fwd(int dt, const float* q, const float* k, const float* v, int pitch, int N, int S, int C, float* out, float* lse,
                         cudaStream_t s);
int launch_attn8_mma_bwd(int dt, const float* q, const float* k, const float* v, int pitch, const float* o, const float* dout, const float* lse,
                         int N, int S, int C, float* dq, float* dk, float* dv, float* delta, cudaStream_t s);

// tcgen05 weight gradient of a stride-1 'same' convolution (k = 1 or 3): stage[tap][co][ci] += sum_pixels dY[p, co] * X[p @ tap, ci],
// K = pixels.  x1 / x2: the NHWC 16-bit sources of the conv input (channel concat), dy: (N, H, W, Cout) 16-bit.
struct WgradTcDesc {
    int dt;
    const void *x1, *x2;
    int C1, C2, N, H, W, Cout, ksize;      // H, W: extent of X
    const void* dy;
    float* stage;          // (k*k, Cout, C1 + C2) fp32, accumulated with vector reductions (zeroed by the caller)
    int stride;            // 0 / 1, or 2: 3x3 stride-2 padding-1 convolution (dY is (N, H/2, W/2, Cout))
};
struct WgradTcPlan;
bool wgrad_tc_supported(const WgradTcDesc& d, std::string* why);
int wgrad_tc_plan_create(const WgradTcDesc& d, WgradTcPlan** out);
void wgrad_tc_plan_destroy(WgradTcPlan* p);
int wgrad_tc_launch(const WgradTcPlan* p, cudaStream_t s);

}  // namespace pd
