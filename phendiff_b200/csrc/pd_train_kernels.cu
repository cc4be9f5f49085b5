// phendiff_b200 — kernels of the TRAINING step (SURVEY §8 row f2; reference src/utils_training.py:244-456: noise / timestep
// sampling, `_diffusion_and_backward`, loss by prediction type :415-433, clip_grad_norm_(1.0) :439, AdamW train.py:279-285, EMA
// utils_training.py:224-241).  This file is the fp32 path of the backward pass: every backward operator of the UNet graph as a
// CUDA-core kernel over NHWC fp32 activations, checked against torch.autograd on the oracle (tests/test_gpu_training.py).  It
// plays the role the SIMT kernels play for inference: the validation mode the tensor-core backward is compared against.
//   conv wgrad    dW[co, ci, r, s] += sum_pixels dY[p, co] * X[p @ (r, s), ci]        (split over pixel chunks, atomics)
//   conv dgrad    stride 1: the forward SIMT conv on tap-flipped, transposed weights; stride 2: gather kernel below
//   bias / time-embedding grads: column sums of dY per tensor / per image
//   GroupNorm (+SiLU) backward, softmax attention backward (head_dim 8, probabilities recomputed from the saved log-sum-exp),
//   nearest-upsample backward, small dense GEMMs of the embedding MLP, the weighted-MSE loss and its gradient,
//   global-norm clip + AdamW + EMA over flat parameter vectors.
#include "pd_kernels.h"
#include "pd_train.h"

namespace pd {

template <typename T> struct alignas(16) Half8 { T v[8]; };

// ---------------------------------------------------------------------------------------------------------------------
// weight re-layouts for the backward convolutions
// ---------------------------------------------------------------------------------------------------------------------
// OIHW (O, I, k, k) -> dgrad weights (k*k*O, Isub) for input channels [i0, i0 + Isub): row = tap' * O + o with tap' the FLIPPED
// tap (k*k - 1 - tap), so that the stride-1 forward kernel computes dX = conv(dY, W^T flipped)
__global__ void relayout_dgrad_kernel(const float* __restrict__ w, int O, int I, int k, int i0, int Isub, float* __restrict__ out) {
    const int kk = k * k;
    const size_t total = (size_t)kk * O * Isub;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int i = idx % Isub;
        const size_t r = idx / Isub;
        const int o = r % O, tapf = r / O;
        const int tap = kk - 1 - tapf;
        out[idx] = w[((size_t)o * I + i0 + i) * kk + tap];
    }
}
int launch_relayout_dgrad(const float* w, int O, int I, int k, int i0, int Isub, float* out, cudaStream_t s) {
    const size_t total = (size_t)k * k * O * Isub;
    relayout_dgrad_kernel<<<(int)std::min<size_t>((total + 255) / 256, 4096), 256, 0, s>>>(w, O, I, k, i0, Isub, out);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// conv wgrad: 64 (ci) x 64 (co) tile of one tap per CTA over a chunk of output pixels, K = pixels, fp32 atomics into OIHW
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv_wgrad_kernel(WgradArgs a) {
    constexpr int BM = 64, BN = 64, BK = 16;
    __shared__ __align__(16) float Xs[BK][BM + 4];   // [pixel][ci]
    __shared__ __align__(16) float Gs[BK][BN + 4];   // [pixel][co]
    const int tid = threadIdx.x;
    const int Ct = a.C1 + a.C2, kk = a.ksize * a.ksize;
    const int citiles = (Ct + BM - 1) / BM;
    const int tap = blockIdx.x / citiles, ci0 = (blockIdx.x - tap * citiles) * BM;
    const int co0 = blockIdx.y * BN;
    const int r = tap / a.ksize, sx = tap - r * a.ksize;
    const int M = a.N * a.Ho * a.Wo;
    const int m_begin = blockIdx.z * a.chunk, m_end = min(m_begin + a.chunk, M);
    // load roles: pixel row lp (0..15), 4 consecutive channels at lc
    const int lp = tid >> 4, lc = (tid & 15) * 4;
    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int m0 = m_begin; m0 < m_end; m0 += BK) {
        const int m = m0 + lp;
        float xv[4] = {0.f, 0.f, 0.f, 0.f}, gv[4] = {0.f, 0.f, 0.f, 0.f};
        if (m < m_end) {
            const int img = m / (a.Ho * a.Wo), rem = m - img * a.Ho * a.Wo, ho = rem / a.Wo, wo = rem - ho * a.Wo;
            const int ih = ho * a.stride - a.pad + r, iw = wo * a.stride - a.pad + sx;
            if (ih >= 0 && ih < a.H && iw >= 0 && iw < a.W) {
                const size_t pix = ((size_t)img * a.H + ih) * a.W + iw;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int ci = ci0 + lc + i;
                    if (ci < a.C1) xv[i] = a.x1[pix * a.C1 + ci];
                    else if (ci < Ct) xv[i] = a.x2[pix * a.C2 + (ci - a.C1)];
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (co0 + lc + i < a.Cout) gv[i] = a.dy[(size_t)m * a.dy_pitch + co0 + lc + i];
        }
        __syncthreads();
        *reinterpret_cast<float4*>(&Xs[lp][lc]) = make_float4(xv[0], xv[1], xv[2], xv[3]);
        *reinterpret_cast<float4*>(&Gs[lp][lc]) = make_float4(gv[0], gv[1], gv[2], gv[3]);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 xf = *reinterpret_cast<const float4*>(&Xs[k][ty * 4]);
            const float4 gf = *reinterpret_cast<const float4*>(&Gs[k][tx * 4]);
            const float xx[4] = {xf.x, xf.y, xf.z, xf.w}, gg[4] = {gf.x, gf.y, gf.z, gf.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xx[i], gg[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int ci = ci0 + ty * 4 + i;
        if (ci >= a.Iw) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = co0 + tx * 4 + j;
            if (co < a.Cout) atomicAdd(a.dw + ((size_t)co * a.Iw + ci) * kk + tap, acc[i][j] * a.scale);
        }
    }
}
int launch_conv_wgrad(const WgradArgs& a_, cudaStream_t s) {
    WgradArgs a = a_;
    const int Ct = a.C1 + a.C2, M = a.N * a.Ho * a.Wo;
    if (a.Iw <= 0) a.Iw = Ct;
    if (a.dy_pitch <= 0) a.dy_pitch = a.Cout;
    PD_REQUIRE(a.C1 % 4 == 0 && Ct % 4 == 0, "conv_wgrad needs channel counts that are multiples of 4");
    const int tiles = ((Ct + 63) / 64) * a.ksize * a.ksize * ((a.Cout + 63) / 64);
    int split = std::max(1, std::min((M + 255) / 256, (148 * 6 + tiles - 1) / tiles));
    a.chunk = (((M + split - 1) / split) + 15) / 16 * 16;
    split = (M + a.chunk - 1) / a.chunk;
    dim3 grid(((Ct + 63) / 64) * a.ksize * a.ksize, (a.Cout + 63) / 64, split);
    conv_wgrad_kernel<<<grid, 256, 0, s>>>(a);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// column sums of dY (M rows x C): per tensor (rows_per_seg = M) or per image (rows_per_seg = H*W) -> out[seg, c] += scale * sum
// (C = row pitch of dy; only the first Cvalid columns are summed: conv_out's gradient rows are padded from 3 to 4 channels)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ dy, int M, int C, int Cvalid, int rows_per_seg,
                                                      int rows_per_block, float scale, float* __restrict__ out) {
    const int seg = blockIdx.y;
    const int r0 = seg * rows_per_seg + blockIdx.x * rows_per_block;
    const int r1 = min(min(r0 + rows_per_block, (seg + 1) * rows_per_seg), M);
    for (int c = threadIdx.x; c < Cvalid; c += blockDim.x) {
        float acc = 0.f;
        for (int r = r0; r < r1; ++r) acc += dy[(size_t)r * C + c];
        atomicAdd(out + (size_t)seg * Cvalid + c, acc * scale);
    }
}
int launch_colsum(const float* dy, int M, int C, int rows_per_seg, float scale, float* out, cudaStream_t s, int Cvalid) {
    if (Cvalid <= 0) Cvalid = C;
    const int segs = M / rows_per_seg;
    const int rpb = std::max(16, std::min(rows_per_seg, 256));
    dim3 grid((rows_per_seg + rpb - 1) / rpb, segs);
    colsum_kernel<<<grid, 256, 0, s>>>(dy, M, C, Cvalid, rows_per_seg, rpb, scale, out);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// gather dgrad for the shapes the GEMM-style path does not take (stride-2 Downsample2D, conv_out's 3 output channels):
// dX[n, ih, iw, ci] += sum_{taps with (ih + pad - r) divisible by stride, co} dY[n, oh, ow, co] W[co, ci, r, s]
// one warp per input pixel, lanes over ci (weights OIHW through L1 / L2: three layers per model, validation path)
__global__ void __launch_bounds__(256) conv_dgrad_gather_kernel(const float* __restrict__ dy, int dy_pitch, const float* __restrict__ w, int N,
                                                                 int H, int W, int C, int Ho, int Wo, int Cout, int pad, int stride,
                                                                 float* __restrict__ dx) {
    const int lane = threadIdx.x & 31;
    const size_t pixel = (size_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pixel >= (size_t)N * H * W) return;
    const int n = pixel / ((size_t)H * W), rem = pixel - (size_t)n * H * W, ih = rem / W, iw = rem - ih * W;
    for (int ci = lane; ci < C; ci += 32) {
        float acc = 0.f;
        for (int r = 0; r < 3; ++r) {
            const int t = ih + pad - r;
            if (t < 0 || (t % stride)) continue;
            const int oh = t / stride;
            if (oh >= Ho) continue;
            for (int sx = 0; sx < 3; ++sx) {
                const int u = iw + pad - sx;
                if (u < 0 || (u % stride)) continue;
                const int ow = u / stride;
                if (ow >= Wo) continue;
                const float* g = dy + (((size_t)n * Ho + oh) * Wo + ow) * dy_pitch;
                const float* wp = w + (size_t)ci * 9 + r * 3 + sx;
                for (int co = 0; co < Cout; ++co) acc = fmaf(g[co], wp[(size_t)co * C * 9], acc);
            }
        }
        dx[pixel * C + ci] += acc;
    }
}
int launch_conv_dgrad_gather(const float* dy, int dy_pitch, const float* w, int N, int H, int W, int C, int Ho, int Wo, int Cout, int pad,
                             int stride, float* dx, cudaStream_t s) {
    const size_t pixels = (size_t)N * H * W;
    conv_dgrad_gather_kernel<<<(int)((pixels + 7) / 8), 256, 0, s>>>(dy, dy_pitch, w, N, H, W, C, Ho, Wo, Cout, pad, stride, dx);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// nearest 2x upsample backward: dx[n, h, w, c] += sum of the 2x2 block of dy
__global__ void upsample2x_bwd_kernel(const float* __restrict__ dy, int N, int H, int W, int C, float* __restrict__ dx) {
    const size_t total = (size_t)N * H * W * C;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = i % C;
        size_t p = i / C;
        const int w = p % W; p /= W;
        const int h = p % H;
        const int n = p / H;
        const float* b = dy + (((size_t)n * 2 * H + 2 * h) * 2 * W + 2 * w) * C + c;
        dx[i] += b[0] + b[C] + b[(size_t)2 * W * C] + b[(size_t)2 * W * C + C];
    }
}
int launch_upsample2x_bwd(const float* dy, int N, int H, int W, int C, float* dx, cudaStream_t s) {
    const size_t total = (size_t)N * H * W * C;
    upsample2x_bwd_kernel<<<(int)std::min<size_t>((total + 255) / 256, 148 * 16), 256, 0, s>>>(dy, N, H, W, C, dx);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// GroupNorm (+SiLU) backward over concat(x1, x2).  y = act(z), z = xhat * gamma + beta, xhat = (x - mean) * rstd.
//   pass 1 (reduce): dz = dy * act'(z); dbeta_c += sum dz; dgamma_c += sum dz xhat; s1[n,g] += gamma_c dz; s2[n,g] += gamma_c dz xhat
//   pass 2 (apply):  dx += rstd * (gamma dz - (s1 + xhat s2) / count)
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float silu_grad(float z) {
    // fast exponential / division (2 MUFU + a few FMAs instead of ~25 instructions): relative error ~1e-6, far inside the 3e-5 the
    // fp32 gradient tests hold, and the GroupNorm backward passes are instruction-co-bound (ncu r7e: issue 41 %, DRAM 28 %)
    const float sg = __fdividef(1.0f, 1.0f + __expf(-z));
    return sg * (1.0f + z * (1.0f - sg));
}
__device__ __forceinline__ void gn_mean_rstd(const GNBwdArgs& a, int n, int g, float* mean, float* rstd) {
    const int C = a.C1 + a.C2, cpg = C / a.groups, cw = a.stats_cw;
    double sum = 0.0, sq = 0.0;
    for (int cc = g * cpg; cc < (g + 1) * cpg; cc += cw) {
        const double* st = (cc < a.C1) ? a.stats1 + ((size_t)n * (a.C1 / cw) + cc / cw) * 2
                                       : a.stats2 + ((size_t)n * (a.C2 / cw) + (cc - a.C1) / cw) * 2;
        sum += st[0]; sq += st[1];
    }
    const double inv = 1.0 / ((double)cpg * a.HW), mu = sum * inv;
    *mean = (float)mu;
    *rstd = 1.0f / sqrtf((float)fmax(sq * inv - mu * mu, 0.0) + a.eps);
}
template <typename TD> __device__ __forceinline__ float4 ld_dy4(const TD* p);
template <> __device__ __forceinline__ float4 ld_dy4<float>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <> __device__ __forceinline__ float4 ld_dy4<bf16>(const bf16* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x), b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
    return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
}
template <> __device__ __forceinline__ float4 ld_dy4<f16>(const f16* p) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const __half2 a = *reinterpret_cast<const __half2*>(&u.x), b = *reinterpret_cast<const __half2*>(&u.y);
    return make_float4(__low2float(a), __high2float(a), __low2float(b), __high2float(b));
}
// four channels per thread (float4 rows), rows strided over the block; TD = type of dy (fp32, or the 16-bit gradient a tensor-core
// dgrad wrote directly)
template <int PASS, typename TD>
__global__ void __launch_bounds__(256) gn_bwd_kernel(GNBwdArgs a, int rows_per_block) {
    extern __shared__ float sm[];   // mean[groups], rstd[groups], s1[groups], s2[groups], then (pass 1) the reduction buffer
    const int C = a.C1 + a.C2, cpg = C / a.groups, C4 = C / 4;
    const int n = blockIdx.y;
    float* s_mean = sm;
    float* s_rstd = sm + a.groups;
    float* s_s1 = sm + 2 * a.groups;
    float* s_s2 = sm + 3 * a.groups;
    float4* red = reinterpret_cast<float4*>(sm + 4 * a.groups);   // [2][256]
    for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
        gn_mean_rstd(a, n, g, &s_mean[g], &s_rstd[g]);
        if (PASS == 2) { s_s1[g] = a.gsum[((size_t)n * a.groups + g) * 2]; s_s2[g] = a.gsum[((size_t)n * a.groups + g) * 2 + 1]; }
    }
    __syncthreads();
    const int r0 = blockIdx.x * rows_per_block, r1 = min(r0 + rows_per_block, a.HW);
    const float inv_cnt = 1.0f / ((float)cpg * (float)a.HW);
    const int rstep = max(1, 256 / C4);
    const TD* dyp = reinterpret_cast<const TD*>(a.dy);
    for (int cg0 = 0; cg0 < C4; cg0 += 256) {
        const int cg = cg0 + (C4 >= 256 ? threadIdx.x : threadIdx.x % C4);
        const int rr = C4 >= 256 ? 0 : threadIdx.x / C4;
        const bool worker = cg < C4 && rr < rstep;
        const int c = cg * 4;
        float mu[4], rs[4], ga[4], be[4], k1[4], k2[4];
        const float* x = nullptr;
        float* dx = nullptr;
        int pitch = 0, co = 0;
        if (worker) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int g = (c + j) / cpg;
                mu[j] = s_mean[g]; rs[j] = s_rstd[g]; ga[j] = a.gamma[c + j]; be[j] = a.beta[c + j];
                k1[j] = PASS == 2 ? s_s1[g] * inv_cnt : 0.f; k2[j] = PASS == 2 ? s_s2[g] * inv_cnt : 0.f;
            }
            if (c < a.C1) { x = a.x1; dx = a.dx1; pitch = a.C1; co = c; } else { x = a.x2; dx = a.dx2; pitch = a.C2; co = c - a.C1; }
        }
        const size_t base = (size_t)n * a.HW;
        float sa[4] = {0.f, 0.f, 0.f, 0.f}, sb[4] = {0.f, 0.f, 0.f, 0.f};
        if (worker) {
#pragma unroll 4
            for (int r = r0 + rr; r < r1; r += rstep) {
                const float4 xv = *reinterpret_cast<const float4*>(x + (base + r) * pitch + co);
                const float4 dv = ld_dy4<TD>(dyp + (base + r) * C + c);
                const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
                float dz[4] = {dv.x, dv.y, dv.z, dv.w}, xh[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    xh[j] = (xs[j] - mu[j]) * rs[j];
                    if (a.silu) dz[j] *= silu_grad(fmaf(xh[j], ga[j], be[j]));
                    if (PASS == 1) { sa[j] += dz[j]; sb[j] += dz[j] * xh[j]; }
                }
                if (PASS == 2) {
                    float4* dp = reinterpret_cast<float4*>(dx + (base + r) * pitch + co);
                    float4 d = *dp;
                    d.x += rs[0] * (ga[0] * dz[0] - (k1[0] + xh[0] * k2[0]));
                    d.y += rs[1] * (ga[1] * dz[1] - (k1[1] + xh[1] * k2[1]));
                    d.z += rs[2] * (ga[2] * dz[2] - (k1[2] + xh[2] * k2[2]));
                    d.w += rs[3] * (ga[3] * dz[3] - (k1[3] + xh[3] * k2[3]));
                    *dp = d;
                }
            }
        }
        if (PASS == 1) {
            red[threadIdx.x] = make_float4(sa[0], sa[1], sa[2], sa[3]);
            red[256 + threadIdx.x] = make_float4(sb[0], sb[1], sb[2], sb[3]);
            __syncthreads();
            if (worker && rr == 0) {
                for (int k = 1; k < rstep; ++k) {
                    const float4 u = red[threadIdx.x + k * C4], v = red[256 + threadIdx.x + k * C4];
                    sa[0] += u.x; sa[1] += u.y; sa[2] += u.z; sa[3] += u.w; sb[0] += v.x; sb[1] += v.y; sb[2] += v.z; sb[3] += v.w;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int g = (c + j) / cpg;
                    if (a.dbeta) atomicAdd(a.dbeta + c + j, sa[j] * a.scale);      // null: input-gradient-only backward
                    if (a.dgamma) atomicAdd(a.dgamma + c + j, sb[j] * a.scale);
                    atomicAdd(a.gsum + ((size_t)n * a.groups + g) * 2, ga[j] * sa[j]);
                    atomicAdd(a.gsum + ((size_t)n * a.groups + g) * 2 + 1, ga[j] * sb[j]);
                }
            }
            __syncthreads();
        }
    }
}
int launch_gn_bwd(const GNBwdArgs& a, cudaStream_t s) {
    const int C = a.C1 + a.C2;
    PD_REQUIRE(C % a.groups == 0, "channels not divisible by groups");
    PD_REQUIRE(C % 4 == 0 && a.C1 % 4 == 0, "GroupNorm backward: channel counts must be multiples of 4");
    PD_CHECK_CUDA(cudaMemsetAsync(a.gsum, 0, (size_t)a.N * a.groups * 2 * sizeof(float), s));
    // rows per block: at least ~8 blocks per SM in flight (small feature maps), at most 128 rows (prologue amortisation)
    int rpb = (int)std::min<size_t>(128, std::max<size_t>(16, ((size_t)a.N * a.HW) / (148 * 8)));
    rpb = std::max(8, std::min(a.HW, rpb));
    dim3 grid((a.HW + rpb - 1) / rpb, a.N);
    const size_t smem = (size_t)4 * a.groups * sizeof(float) + 2 * 256 * sizeof(float4);
    if (a.dy_dt == DT_BF16) {
        gn_bwd_kernel<1, bf16><<<grid, 256, smem, s>>>(a, rpb);
        gn_bwd_kernel<2, bf16><<<grid, 256, smem, s>>>(a, rpb);
    } else if (a.dy_dt == DT_F16) {
        gn_bwd_kernel<1, f16><<<grid, 256, smem, s>>>(a, rpb);
        gn_bwd_kernel<2, f16><<<grid, 256, smem, s>>>(a, rpb);
    } else {
        gn_bwd_kernel<1, float><<<grid, 256, smem, s>>>(a, rpb);
        gn_bwd_kernel<2, float><<<grid, 256, smem, s>>>(a, rpb);
    }
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// GroupNorm (+SiLU) forward of the mixed-precision path: fp32 sources (concat) -> 16-bit NHWC output only (the operand of the
// tensor-core convolution that consumes it; the fp32 copy is never written).  Eight channels per thread.
template <typename T>
__global__ void __launch_bounds__(256) gn_apply16_kernel(GNBwdArgs a, T* __restrict__ out, int rows_per_block) {
    extern __shared__ float sm[];   // mean[groups], rstd[groups]
    const int C = a.C1 + a.C2, cpg = C / a.groups, C8 = C / 8;
    const int n = blockIdx.y;
    float* s_mean = sm;
    float* s_rstd = sm + a.groups;
    for (int g = threadIdx.x; g < a.groups; g += blockDim.x) gn_mean_rstd(a, n, g, &s_mean[g], &s_rstd[g]);
    __syncthreads();
    const int r0 = blockIdx.x * rows_per_block, r1 = min(r0 + rows_per_block, a.HW);
    const int rstep = max(1, 256 / C8);
    const size_t base = (size_t)n * a.HW;
    for (int cg0 = 0; cg0 < C8; cg0 += 256) {
        const int cg = cg0 + (C8 >= 256 ? threadIdx.x : threadIdx.x % C8);
        const int rr = C8 >= 256 ? 0 : threadIdx.x / C8;
        if (cg >= C8 || rr >= rstep) continue;
        const int c = cg * 8;
        float sc[8], sh[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int g = (c + j) / cpg;
            sc[j] = s_rstd[g] * a.gamma[c + j];
            sh[j] = a.beta[c + j] - s_mean[g] * sc[j];
        }
        const float* x;
        int pitch, co;
        if (c < a.C1) { x = a.x1; pitch = a.C1; co = c; } else { x = a.x2; pitch = a.C2; co = c - a.C1; }
#pragma unroll 4
        for (int r = r0 + rr; r < r1; r += rstep) {
            const float4 u = *reinterpret_cast<const float4*>(x + (base + r) * pitch + co), v = *reinterpret_cast<const float4*>(x + (base + r) * pitch + co + 4);
            float y[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
            Half8<T> h;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float z = fmaf(y[j], sc[j], sh[j]);
                if (a.silu) z = __fdividef(z, 1.0f + __expf(-z));
                h.v[j] = from_f<T>(z);
            }
            *reinterpret_cast<Half8<T>*>(out + (base + r) * C + c) = h;
        }
    }
}
int launch_gn_apply16(int dt, const GNBwdArgs& a, void* out, cudaStream_t s) {
    const int C = a.C1 + a.C2;
    PD_REQUIRE(C % a.groups == 0 && C % 8 == 0 && a.C1 % 8 == 0, "gn_apply16: channel counts must be multiples of 8");
    const int rpb = std::max(8, std::min(a.HW, 128));
    dim3 grid((a.HW + rpb - 1) / rpb, a.N);
    const size_t smem = (size_t)2 * a.groups * sizeof(float);
    PD_DISPATCH_HALF(dt, T, (gn_apply16_kernel<T><<<grid, 256, smem, s>>>(a, (T*)out, rpb)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// attention, head_dim 8: forward that also stores the log-sum-exp of every query row, and the backward that recomputes P from it
// ---------------------------------------------------------------------------------------------------------------------
constexpr float kAttnScale8 = 0.35355339059327373f;   // 1 / sqrt(8)
__global__ void __launch_bounds__(128) attn8_fwd_kernel(const float* __restrict__ qp, const float* __restrict__ kp,
                                                         const float* __restrict__ vp, int pitch, int S, int C, float* __restrict__ out,
                                                         float* __restrict__ lse) {
    constexpr int D = 8, TK = 128;
    __shared__ float Ks[TK][D], Vs[TK][D];
    const int n = blockIdx.z, head = blockIdx.y, qi = blockIdx.x * 128 + threadIdx.x;
    const size_t rowp = (size_t)pitch, off = (size_t)n * S * rowp + head * D;
    const float *qb = qp + off, *kb = kp + off, *vb = vp + off;
    float q[D], o[D];
#pragma unroll
    for (int i = 0; i < D; ++i) { q[i] = qi < S ? qb[(size_t)qi * rowp + i] * kAttnScale8 : 0.f; o[i] = 0.f; }
    float mx = -INFINITY, l = 0.f;
    for (int k0 = 0; k0 < S; k0 += TK) {
        __syncthreads();
        const int kj = k0 + threadIdx.x;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            Ks[threadIdx.x][i] = kj < S ? kb[(size_t)kj * rowp + i] : 0.f;
            Vs[threadIdx.x][i] = kj < S ? vb[(size_t)kj * rowp + i] : 0.f;
        }
        __syncthreads();
        const int kmax = min(TK, S - k0);
        for (int j = 0; j < kmax; ++j) {
            float sc = 0.f;
#pragma unroll
            for (int i = 0; i < D; ++i) sc = fmaf(q[i], Ks[j][i], sc);
            const float nm = fmaxf(mx, sc), corr = expf(mx - nm), p = expf(sc - nm);
            l = l * corr + p;
#pragma unroll
            for (int i = 0; i < D; ++i) o[i] = fmaf(o[i], corr, p * Vs[j][i]);
            mx = nm;
        }
    }
    if (qi < S) {
        const float inv = 1.0f / l;
        float* op = out + ((size_t)n * S + qi) * C + head * D;
#pragma unroll
        for (int i = 0; i < D; ++i) op[i] = o[i] * inv;
        lse[((size_t)n * (C / D) + head) * S + qi] = mx + logf(l);
    }
}
// dq: thread per query, keys staged; dk / dv: thread per key, queries staged.  delta[q] = sum_d dO[q, d] O[q, d].
__global__ void __launch_bounds__(128) attn8_bwd_q_kernel(const float* __restrict__ qp, const float* __restrict__ kp,
                                                           const float* __restrict__ vp, int pitch, const float* __restrict__ o,
                                                           const float* __restrict__ dout, const float* __restrict__ lse, int S, int C,
                                                           float* __restrict__ dq_out, float* __restrict__ delta) {
    constexpr int D = 8, TK = 128;
    __shared__ float Ks[TK][D], Vs[TK][D];
    const int n = blockIdx.z, head = blockIdx.y, qi = blockIdx.x * 128 + threadIdx.x;
    const size_t rowp = (size_t)pitch, off = (size_t)n * S * rowp + head * D;
    const float *qb = qp + off, *kb = kp + off, *vb = vp + off;
    float q[D], dq[D], g[D];
    float dl = 0.f, L = 0.f;
    if (qi < S) {
        const size_t orow = ((size_t)n * S + qi) * C + head * D;
#pragma unroll
        for (int i = 0; i < D; ++i) { q[i] = qb[(size_t)qi * rowp + i] * kAttnScale8; g[i] = dout[orow + i]; dl = fmaf(g[i], o[orow + i], dl); }
        L = lse[((size_t)n * (C / D) + head) * S + qi];
        delta[((size_t)n * (C / D) + head) * S + qi] = dl;
    } else {
#pragma unroll
        for (int i = 0; i < D; ++i) { q[i] = 0.f; g[i] = 0.f; }
    }
#pragma unroll
    for (int i = 0; i < D; ++i) dq[i] = 0.f;
    for (int k0 = 0; k0 < S; k0 += TK) {
        __syncthreads();
        const int kj = k0 + threadIdx.x;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            Ks[threadIdx.x][i] = kj < S ? kb[(size_t)kj * rowp + i] : 0.f;
            Vs[threadIdx.x][i] = kj < S ? vb[(size_t)kj * rowp + i] : 0.f;
        }
        __syncthreads();
        const int kmax = min(TK, S - k0);
        for (int j = 0; j < kmax; ++j) {
            float sc = 0.f, dp = 0.f;
#pragma unroll
            for (int i = 0; i < D; ++i) { sc = fmaf(q[i], Ks[j][i], sc); dp = fmaf(g[i], Vs[j][i], dp); }
            const float ds = expf(sc - L) * (dp - dl);
#pragma unroll
            for (int i = 0; i < D; ++i) dq[i] = fmaf(ds, Ks[j][i], dq[i]);
        }
    }
    if (qi < S) {
        float* dp = dq_out + off + (size_t)qi * rowp;
#pragma unroll
        for (int i = 0; i < D; ++i) dp[i] += dq[i] * kAttnScale8;
    }
}
__global__ void __launch_bounds__(128) attn8_bwd_kv_kernel(const float* __restrict__ qp, const float* __restrict__ kp,
                                                            const float* __restrict__ vp, int pitch, const float* __restrict__ dout,
                                                            const float* __restrict__ lse, const float* __restrict__ delta, int S, int C,
                                                            float* __restrict__ dk_out, float* __restrict__ dv_out) {
    constexpr int D = 8, TQ = 128;
    __shared__ float Qs[TQ][D], Gs[TQ][D], Ls[TQ], Ds[TQ];
    const int n = blockIdx.z, head = blockIdx.y, kj = blockIdx.x * 128 + threadIdx.x;
    const size_t rowp = (size_t)pitch, off = (size_t)n * S * rowp + head * D;
    const float *qb = qp + off, *kb = kp + off, *vb = vp + off;
    float k[D], v[D], dk[D], dv[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        k[i] = kj < S ? kb[(size_t)kj * rowp + i] : 0.f;
        v[i] = kj < S ? vb[(size_t)kj * rowp + i] : 0.f;
        dk[i] = 0.f; dv[i] = 0.f;
    }
    for (int q0 = 0; q0 < S; q0 += TQ) {
        __syncthreads();
        const int qi = q0 + threadIdx.x;
        const size_t orow = ((size_t)n * S + qi) * C + head * D;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            Qs[threadIdx.x][i] = qi < S ? qb[(size_t)qi * rowp + i] * kAttnScale8 : 0.f;
            Gs[threadIdx.x][i] = qi < S ? dout[orow + i] : 0.f;
        }
        Ls[threadIdx.x] = qi < S ? lse[((size_t)n * (C / D) + head) * S + qi] : INFINITY;   // exp(s - inf) = 0 for padding queries
        Ds[threadIdx.x] = qi < S ? delta[((size_t)n * (C / D) + head) * S + qi] : 0.f;
        __syncthreads();
        const int qmax = min(TQ, S - q0);
        for (int j = 0; j < qmax; ++j) {
            float sc = 0.f, dp = 0.f;
#pragma unroll
            for (int i = 0; i < D; ++i) { sc = fmaf(Qs[j][i], k[i], sc); dp = fmaf(Gs[j][i], v[i], dp); }
            const float p = expf(sc - Ls[j]), ds = p * (dp - Ds[j]);
#pragma unroll
            for (int i = 0; i < D; ++i) { dv[i] = fmaf(p, Gs[j][i], dv[i]); dk[i] = fmaf(ds, Qs[j][i], dk[i]); }   // Qs carries 1/sqrt(d)
        }
    }
    if (kj < S) {
#pragma unroll
        for (int i = 0; i < D; ++i) { dk_out[off + (size_t)kj * rowp + i] += dk[i]; dv_out[off + (size_t)kj * rowp + i] += dv[i]; }
    }
}
int launch_attn8_fwd(const float* q, const float* k, const float* v, int pitch, int N, int S, int C, float* out, float* lse, cudaStream_t s) {
    PD_REQUIRE(C % 8 == 0, "attention channels must be a multiple of 8");
    attn8_fwd_kernel<<<dim3((S + 127) / 128, C / 8, N), 128, 0, s>>>(q, k, v, pitch, S, C, out, lse);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
int launch_attn8_bwd(const float* q, const float* k, const float* v, int pitch, const float* o, const float* dout, const float* lse, int N,
                     int S, int C, float* dq, float* dk, float* dv, float* delta, cudaStream_t s) {
    dim3 grid((S + 127) / 128, C / 8, N);
    attn8_bwd_q_kernel<<<grid, 128, 0, s>>>(q, k, v, pitch, o, dout, lse, S, C, dq, delta);
    attn8_bwd_kv_kernel<<<grid, 128, 0, s>>>(q, k, v, pitch, dout, lse, delta, S, C, dk, dv);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// small dense GEMMs of the embedding MLP (rows = batch): C[M, N] (+)= alpha * op(A)[M, K] op(B)[K, N]; one thread per output
// ---------------------------------------------------------------------------------------------------------------------
__global__ void sgemm_kernel(int ta, int tb, int M, int N, int K, float alpha, const float* __restrict__ A, int lda,
                             const float* __restrict__ B, int ldb, float* __restrict__ Cm, int ldc, int accumulate) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
    if (n >= N || m >= M) return;
    float acc = 0.f;
    for (int k = 0; k < K; ++k) {
        const float av = ta ? A[(size_t)k * lda + m] : A[(size_t)m * lda + k];
        const float bv = tb ? B[(size_t)n * ldb + k] : B[(size_t)k * ldb + n];
        acc = fmaf(av, bv, acc);
    }
    float* c = Cm + (size_t)m * ldc + n;
    *c = (accumulate ? *c : 0.f) + alpha * acc;
}
int launch_sgemm(int ta, int tb, int M, int N, int K, float alpha, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                 int accumulate, cudaStream_t s) {
    sgemm_kernel<<<dim3((N + 127) / 128, M), 128, 0, s>>>(ta, tb, M, N, K, alpha, A, lda, B, ldb, C, ldc, accumulate);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// elementwise helpers of the embedding path
__global__ void sinusoid_kernel(const float* __restrict__ t, int B, int C0, int flip, float shift, float* __restrict__ out) {
    const int b = blockIdx.x, half = C0 / 2;
    for (int k = threadIdx.x; k < half; k += blockDim.x) {
        const float f = expf((-9.210340371976184f * (float)k) / ((float)half - shift));
        const float arg = t[b] * f, sn = sinf(arg), cs = cosf(arg);
        if (flip) { out[(size_t)b * C0 + k] = cs; out[(size_t)b * C0 + half + k] = sn; }
        else { out[(size_t)b * C0 + k] = sn; out[(size_t)b * C0 + half + k] = cs; }
    }
}
// y = silu(x + bias [+ table[label]]) with the pre-activation kept; backward: dpre = dy * silu'(pre)
__global__ void bias_silu_fwd_kernel(float* __restrict__ pre, const float* __restrict__ bias, const float* __restrict__ table,
                                     const int64_t* __restrict__ labels, int B, int D, float* __restrict__ act) {
    const size_t total = (size_t)B * D;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = i / D, j = i - (size_t)b * D;
        float v = pre[i] + bias[j];
        if (table && labels) v += table[(size_t)labels[b] * D + j];
        pre[i] = v;
        act[i] = v / (1.0f + expf(-v));
    }
}
__global__ void silu_bwd_kernel(const float* __restrict__ pre, const float* __restrict__ dact, size_t total, float* __restrict__ dpre) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
        dpre[i] = dact[i] * silu_grad(pre[i]);
}
// table_grad[labels[b], :] += scale * d[b, :]
__global__ void scatter_rows_kernel(const float* __restrict__ d, const int64_t* __restrict__ labels, int B, int D, float scale,
                                    float* __restrict__ table_grad) {
    const size_t total = (size_t)B * D;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = i / D, j = i - (size_t)b * D;
        atomicAdd(table_grad + (size_t)labels[b] * D + j, d[i] * scale);
    }
}
// x[b, j] += bias[j]
__global__ void add_bias_rows_kernel(float* __restrict__ x, const float* __restrict__ bias, int B, int D) {
    const size_t total = (size_t)B * D;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) x[i] += bias[i % D];
}
int launch_add_bias_rows(float* x, const float* bias, int B, int D, cudaStream_t s) {
    add_bias_rows_kernel<<<std::min((B * D + 255) / 256, 1024), 256, 0, s>>>(x, bias, B, D);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
int launch_sinusoid(const float* t, int B, int C0, int flip, float shift, float* out, cudaStream_t s) {
    sinusoid_kernel<<<B, 128, 0, s>>>(t, B, C0, flip, shift, out);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
int launch_bias_silu_fwd(float* pre, const float* bias, const float* table, const int64_t* labels, int B, int D, float* act, cudaStream_t s) {
    bias_silu_fwd_kernel<<<std::min((B * D + 255) / 256, 1024), 256, 0, s>>>(pre, bias, table, labels, B, D, act);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
int launch_silu_bwd(const float* pre, const float* dact, size_t total, float* dpre, cudaStream_t s) {
    silu_bwd_kernel<<<(int)std::min<size_t>((total + 255) / 256, 1024), 256, 0, s>>>(pre, dact, total, dpre);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
int launch_scatter_rows(const float* d, const int64_t* labels, int B, int D, float scale, float* table_grad, cudaStream_t s) {
    scatter_rows_kernel<<<std::min((B * D + 255) / 256, 1024), 256, 0, s>>>(d, labels, B, D, scale, table_grad);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// NCHW fp32 (N, C, HW) -> NHWC fp32 (N, HW, Cp) zero-padded to Cp channels (the loss gradient entering conv_out's backward)
__global__ void nchw_to_nhwc_pad_kernel(const float* __restrict__ x, int N, int C, int HW, int Cp, float* __restrict__ out) {
    const size_t total = (size_t)N * HW * Cp;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = i % Cp;
        const size_t p = i / Cp;
        const int hw = p % HW, n = p / HW;
        out[i] = c < C ? x[((size_t)n * C + c) * HW + hw] : 0.f;
    }
}
int launch_nchw_to_nhwc_pad(const float* x, int N, int C, int HW, int Cp, float* out, cudaStream_t s) {
    const size_t total = (size_t)N * HW * Cp;
    nchw_to_nhwc_pad_kernel<<<(int)std::min<size_t>((total + 255) / 256, 148 * 16), 256, 0, s>>>(x, N, C, HW, Cp, out);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
// y += x (elementwise)
__global__ void add_inplace_kernel(float* __restrict__ y, const float* __restrict__ x, float alpha, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) y[i] = fmaf(alpha, x[i], y[i]);
}
int launch_add_inplace(float* y, const float* x, float alpha, size_t n, cudaStream_t s) {
    add_inplace_kernel<<<(int)std::min<size_t>((n + 255) / 256, 148 * 16), 256, 0, s>>>(y, x, alpha, n);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// loss of utils_training.py:415-433 in one form: mean over all elements of weight[b] * (m - target)^2 (epsilon: target = noise,
// weight = 1; v_prediction: target = velocity; sample: target = clean images, weight = alpha_t / (1 - alpha_t)), and its gradient
// ---------------------------------------------------------------------------------------------------------------------
// dm carries the loss scale S (GradScaler.scale(loss).backward()); the loss does not.  S = 1 multiplies exactly: unscaled runs are unchanged.
__global__ void __launch_bounds__(256) mse_loss_kernel(const float* __restrict__ m, const float* __restrict__ target,
                                                        const float* __restrict__ weight, int B, size_t per, const float* __restrict__ loss_scale,
                                                        float* __restrict__ loss, float* __restrict__ dm) {
    const size_t total = (size_t)B * per;
    const float inv = 1.0f / (float)total;
    const float sc = loss_scale ? *loss_scale : 1.0f;
    float acc = 0.f;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const float w = weight ? weight[i / per] : 1.0f, d = m[i] - target[i];
        acc = fmaf(w * d, d, acc);
        dm[i] = 2.0f * w * d * inv * sc;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) atomicAdd(loss, acc * inv);
}
int launch_mse_loss(const float* m, const float* target, const float* weight, int B, size_t per, const float* loss_scale, float* loss, float* dm,
                    cudaStream_t s) {
    PD_CHECK_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), s));
    mse_loss_kernel<<<(int)std::min<size_t>(((size_t)B * per + 255) / 256, 148 * 8), 256, 0, s>>>(m, target, weight, B, per, loss_scale, loss, dm);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// clip_grad_norm_(max_norm) + AdamW (torch.optim.AdamW semantics, decoupled weight decay) + EMA over flat fp32 vectors
// ---------------------------------------------------------------------------------------------------------------------
// global gradient norm, DETERMINISTIC (fixed summation tree, no atomics): data-parallel replicas must compute bit-identical clip
// coefficients or their parameters drift apart in the last bits (tools/check_ddp_train.py).  Stage 1: one partial per block in
// partial[1 + block]; stage 2: one block folds them in a fixed order into partial[0].
constexpr int kSumsqBlocks = 148 * 8;
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, size_t n, float* __restrict__ partial) {
    __shared__ float red[8];
    float acc = 0.f;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc = fmaf(g[i], g[i], acc);
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        partial[1 + blockIdx.x] = t;
    }
}
__global__ void __launch_bounds__(1024) sumsq_final_kernel(float* __restrict__ partial, int nblocks) {
    __shared__ double red[1024];
    double acc = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += 1024) acc += (double)partial[1 + i];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[0] = (float)red[0];
}
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                     float* __restrict__ v, float* __restrict__ ema, size_t n, float lr, float b1, float b2,
                                                     float eps, float wd, float bc1, float bc2_sqrt, float max_norm,
                                                     const float* __restrict__ sumsq, float ema_decay, float* __restrict__ norm_out) {
    const float norm = sqrtf(*sumsq);
    // torch.nn.utils.clip_grad_norm_: coef = max_norm / (norm + 1e-6), clamped to 1
    const float coef = max_norm > 0.f ? fminf(max_norm / (norm + 1e-6f), 1.0f) : 1.0f;
    if (norm_out && blockIdx.x == 0 && threadIdx.x == 0) *norm_out = norm;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float gi = g[i] * coef;
        float pi = p[i] * (1.0f - lr * wd);
        const float mi = b1 * m[i] + (1.0f - b1) * gi, vi = b2 * v[i] + (1.0f - b2) * gi * gi;
        m[i] = mi; v[i] = vi;
        pi -= (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
        p[i] = pi;
        if (ema) ema[i] -= (1.0f - ema_decay) * (ema[i] - pi);   // diffusers EMAModel.step: s -= (1 - decay) (s - p)
    }
}
int launch_adamw(float* p, const float* g, float* m, float* v, float* ema, size_t n, float lr, float b1, float b2, float eps, float wd,
                 int step, float max_norm, float ema_decay, float* scratch_sumsq, float* norm_out, cudaStream_t s) {
    const int grid = (int)std::min<size_t>((n + 255) / 256, kSumsqBlocks);
    sumsq_kernel<<<grid, 256, 0, s>>>(g, n, scratch_sumsq);
    sumsq_final_kernel<<<1, 1024, 0, s>>>(scratch_sumsq, grid);
    const float bc1 = 1.0f - powf(b1, (float)step), bc2 = 1.0f - powf(b2, (float)step);
    adamw_kernel<<<grid, 256, 0, s>>>(p, g, m, v, ema, n, lr, b1, b2, eps, wd, bc1, sqrtf(bc2), max_norm, scratch_sumsq, ema_decay, norm_out);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// the same step on loss-scaled gradients (fp16 mixed precision): torch.amp.GradScaler unscale_ / step / update around clip + AdamW,
// three launches like launch_adamw and just as deterministic (replicas keep bit-identical parameters AND scaler state).
//   stage 1: per block, the sum of squares of g * inv and whether any g is inf / NaN (inv = float(1 / double(S)), GradScaler's)
//   stage 2: one block folds both in a fixed order; one thread takes the decision: norm, clip coefficient, skip or apply, the AdamW
//            step count and its bias corrections, the scale update.  It rewrites S, so it leaves the S the gradients were made with
//            as inv in scratch: stage 1 has finished reading S, stage 3 reads only scratch.
//   stage 3: AdamW on (g * inv) * coef unless skipped, then the EMA step either way.
// scratch: [0, 8) decision (kScHdr*), [8, 8 + kSumsqBlocks) partial sums, then kSumsqBlocks non-finite flags
// ---------------------------------------------------------------------------------------------------------------------
enum { kScInv = 0, kScCoef = 1, kScStepSize = 2, kScBc2Sqrt = 3, kScApply = 4, kScHdr = 8 };
static_assert(kScHdr + 2 * kSumsqBlocks == PD_ADAMW_SCALED_SCRATCH_FLOATS, "scratch layout of pd_adamw_step_scaled");
__device__ __forceinline__ float inv_scale_of(float S) { return (float)(1.0 / (double)S); }
__global__ void __launch_bounds__(256) sumsq_unscale_kernel(const float* __restrict__ g, size_t n, const pd_grad_scaler_state_t* __restrict__ st,
                                                            float* __restrict__ scratch) {
    __shared__ float red[8];
    const float inv = inv_scale_of(st->scale);
    float acc = 0.f;
    bool bad = false;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float gi = g[i];
        bad |= !isfinite(gi);
        const float u = gi * inv;
        acc = fmaf(u, u, acc);
    }
    bad = __syncthreads_or(bad);
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        scratch[kScHdr + blockIdx.x] = t;
        scratch[kScHdr + kSumsqBlocks + blockIdx.x] = bad ? 1.f : 0.f;
    }
}
__global__ void __launch_bounds__(1024) scaler_decide_kernel(float* __restrict__ scratch, int nblocks, pd_grad_scaler_state_t* __restrict__ st,
                                                             float lr, float b1, float b2, float max_norm, float growth, float backoff, int interval,
                                                             float* __restrict__ norm_out) {
    __shared__ double red[1024];
    double acc = 0.0;
    bool bad = false;
    for (int i = threadIdx.x; i < nblocks; i += 1024) {
        acc += (double)scratch[kScHdr + i];
        bad |= scratch[kScHdr + kSumsqBlocks + i] != 0.f;
    }
    bad = __syncthreads_or(bad);
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x != 0) return;
    const float S = st->scale;
    const float norm = sqrtf((float)red[0]);
    if (norm_out) *norm_out = norm;
    scratch[kScInv] = inv_scale_of(S);
    scratch[kScCoef] = max_norm > 0.f ? fminf(max_norm / (norm + 1e-6f), 1.0f) : 1.0f;
    scratch[kScApply] = bad ? 0.f : 1.f;
    if (bad) {                                     // GradScaler.step skips optimizer.step(); update() backs off
        st->found_inf = 1;
        st->skipped_steps += 1;
        st->scale = S * backoff;
        st->growth_tracker = 0;
        return;
    }
    st->found_inf = 0;
    const int step = ++st->optimizer_steps;
    scratch[kScStepSize] = (float)((double)lr / (1.0 - pow((double)b1, (double)step)));
    scratch[kScBc2Sqrt] = (float)sqrt(1.0 - pow((double)b2, (double)step));
    const int tracker = st->growth_tracker + 1;    // torch._amp_update_scale_
    if (tracker == interval) {
        const float grown = S * growth;
        if (isfinite(grown)) st->scale = grown;
        st->growth_tracker = 0;
    } else {
        st->growth_tracker = tracker;
    }
}
__global__ void __launch_bounds__(256) adamw_scaled_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                            float* __restrict__ v, float* __restrict__ ema, size_t n, float b1, float b2, float eps,
                                                            float lr_wd, const float* __restrict__ scratch, float ema_decay) {
    const bool apply = scratch[kScApply] != 0.f;
    if (!apply && !ema) return;
    const float inv = scratch[kScInv], coef = scratch[kScCoef], step_size = scratch[kScStepSize], bc2_sqrt = scratch[kScBc2Sqrt];
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float pi = p[i];
        if (apply) {
            const float gi = (g[i] * inv) * coef;
            pi *= 1.0f - lr_wd;
            const float mi = b1 * m[i] + (1.0f - b1) * gi, vi = b2 * v[i] + (1.0f - b2) * gi * gi;
            m[i] = mi; v[i] = vi;
            pi -= step_size * mi / (sqrtf(vi) / bc2_sqrt + eps);
            p[i] = pi;
        }
        if (ema) ema[i] -= (1.0f - ema_decay) * (ema[i] - pi);
    }
}
int launch_adamw_scaled(float* p, const float* g, float* m, float* v, float* ema, size_t n, float lr, float b1, float b2, float eps, float wd,
                        float max_norm, float ema_decay, pd_grad_scaler_state_t* state, float growth, float backoff, int interval,
                        float* scratch, float* norm_out, cudaStream_t s) {
    const int grid = (int)std::min<size_t>((n + 255) / 256, kSumsqBlocks);
    sumsq_unscale_kernel<<<grid, 256, 0, s>>>(g, n, state, scratch);
    scaler_decide_kernel<<<1, 1024, 0, s>>>(scratch, grid, state, lr, b1, b2, max_norm, growth, backoff, interval, norm_out);
    adamw_scaled_kernel<<<grid, 256, 0, s>>>(p, g, m, v, ema, n, b1, b2, eps, lr * wd, scratch, ema_decay);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// mixed-precision (bf16 tensor-core) path: casts between the fp32 activations / gradients and the 16-bit conv operands
// ---------------------------------------------------------------------------------------------------------------------
// OIHW (O, I, k, k) fp32 -> 16-bit dgrad GEMM weights (Isub, k*k*O) for input channels [i0, i0 + Isub): K index = tap' * O + o with
// tap' the FLIPPED tap, so that the stride-1 tensor-core conv computes dX = conv(dY, W^T flipped)
template <typename T>
__global__ void relayout_tc_dgrad_kernel(const float* __restrict__ w, int O, int I, int k, int i0, int Isub, T* __restrict__ out, int ktot,
                                         int koff, int ostride) {
    const int kk = k * k;
    const size_t total = (size_t)Isub * kk * O;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int o = idx % O;
        const size_t r = idx / O;
        const int tapf = r % kk, i = r / kk;
        out[(size_t)i * ktot + koff + (size_t)tapf * ostride + o] = from_f<T>(w[((size_t)o * I + i0 + i) * kk + (kk - 1 - tapf)]);
    }
}
// ktot / koff: row pitch and column offset of `out` (several weights side by side along K, e.g. the fused q / k / v projection); 0: k*k*O
// ostride: K distance between taps (output channels zero-padded to ostride, the caller zeroes `out`); 0: O
int launch_relayout_tc_dgrad(int dt, const float* w, int O, int I, int k, int i0, int Isub, void* out, cudaStream_t s, int ktot, int koff, int ostride) {
    const size_t total = (size_t)k * k * O * Isub;
    if (ostride <= 0) ostride = O;
    if (ktot <= 0) { ktot = k * k * ostride; koff = 0; }
    const int grid = (int)std::min<size_t>((total + 255) / 256, 4096);
    PD_DISPATCH_HALF(dt, T, (relayout_tc_dgrad_kernel<T><<<grid, 256, 0, s>>>(w, O, I, k, i0, Isub, (T*)out, ktot, koff, ostride)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}


// out16 = T(x) (n a multiple of 8)
template <typename T>
__global__ void __launch_bounds__(256) f2h_kernel(const float4* __restrict__ x, Half8<T>* __restrict__ out, size_t n8) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
        const float4 a = x[2 * i], b = x[2 * i + 1];
        Half8<T> h;
        h.v[0] = from_f<T>(a.x); h.v[1] = from_f<T>(a.y); h.v[2] = from_f<T>(a.z); h.v[3] = from_f<T>(a.w);
        h.v[4] = from_f<T>(b.x); h.v[5] = from_f<T>(b.y); h.v[6] = from_f<T>(b.z); h.v[7] = from_f<T>(b.w);
        out[i] = h;
    }
}
int launch_f2h(int dt, const float* x, void* out, size_t n, cudaStream_t s) {
    PD_REQUIRE(n % 8 == 0, "f2h: element count must be a multiple of 8");
    const int grid = (int)std::min<size_t>((n / 8 + 255) / 256, 148 * 16);
    PD_DISPATCH_HALF(dt, T, (f2h_kernel<T><<<grid, 256, 0, s>>>((const float4*)x, (Half8<T>*)out, n / 8)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// forward epilogue of a tensor-core conv: out = (float(y16) + addvec[img] + residual) * scale      (rows of C channels, HW rows per image)
// ACC: out += float(y16) (gradient accumulation of a tensor-core dgrad)
template <typename T, bool ACC>
__global__ void __launch_bounds__(256) h2f_kernel(const Half8<T>* __restrict__ y, const float* __restrict__ addvec, const float4* __restrict__ residual,
                                                  float scale, float4* __restrict__ out, size_t n8, int C8, size_t per_img8) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
        const Half8<T> h = y[i];
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = to_f(h.v[j]);
        if (ACC) {
            const float4 a = out[2 * i], b = out[2 * i + 1];
            out[2 * i] = make_float4(a.x + v[0], a.y + v[1], a.z + v[2], a.w + v[3]);
            out[2 * i + 1] = make_float4(b.x + v[4], b.y + v[5], b.z + v[6], b.w + v[7]);
        } else {
            if (addvec) {
                const float* av = addvec + (i / per_img8) * (size_t)(C8 * 8) + (i % C8) * 8;
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] += av[j];
            }
            if (residual) {
                const float4 a = residual[2 * i], b = residual[2 * i + 1];
                v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
            }
            out[2 * i] = make_float4(v[0] * scale, v[1] * scale, v[2] * scale, v[3] * scale);
            out[2 * i + 1] = make_float4(v[4] * scale, v[5] * scale, v[6] * scale, v[7] * scale);
        }
    }
}
int launch_h2f_epilogue(int dt, const void* y16, const float* addvec, const float* residual, float scale, float* out, int B, int HW, int C,
                        cudaStream_t s) {
    PD_REQUIRE(C % 8 == 0, "h2f: channel count must be a multiple of 8");
    const size_t n8 = (size_t)B * HW * C / 8;
    const int grid = (int)std::min<size_t>((n8 + 255) / 256, 148 * 16);
    PD_DISPATCH_HALF(dt, T, (h2f_kernel<T, false><<<grid, 256, 0, s>>>((const Half8<T>*)y16, addvec, (const float4*)residual, scale, (float4*)out,
                                                                        n8, C / 8, (size_t)HW * C / 8)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}
int launch_h2f_accumulate(int dt, const void* y16, float* out, size_t n, cudaStream_t s) {
    PD_REQUIRE(n % 8 == 0, "h2f: element count must be a multiple of 8");
    const int grid = (int)std::min<size_t>((n / 8 + 255) / 256, 148 * 16);
    PD_DISPATCH_HALF(dt, T, (h2f_kernel<T, true><<<grid, 256, 0, s>>>((const Half8<T>*)y16, nullptr, nullptr, 1.f, (float4*)out, n / 8, 1, 1)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// dW (O, I, k, k) += stage (k*k, O, I): the tensor-core wgrad accumulates into a [tap][co][ci] staging buffer (coalesced vector
// reductions); this folds it into the OIHW gradient
__global__ void wgrad_unstage_kernel(const float* __restrict__ stage, int O, int I, int kk, float* __restrict__ dw, int Opad, int Ipad) {
    const size_t total = (size_t)O * I * kk;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int tap = idx % kk;
        const size_t oi = idx / kk;
        const int i = oi % I, o = oi / I;
        dw[idx] += stage[((size_t)tap * Opad + o) * Ipad + i];
    }
}
// Opad / Ipad: extents of the staging tile when the GEMM ran on zero-padded channels (conv_in, conv_out); 0: O / I
int launch_wgrad_unstage(const float* stage, int O, int I, int kk, float* dw, cudaStream_t s, int Opad, int Ipad) {
    const size_t total = (size_t)O * I * kk;
    if (Opad <= 0) Opad = O;
    if (Ipad <= 0) Ipad = I;
    wgrad_unstage_kernel<<<(int)std::min<size_t>((total + 255) / 256, 148 * 8), 256, 0, s>>>(stage, O, I, kk, dw, Opad, Ipad);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// OIHW (O, I, 3, 3) fp32 -> 16-bit phase weights of the stride-2 (padding 1) dgrad, in the layout of the halo kernel's upsample mode:
// dX(2i + a, 2j + b) = sum_{dr, dc} Wd[(a, b)][(dr, dc)] dY(i - 1 + a + dr, j - 1 + b + dc); out (4*I, 4*O), row = (a*2+b)*I + i,
// k = (dr*2+dc)*O + o.  Input row 2i + a receives kernel row r through output row (2i + a + 1 - r) / 2: a = 0 -> r = 1 (dr = 1);
// a = 1 -> r = 2 (dr = 0), r = 0 (dr = 1); the remaining (a, dr) = (0, 0) slot is zero.  Same for columns.
template <typename T>
__global__ void relayout_tc_dgrad_s2_kernel(const float* __restrict__ w, int O, int I, T* __restrict__ out) {
    const size_t total = (size_t)16 * O * I;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int o = idx % O;
        size_t q = idx / O;
        const int tap = q % 4; q /= 4;
        const int i = q % I;
        const int ph = q / I;
        const int a = ph >> 1, b = ph & 1, dr = tap >> 1, dc = tap & 1;
        const int r = a == 0 ? (dr == 1 ? 1 : -1) : (dr == 0 ? 2 : 0);
        const int sx = b == 0 ? (dc == 1 ? 1 : -1) : (dc == 0 ? 2 : 0);
        out[idx] = from_f<T>((r < 0 || sx < 0) ? 0.f : w[((size_t)o * I + i) * 9 + r * 3 + sx]);
    }
}
int launch_relayout_tc_dgrad_s2(int dt, const float* w, int O, int I, void* out, cudaStream_t s) {
    const size_t total = (size_t)16 * O * I;
    const int grid = (int)std::min<size_t>((total + 255) / 256, 4096);
    PD_DISPATCH_HALF(dt, T, (relayout_tc_dgrad_s2_kernel<T><<<grid, 256, 0, s>>>(w, O, I, (T*)out)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// column sums of dY (M rows x C fp32) in one pass, four columns per thread: out_all[c] += sum over all rows, out_img[n][c] += sum over
// image n's rows (either may be null), and optionally the 16-bit copy of dY that the tensor-core dgrad / wgrad read (same pass).
template <typename T>
__global__ void __launch_bounds__(256) colsum_cast_kernel(const float4* __restrict__ dy, int C4, int rows_per_img, int rows_per_block,
                                                          float* __restrict__ out_all, float* __restrict__ out_img, T* __restrict__ out16) {
    __shared__ float4 red[256];
    const int img = blockIdx.y;
    const int r0 = blockIdx.x * rows_per_block, r1 = min(r0 + rows_per_block, rows_per_img);
    const int rstep = max(1, 256 / C4);
    const size_t base = (size_t)img * rows_per_img;
    for (int cg0 = 0; cg0 < C4; cg0 += 256) {
        const int cg = cg0 + (C4 >= 256 ? threadIdx.x : threadIdx.x % C4);
        const int rr = C4 >= 256 ? 0 : threadIdx.x / C4;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cg < C4 && rr < rstep) {
#pragma unroll 4
            for (int r = r0 + rr; r < r1; r += rstep) {
                const float4 v = dy[(base + r) * C4 + cg];
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
                if (out16) {
                    T* o = out16 + ((base + r) * C4 + cg) * 4;
                    union { T h[4]; uint2 u; } pk;
                    pk.h[0] = from_f<T>(v.x); pk.h[1] = from_f<T>(v.y); pk.h[2] = from_f<T>(v.z); pk.h[3] = from_f<T>(v.w);
                    *reinterpret_cast<uint2*>(o) = pk.u;
                }
            }
        }
        red[threadIdx.x] = acc;
        __syncthreads();
        if (rr == 0 && cg < C4) {
            for (int k = 1; k < rstep; ++k) {
                const float4 v = red[threadIdx.x + k * C4];
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
            if (out_all) {
                float* o = out_all + cg * 4;
                atomicAdd(o, acc.x); atomicAdd(o + 1, acc.y); atomicAdd(o + 2, acc.z); atomicAdd(o + 3, acc.w);
            }
            if (out_img) {
                float* o = out_img + ((size_t)img * C4 + cg) * 4;
                atomicAdd(o, acc.x); atomicAdd(o + 1, acc.y); atomicAdd(o + 2, acc.z); atomicAdd(o + 3, acc.w);
            }
        }
        __syncthreads();
    }
}
int launch_colsum_cast(int dt, const float* dy, int B, int rows_per_img, int C, float* out_all, float* out_img, void* out16, cudaStream_t s) {
    PD_REQUIRE(C % 4 == 0, "colsum_cast: channel count must be a multiple of 4");
    const int rpb = 256;
    dim3 grid((rows_per_img + rpb - 1) / rpb, B);
    if (dt == DT_F16) colsum_cast_kernel<f16><<<grid, 256, 0, s>>>((const float4*)dy, C / 4, rows_per_img, rpb, out_all, out_img, (f16*)out16);
    else colsum_cast_kernel<bf16><<<grid, 256, 0, s>>>((const float4*)dy, C / 4, rows_per_img, rpb, out_all, out_img, (bf16*)out16);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

template <typename T>
__global__ void __launch_bounds__(256) nchw_to_nhwc16_pad_kernel(const float* __restrict__ x, int C, size_t HW, int Cp, T* __restrict__ out, size_t total8) {
    const int Cp8 = Cp / 8;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total8; i += (size_t)gridDim.x * blockDim.x) {
        const int cg = i % Cp8;
        const size_t pix = i / Cp8;
        const size_t n = pix / HW, p = pix - n * HW;
        Half8<T> h;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int c = cg * 8 + j;
            h.v[j] = from_f<T>(c < C ? x[(n * C + c) * HW + p] : 0.f);
        }
        reinterpret_cast<Half8<T>*>(out)[i] = h;
    }
}
int launch_nchw_to_nhwc16_pad(int dt, const float* x, int N, int C, int HW, int Cp, void* out, cudaStream_t s) {
    PD_REQUIRE(Cp % 8 == 0 && C <= Cp, "nchw_to_nhwc16_pad: padded channel count must be a multiple of 8");
    const size_t total8 = (size_t)N * HW * (Cp / 8);
    const int grid = (int)std::min<size_t>((total8 + 255) / 256, 148 * 16);
    PD_DISPATCH_HALF(dt, T, (nchw_to_nhwc16_pad_kernel<T><<<grid, 256, 0, s>>>(x, C, (size_t)HW, Cp, (T*)out, total8)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// gradient-guided generation (SURVEY §8 row f4; reference _custom_guided_generation, src/utils_Img2Img.py:716-745):
//   x0 = pred_original_sample(x_t, m)  (DDIMScheduler.step: by prediction type, clipped);  loss_i = || x0_i - ref_i ||_p  (Lp_loss, :245-270)
// pass 1 reduces sum |d|^p per image, pass 2 writes the loss and its gradients w.r.t. the model output (the upstream gradient of the
// UNet's backward) and w.r.t. x_t directly (the path that does not go through the UNet).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float guidance_x0(const pd_step_coeffs_t& c, float x, float m, float* dx0_dx, float* dx0_dm) {
    float x0;
    if (c.pred_type == PD_PRED_EPSILON) { x0 = (x - c.sqrt_beta * m) / c.sqrt_alpha; *dx0_dx = 1.0f / c.sqrt_alpha; *dx0_dm = -c.sqrt_beta / c.sqrt_alpha; }
    else if (c.pred_type == PD_PRED_SAMPLE) { x0 = m; *dx0_dx = 0.f; *dx0_dm = 1.f; }
    else { x0 = c.sqrt_alpha * x - c.sqrt_beta * m; *dx0_dx = c.sqrt_alpha; *dx0_dm = -c.sqrt_beta; }
    if (c.clip) {
        // torch.clamp: the gradient passes where -r <= x0 <= r (bounds included)
        if (!(x0 >= -c.clip_range && x0 <= c.clip_range)) { *dx0_dx = 0.f; *dx0_dm = 0.f; }
        x0 = (x0 < -c.clip_range) ? -c.clip_range : ((x0 > c.clip_range) ? c.clip_range : x0);
    }
    return x0;
}
__global__ void __launch_bounds__(256) guidance_lp_reduce_kernel(pd_step_coeffs_t c, const float* __restrict__ x, const float* __restrict__ m,
                                                                 const float* __restrict__ ref, size_t per, float p, float* __restrict__ sums) {
    __shared__ float red[8];
    const int img = blockIdx.y;
    const size_t base = (size_t)img * per;
    float acc = 0.f;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < per; i += (size_t)gridDim.x * blockDim.x) {
        float a, b;
        const float d = fabsf(guidance_x0(c, x[base + i], m[base + i], &a, &b) - ref[base + i]);
        acc += p == 2.f ? d * d : (p == 1.f ? d : powf(d, p));
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        atomicAdd(sums + img, t);
    }
}
__global__ void __launch_bounds__(256) guidance_lp_grad_kernel(pd_step_coeffs_t c, const float* __restrict__ x, const float* __restrict__ m,
                                                               const float* __restrict__ ref, size_t per, float p, const float* __restrict__ sums,
                                                               float* __restrict__ losses, float* __restrict__ dm, float* __restrict__ dx) {
    const int img = blockIdx.y;
    const size_t base = (size_t)img * per;
    const float sum = sums[img];
    const float loss = p == 2.f ? sqrtf(sum) : (p == 1.f ? sum : powf(sum, 1.0f / p));
    if (blockIdx.x == 0 && threadIdx.x == 0 && losses) losses[img] = loss;
    // d loss / d d_j = sign(d_j) |d_j|^(p-1) / loss^(p-1)   (0 where the norm is 0)
    const float inv = loss > 0.f ? (p == 2.f ? 1.0f / loss : (p == 1.f ? 1.0f : powf(loss, 1.0f - p))) : 0.f;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < per; i += (size_t)gridDim.x * blockDim.x) {
        float a, b;
        const float d = guidance_x0(c, x[base + i], m[base + i], &a, &b) - ref[base + i];
        const float ad = fabsf(d);
        const float mag = p == 2.f ? ad : (p == 1.f ? (ad > 0.f ? 1.f : 0.f) : (ad > 0.f ? powf(ad, p - 1.0f) : 0.f));
        const float g = (d < 0.f ? -mag : mag) * inv;
        dm[base + i] = g * b;
        dx[base + i] = g * a;
    }
}
int launch_guidance_lp_grad(const pd_step_coeffs_t& c, const float* x, const float* m, const float* ref, int B, size_t per, float p, float* sums,
                            float* losses, float* dm, float* dx, cudaStream_t s) {
    PD_REQUIRE(p > 0.f && isfinite(p), "guidance loss: p must be a finite positive number (the 'inf' norms are not implemented)");
    PD_CHECK_CUDA(cudaMemsetAsync(sums, 0, (size_t)B * sizeof(float), s));
    dim3 grid((unsigned)std::min<size_t>((per + 255) / 256, 64), B);
    guidance_lp_reduce_kernel<<<grid, 256, 0, s>>>(c, x, m, ref, per, p, sums);
    guidance_lp_grad_kernel<<<grid, 256, 0, s>>>(c, x, m, ref, per, p, sums, losses, dm, dx);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// (N, HW, Cp) 16-bit or fp32 NHWC -> first C channels as NCHW fp32 (the input gradient of conv_in leaves the library in the boundary layout)
template <typename T>
__global__ void nhwc_to_nchw_f32_kernel(const T* __restrict__ x, int C, size_t HW, int Cp, float* __restrict__ out, size_t total) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t p = i % HW;
        const size_t nc = i / HW;
        const int c = nc % C;
        const size_t n = nc / C;
        out[i] = to_f(x[(n * HW + p) * Cp + c]);
    }
}
int launch_nhwc_to_nchw_f32(int dt, const void* x, int N, int C, int HW, int Cp, float* out, cudaStream_t s) {
    const size_t total = (size_t)N * C * HW;
    const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
    if (dt == DT_F32) nhwc_to_nchw_f32_kernel<float><<<grid, 256, 0, s>>>((const float*)x, C, (size_t)HW, Cp, out, total);
    else if (dt == DT_BF16) nhwc_to_nchw_f32_kernel<bf16><<<grid, 256, 0, s>>>((const bf16*)x, C, (size_t)HW, Cp, out, total);
    else nhwc_to_nchw_f32_kernel<f16><<<grid, 256, 0, s>>>((const f16*)x, C, (size_t)HW, Cp, out, total);
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// forward epilogue of a tensor-core conv fused with the GroupNorm chunk statistics of its fp32 result (the consumer's GroupNorm would
// otherwise re-read the tensor): out = (float(y16) + addvec[img] + residual) * scale, stats[img][chunk] += (sum, sum of squares) of out.
// Same thread mapping and pivoted fp32 partials -> fp64 atomics as gn_chunk_stats_kernel (pd_kernels_simt.cu).
template <typename T>
__global__ void __launch_bounds__(256) h2f_stats_kernel(const Half8<T>* __restrict__ y, const float* __restrict__ addvec, const float* __restrict__ residual,
                                                        float scale, float* __restrict__ out, int HW, int C, int cw, int rows_per_block,
                                                        double* __restrict__ stats) {
    const int ncv = C / 8;
    const int n = blockIdx.y;
    const int cv = threadIdx.x % ncv, r0 = threadIdx.x / ncv, rstep = blockDim.x / ncv;
    if (r0 >= rstep) return;
    const int row_begin = blockIdx.x * rows_per_block, row_end = min(row_begin + rows_per_block, HW);
    const size_t base = (size_t)n * HW;
    float av[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) av[i] = addvec ? addvec[(size_t)n * C + cv * 8 + i] : 0.f;
    float s[8], q[8], pv[8];
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { s[i] = 0.f; q[i] = 0.f; pv[i] = 0.f; }
#pragma unroll 2
    for (int r = row_begin + r0; r < row_end; r += rstep) {
        const size_t e = (base + r) * C + cv * 8;
        const Half8<T> h = y[e / 8];
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = to_f(h.v[i]) + av[i];
        if (residual) {
            const float4 a = *reinterpret_cast<const float4*>(residual + e), b = *reinterpret_cast<const float4*>(residual + e + 4);
            v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] *= scale;
        *reinterpret_cast<float4*>(out + e) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(out + e + 4) = make_float4(v[4], v[5], v[6], v[7]);
        if (cnt == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) pv[i] = v[i];
        }
        ++cnt;
#pragma unroll
        for (int i = 0; i < 8; ++i) { const float d = v[i] - pv[i]; s[i] += d; q[i] += d * d; }
    }
    if (cnt == 0) return;
    double S[8], Q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const double pd_ = (double)pv[i], nn = (double)cnt;
        S[i] = nn * pd_ + (double)s[i];
        Q[i] = (double)q[i] + 2.0 * pd_ * (double)s[i] + nn * pd_ * pd_;
    }
    double* dst = stats + ((size_t)n * (C / cw) + (cv * 8) / cw) * 2;
    if (cw == 4) {
        atomicAdd(dst + 0, (S[0] + S[1]) + (S[2] + S[3])); atomicAdd(dst + 1, (Q[0] + Q[1]) + (Q[2] + Q[3]));
        atomicAdd(dst + 2, (S[4] + S[5]) + (S[6] + S[7])); atomicAdd(dst + 3, (Q[4] + Q[5]) + (Q[6] + Q[7]));
    } else if (cw == 2) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { atomicAdd(dst + 2 * j, S[2 * j] + S[2 * j + 1]); atomicAdd(dst + 2 * j + 1, Q[2 * j] + Q[2 * j + 1]); }
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) { atomicAdd(dst + 2 * j, S[j]); atomicAdd(dst + 2 * j + 1, Q[j]); }
    }
}
int launch_h2f_epilogue_stats(int dt, const void* y16, const float* addvec, const float* residual, float scale, float* out, int B, int HW, int C,
                              int cw, double* stats, cudaStream_t s) {
    PD_REQUIRE(C % 8 == 0 && C / 8 <= 256 && (cw == 4 || cw == 2 || cw == 1), "h2f_stats: channel count must be a multiple of 8 (<= 2048)");
    const int ncv = C / 8, rstep = 256 / ncv;
    int rows = rstep * 16;
    if (rows > HW) rows = HW;
    dim3 grid((HW + rows - 1) / rows, B);
    PD_DISPATCH_HALF(dt, T, (h2f_stats_kernel<T><<<grid, 256, 0, s>>>((const Half8<T>*)y16, addvec, residual, scale, out, HW, C, cw, rows, stats)));
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace pd
