// phendiff_b200 — softmax attention of the TRAINING step on the warp-level tensor cores (head_dim 8; SURVEY §8 row f2, A.2): the
// forward that also stores the log-sum-exp of every query row, and the backward that recomputes the probabilities from it
// (dQ by a query-stationary kernel, dK / dV by a key-stationary kernel: no atomics, the exponentials are paid twice).
//
// q, k, v, out and their gradients are the fp32 NHWC activations of the training walk ((N, S, pitch) rows, head h at channels 8h..8h+7);
// operands are rounded to the 16-bit type of the run (bf16, or fp16 for mixed_precision="fp16") when they are staged in shared memory ([row][8 dims] = 16-byte rows, the whole head at once), the
// products accumulate in fp32: S = Q K^T and dP = dO V^T are m16n8k8 MMAs (K = the 8 head dims), P V, dS K, P^T dO, dS^T Q are
// m16n8k16 MMAs whose A operand is the accumulator fragment of the previous product re-packed in registers and whose B operand
// comes from the same 16-byte rows through ldmatrix.trans.  Scores are kept in the log2 domain (Q is pre-scaled by
// log2(e) / sqrt(8)), one ex2.approx per score.
// One CTA = 16 warps = 256 rows of one (image, head), each warp owns 16 rows (8 warps: -3 % on the step, 4 warps: -9 %: the CTA stages the
// whole head for its rows, so fewer rows per CTA means more staging traffic per score).  Validated against torch.autograd on the oracle
// through tests/test_gpu_training.py (bf16) and tests/test_gpu_training_fp16.py (fp16); the fp32 kernels in pd_train_kernels.cu remain the validation path.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "pd_kernels.h"
#include "pd_train.h"

namespace pd {

namespace {

constexpr float kScale8 = 0.35355339059327373f;       // 1 / sqrt(8)
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
#ifndef TRAIN_AT_WARPS
#define TRAIN_AT_WARPS 16       // warps per CTA; each owns 16 rows, the CTA stages the whole head once for all of them
#endif
constexpr int AT_THREADS = 32 * TRAIN_AT_WARPS, AT_ROWS = 16 * TRAIN_AT_WARPS;
#ifndef AT_KB
#define AT_KB 64          // keys (queries) per iteration of the backward kernels: independent MMA / ex2 chains in flight per warp
#endif

// T = bf16 or f16: the operand type of every MMA (both accumulate in fp32)
template <typename T> __device__ __forceinline__ uint32_t pack_h(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack_h<bf16>(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
template <> __device__ __forceinline__ uint32_t pack_h<f16>(float lo, float hi) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
template <typename T> __device__ __forceinline__ void mma_k8(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
    if constexpr (std::is_same<T, f16>::value)
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%0, %1, %2, %3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(b0));
    else
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%0, %1, %2, %3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(b0));
}
template <typename T>
__device__ __forceinline__ void mma_k16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    if constexpr (std::is_same<T, f16>::value)
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    else
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                     : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// B fragment (k = 16 rows, n = 8 dims) of a [row][8] 16-bit tile starting at `row0`: ldmatrix.trans of two 8x8 matrices
__device__ __forceinline__ void ldsm_t2(uint32_t& b0, uint32_t& b1, const uint4* tile, int row0, int lane) {
    const uint32_t addr = static_cast<uint32_t>(__cvta_generic_to_shared(tile + row0 + (lane & 15)));
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(addr));
}
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// stage rows [0, S) of one head (8 fp32 at `src + row * pitch`) as 16-bit 16-byte rows, scaled
template <typename T>
__device__ __forceinline__ void stage_rows(uint4* dst, const float* src, size_t pitch, int S, float scale) {
    for (int r = threadIdx.x; r < S; r += AT_THREADS) {
        const float4 a = *reinterpret_cast<const float4*>(src + (size_t)r * pitch), b = *reinterpret_cast<const float4*>(src + (size_t)r * pitch + 4);
        uint4 v;
        v.x = pack_h<T>(a.x * scale, a.y * scale); v.y = pack_h<T>(a.z * scale, a.w * scale);
        v.z = pack_h<T>(b.x * scale, b.y * scale); v.w = pack_h<T>(b.z * scale, b.w * scale);
        dst[r] = v;
    }
}
// A fragment (16 rows x 8 dims) of this warp's rows straight from global fp32: a0 = (row g, dims 2t, 2t+1), a1 = (row g + 8, ...)
template <typename T>
__device__ __forceinline__ void load_a_frag(uint32_t& a0, uint32_t& a1, const float* src, size_t pitch, int row0, int g, int t, float scale) {
    const float2 lo = *reinterpret_cast<const float2*>(src + (size_t)(row0 + g) * pitch + 2 * t);
    const float2 hi = *reinterpret_cast<const float2*>(src + (size_t)(row0 + g + 8) * pitch + 2 * t);
    a0 = pack_h<T>(lo.x * scale, lo.y * scale);
    a1 = pack_h<T>(hi.x * scale, hi.y * scale);
}

// ---- forward ------------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(AT_THREADS) attn8_mma_fwd_kernel(const float* __restrict__ qp, const float* __restrict__ kp, const float* __restrict__ vp,
                                                                    int pitch, int S, int C, float* __restrict__ out, float* __restrict__ lse) {
    extern __shared__ uint4 sm4[];
    uint4 *Ks = sm4, *Vs = sm4 + S;
    const int n = blockIdx.z, head = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const size_t off = (size_t)n * S * pitch + head * 8;
    stage_rows<T>(Ks, kp + off, pitch, S, 1.f);
    stage_rows<T>(Vs, vp + off, pitch, S, 1.f);
    const int q0 = blockIdx.x * AT_ROWS + warp * 16;
    uint32_t qa0, qa1;
    load_a_frag<T>(qa0, qa1, qp + off, pitch, q0, g, t, kScale8 * kLog2e);
    __syncthreads();
    float o[4] = {0.f, 0.f, 0.f, 0.f};
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;   // rows g and g + 8 (l: this thread's partial sums)
    const uint32_t* Kw = reinterpret_cast<const uint32_t*>(Ks);
    for (int k0 = 0; k0 < S; k0 += 64) {
        float c[8][4];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            c[j][0] = c[j][1] = c[j][2] = c[j][3] = 0.f;
            mma_k8<T>(c[j], qa0, qa1, Kw[(size_t)(k0 + 8 * j + g) * 4 + t]);
        }
        float bm0 = c[0][0], bm1 = c[0][2];
#pragma unroll
        for (int j = 0; j < 8; ++j) { bm0 = fmaxf(bm0, fmaxf(c[j][0], c[j][1])); bm1 = fmaxf(bm1, fmaxf(c[j][2], c[j][3])); }
        bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 1)); bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 2));
        bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 1)); bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 2));
        const float nm0 = fmaxf(m0, bm0), nm1 = fmaxf(m1, bm1);
        const float cr0 = ex2(m0 - nm0), cr1 = ex2(m1 - nm1);
        m0 = nm0; m1 = nm1;
        l0 *= cr0; l1 *= cr1; o[0] *= cr0; o[1] *= cr0; o[2] *= cr1; o[3] *= cr1;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            c[j][0] = ex2(c[j][0] - nm0); c[j][1] = ex2(c[j][1] - nm0); c[j][2] = ex2(c[j][2] - nm1); c[j][3] = ex2(c[j][3] - nm1);
            l0 += c[j][0] + c[j][1]; l1 += c[j][2] + c[j][3];
        }
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            uint32_t b0, b1;
            ldsm_t2(b0, b1, Vs, k0 + 8 * j, lane);
            mma_k16<T>(o, pack_h<T>(c[j][0], c[j][1]), pack_h<T>(c[j][2], c[j][3]), pack_h<T>(c[j + 1][0], c[j + 1][1]),
                    pack_h<T>(c[j + 1][2], c[j + 1][3]), b0, b1);
        }
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = 1.f / l0, i1 = 1.f / l1;
    float* o0 = out + ((size_t)n * S + q0 + g) * C + head * 8 + 2 * t;
    *reinterpret_cast<float2*>(o0) = make_float2(o[0] * i0, o[1] * i0);
    *reinterpret_cast<float2*>(o0 + (size_t)8 * C) = make_float2(o[2] * i1, o[3] * i1);
    if (t == 0) {
        float* L = lse + ((size_t)n * (C / 8) + head) * S + q0 + g;
        L[0] = (m0 + log2f(l0)) * kLn2;
        L[8] = (m1 + log2f(l1)) * kLn2;
    }
}

// ---- backward, query-stationary: dQ, and delta[q] = sum_d dO[q, d] O[q, d] -------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(AT_THREADS) attn8_mma_bwd_q_kernel(const float* __restrict__ qp, const float* __restrict__ kp, const float* __restrict__ vp,
                                                                      int pitch, const float* __restrict__ o, const float* __restrict__ dout,
                                                                      const float* __restrict__ lse, int S, int C, float* __restrict__ dq_out,
                                                                      float* __restrict__ delta) {
    extern __shared__ uint4 sm4[];
    uint4 *Ks = sm4, *Vs = sm4 + S;
    const int n = blockIdx.z, head = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const size_t off = (size_t)n * S * pitch + head * 8;
    stage_rows<T>(Ks, kp + off, pitch, S, 1.f);
    stage_rows<T>(Vs, vp + off, pitch, S, 1.f);
    const int q0 = blockIdx.x * AT_ROWS + warp * 16;
    uint32_t qa0, qa1, ga0, ga1;
    load_a_frag<T>(qa0, qa1, qp + off, pitch, q0, g, t, kScale8 * kLog2e);
    const size_t orow = ((size_t)n * S + q0 + g) * C + head * 8 + 2 * t;
    const float2 g_lo = *reinterpret_cast<const float2*>(dout + orow), g_hi = *reinterpret_cast<const float2*>(dout + orow + (size_t)8 * C);
    const float2 o_lo = *reinterpret_cast<const float2*>(o + orow), o_hi = *reinterpret_cast<const float2*>(o + orow + (size_t)8 * C);
    ga0 = pack_h<T>(g_lo.x, g_lo.y); ga1 = pack_h<T>(g_hi.x, g_hi.y);
    float d0 = g_lo.x * o_lo.x + g_lo.y * o_lo.y, d1 = g_hi.x * o_hi.x + g_hi.y * o_hi.y;
    d0 += __shfl_xor_sync(0xffffffffu, d0, 1); d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 1); d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    const size_t lrow = ((size_t)n * (C / 8) + head) * S + q0 + g;
    const float L0 = lse[lrow] * kLog2e, L1 = lse[lrow + 8] * kLog2e;
    if (t == 0) { delta[lrow] = d0; delta[lrow + 8] = d1; }
    __syncthreads();
    float dq[4] = {0.f, 0.f, 0.f, 0.f};
    const uint32_t* Kw = reinterpret_cast<const uint32_t*>(Ks);
    const uint32_t* Vw = reinterpret_cast<const uint32_t*>(Vs);
    for (int k0 = 0; k0 < S; k0 += AT_KB) {
        float c[AT_KB / 8][4], p[AT_KB / 8][4];
#pragma unroll
        for (int j = 0; j < AT_KB / 8; ++j) {
            c[j][0] = c[j][1] = c[j][2] = c[j][3] = 0.f;
            p[j][0] = p[j][1] = p[j][2] = p[j][3] = 0.f;
            const size_t w = (size_t)(k0 + 8 * j + g) * 4 + t;
            mma_k8<T>(c[j], qa0, qa1, Kw[w]);
            mma_k8<T>(p[j], ga0, ga1, Vw[w]);
        }
#pragma unroll
        for (int j = 0; j < AT_KB / 8; ++j) {
            c[j][0] = ex2(c[j][0] - L0) * (p[j][0] - d0); c[j][1] = ex2(c[j][1] - L0) * (p[j][1] - d0);
            c[j][2] = ex2(c[j][2] - L1) * (p[j][2] - d1); c[j][3] = ex2(c[j][3] - L1) * (p[j][3] - d1);
        }
#pragma unroll
        for (int j = 0; j < AT_KB / 8; j += 2) {
            uint32_t b0, b1;
            ldsm_t2(b0, b1, Ks, k0 + 8 * j, lane);
            mma_k16<T>(dq, pack_h<T>(c[j][0], c[j][1]), pack_h<T>(c[j][2], c[j][3]), pack_h<T>(c[j + 1][0], c[j + 1][1]),
                    pack_h<T>(c[j + 1][2], c[j + 1][3]), b0, b1);
        }
    }
    float* dst = dq_out + off + (size_t)(q0 + g) * pitch + 2 * t;
    float2 a = *reinterpret_cast<float2*>(dst), b = *reinterpret_cast<float2*>(dst + (size_t)8 * pitch);
    a.x += dq[0] * kScale8; a.y += dq[1] * kScale8; b.x += dq[2] * kScale8; b.y += dq[3] * kScale8;
    *reinterpret_cast<float2*>(dst) = a;
    *reinterpret_cast<float2*>(dst + (size_t)8 * pitch) = b;
}

// ---- backward, key-stationary: dK, dV ----------------------------------------------------------------------------------------------
// RT = 16-key row tiles per warp: with RT = 2 every staged Q / dO fragment, (lse, delta) pair and ldmatrix feeds two tiles (half the
// shared-memory reads per score, two independent MMA / ex2 chains per warp); the key block per iteration shrinks to keep the registers.
template <typename T, int RT>
__global__ void __launch_bounds__(AT_THREADS) attn8_mma_bwd_kv_kernel(const float* __restrict__ qp, const float* __restrict__ kp, const float* __restrict__ vp,
                                                                       int pitch, const float* __restrict__ dout, const float* __restrict__ lse,
                                                                       const float* __restrict__ delta, int S, int C, float* __restrict__ dk_out,
                                                                       float* __restrict__ dv_out) {
    constexpr int KB = AT_KB / RT;                                   // queries per iteration
    extern __shared__ uint4 sm4[];
    uint4 *Qs = sm4, *Gs = sm4 + S;                                  // Q pre-scaled by log2(e) / sqrt(8); dO
    float2* LD = reinterpret_cast<float2*>(sm4 + 2 * (size_t)S);     // per query: (lse in log2 units, delta)
    const int n = blockIdx.z, head = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const size_t off = (size_t)n * S * pitch + head * 8;
    stage_rows<T>(Qs, qp + off, pitch, S, kScale8 * kLog2e);
    stage_rows<T>(Gs, dout + (size_t)n * S * C + head * 8, C, S, 1.f);
    const size_t lrow = ((size_t)n * (C / 8) + head) * S;
    for (int r = threadIdx.x; r < S; r += AT_THREADS) LD[r] = make_float2(lse[lrow + r] * kLog2e, delta[lrow + r]);
    const int key0 = blockIdx.x * (AT_ROWS * RT) + warp * (16 * RT);
    uint32_t ka0[RT], ka1[RT], va0[RT], va1[RT];
#pragma unroll
    for (int rt = 0; rt < RT; ++rt) {
        load_a_frag<T>(ka0[rt], ka1[rt], kp + off, pitch, key0 + 16 * rt, g, t, 1.f);
        load_a_frag<T>(va0[rt], va1[rt], vp + off, pitch, key0 + 16 * rt, g, t, 1.f);
    }
    __syncthreads();
    float dk[RT][4], dv[RT][4];
#pragma unroll
    for (int rt = 0; rt < RT; ++rt)
#pragma unroll
        for (int i = 0; i < 4; ++i) { dk[rt][i] = 0.f; dv[rt][i] = 0.f; }
    const uint32_t* Qw = reinterpret_cast<const uint32_t*>(Qs);
    const uint32_t* Gw = reinterpret_cast<const uint32_t*>(Gs);
    for (int q0 = 0; q0 < S; q0 += KB) {
        float c[RT][KB / 8][4], p[RT][KB / 8][4];     // c: S^T (rows = keys g / g + 8, cols = queries 2t, 2t + 1), p: dP^T
#pragma unroll
        for (int j = 0; j < KB / 8; ++j) {
            const size_t w = (size_t)(q0 + 8 * j + g) * 4 + t;
            const uint32_t qb = Qw[w], gb = Gw[w];
#pragma unroll
            for (int rt = 0; rt < RT; ++rt) {
                c[rt][j][0] = c[rt][j][1] = c[rt][j][2] = c[rt][j][3] = 0.f;
                p[rt][j][0] = p[rt][j][1] = p[rt][j][2] = p[rt][j][3] = 0.f;
                mma_k8<T>(c[rt][j], ka0[rt], ka1[rt], qb);
                mma_k8<T>(p[rt][j], va0[rt], va1[rt], gb);
            }
        }
#pragma unroll
        for (int j = 0; j < KB / 8; ++j) {
            const float4 ld = *reinterpret_cast<const float4*>(LD + q0 + 8 * j + 2 * t);   // (L, delta) of queries 2t, 2t + 1
#pragma unroll
            for (int rt = 0; rt < RT; ++rt) {
                const float p0 = ex2(c[rt][j][0] - ld.x), p1 = ex2(c[rt][j][1] - ld.z), p2 = ex2(c[rt][j][2] - ld.x), p3 = ex2(c[rt][j][3] - ld.z);
                c[rt][j][0] = p0; c[rt][j][1] = p1; c[rt][j][2] = p2; c[rt][j][3] = p3;
                p[rt][j][0] = p0 * (p[rt][j][0] - ld.y); p[rt][j][1] = p1 * (p[rt][j][1] - ld.w);
                p[rt][j][2] = p2 * (p[rt][j][2] - ld.y); p[rt][j][3] = p3 * (p[rt][j][3] - ld.w);
            }
        }
#pragma unroll
        for (int j = 0; j < KB / 8; j += 2) {
            uint32_t g0, g1, q0r, q1r;
            ldsm_t2(g0, g1, Gs, q0 + 8 * j, lane);
            ldsm_t2(q0r, q1r, Qs, q0 + 8 * j, lane);
#pragma unroll
            for (int rt = 0; rt < RT; ++rt) {
                mma_k16<T>(dv[rt], pack_h<T>(c[rt][j][0], c[rt][j][1]), pack_h<T>(c[rt][j][2], c[rt][j][3]), pack_h<T>(c[rt][j + 1][0], c[rt][j + 1][1]),
                        pack_h<T>(c[rt][j + 1][2], c[rt][j + 1][3]), g0, g1);
                mma_k16<T>(dk[rt], pack_h<T>(p[rt][j][0], p[rt][j][1]), pack_h<T>(p[rt][j][2], p[rt][j][3]), pack_h<T>(p[rt][j + 1][0], p[rt][j + 1][1]),
                        pack_h<T>(p[rt][j + 1][2], p[rt][j + 1][3]), q0r, q1r);
            }
        }
    }
    // Qs carries log2(e) / sqrt(8): dK = sum dS^T q / sqrt(8) = (sum dS^T Qs) * ln 2
#pragma unroll
    for (int rt = 0; rt < RT; ++rt) {
        float* dkp = dk_out + off + (size_t)(key0 + 16 * rt + g) * pitch + 2 * t;
        float* dvp = dv_out + off + (size_t)(key0 + 16 * rt + g) * pitch + 2 * t;
        float2 a = *reinterpret_cast<float2*>(dkp), b = *reinterpret_cast<float2*>(dkp + (size_t)8 * pitch);
        a.x += dk[rt][0] * kLn2; a.y += dk[rt][1] * kLn2; b.x += dk[rt][2] * kLn2; b.y += dk[rt][3] * kLn2;
        *reinterpret_cast<float2*>(dkp) = a;
        *reinterpret_cast<float2*>(dkp + (size_t)8 * pitch) = b;
        a = *reinterpret_cast<float2*>(dvp); b = *reinterpret_cast<float2*>(dvp + (size_t)8 * pitch);
        a.x += dv[rt][0]; a.y += dv[rt][1]; b.x += dv[rt][2]; b.y += dv[rt][3];
        *reinterpret_cast<float2*>(dvp) = a;
        *reinterpret_cast<float2*>(dvp + (size_t)8 * pitch) = b;
    }
}

int set_smem(const void* fn, size_t bytes, bool* done) {
    if (!*done && bytes > 48 * 1024) {
        PD_CHECK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        *done = true;
    }
    return 0;
}

}  // namespace

bool attn8_mma_supported(int S, int C, int pitch) { return S % AT_ROWS == 0 && C % 8 == 0 && pitch % 4 == 0 && (size_t)S * 40 <= 200 * 1024; }

int launch_attn8_mma_fwd(int dt, const float* q, const float* k, const float* v, int pitch, int N, int S, int C, float* out, float* lse,
                         cudaStream_t s) {
    PD_REQUIRE(attn8_mma_supported(S, C, pitch), "attn8_mma: sequence length must be a multiple of 128 (and fit shared memory)");
    PD_REQUIRE(dt == DT_BF16 || dt == DT_F16, "attn8_mma takes bf16 or fp16 operands");
    static bool done[2][PD_MAX_DEVICES] = {};
    const size_t smem = (size_t)S * 32;
    const int ti = dt == DT_F16;
    PD_DISPATCH_HALF(dt, T, {
        int rc = set_smem((const void*)attn8_mma_fwd_kernel<T>, smem, &done[ti][pd_cur_dev()]);
        if (rc) return rc;
        attn8_mma_fwd_kernel<T><<<dim3(S / AT_ROWS, C / 8, N), AT_THREADS, smem, s>>>(q, k, v, pitch, S, C, out, lse);
    });
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

template <typename T>
static int attn8_mma_bwd(const float* q, const float* k, const float* v, int pitch, const float* o, const float* dout, const float* lse, int N,
                         int S, int C, float* dq, float* dk, float* dv, float* delta, cudaStream_t s) {
    static bool done_q[PD_MAX_DEVICES] = {}, done_kv[PD_MAX_DEVICES] = {}, done_kv2[PD_MAX_DEVICES] = {};
    int rc = set_smem((const void*)attn8_mma_bwd_q_kernel<T>, (size_t)S * 32, &done_q[pd_cur_dev()]);
    if (rc) return rc;
    const dim3 grid(S / AT_ROWS, C / 8, N);
    attn8_mma_bwd_q_kernel<T><<<grid, AT_THREADS, (size_t)S * 32, s>>>(q, k, v, pitch, o, dout, lse, S, C, dq, delta);
    static const int rt2 = [] { const char* e = getenv("PHENDIFF_B200_TRAIN_ATTN_RT"); return e ? atoi(e) : 2; }();
    if (rt2 == 2 && S % (2 * AT_ROWS) == 0) {      // two 16-key tiles per warp
        if ((rc = set_smem((const void*)attn8_mma_bwd_kv_kernel<T, 2>, (size_t)S * 40, &done_kv2[pd_cur_dev()]))) return rc;
        attn8_mma_bwd_kv_kernel<T, 2><<<dim3(S / (2 * AT_ROWS), C / 8, N), AT_THREADS, (size_t)S * 40, s>>>(q, k, v, pitch, dout, lse, delta, S, C, dk, dv);
    } else {
        if ((rc = set_smem((const void*)attn8_mma_bwd_kv_kernel<T, 1>, (size_t)S * 40, &done_kv[pd_cur_dev()]))) return rc;
        attn8_mma_bwd_kv_kernel<T, 1><<<grid, AT_THREADS, (size_t)S * 40, s>>>(q, k, v, pitch, dout, lse, delta, S, C, dk, dv);
    }
    PD_CHECK_CUDA(cudaGetLastError());
    return 0;
}

int launch_attn8_mma_bwd(int dt, const float* q, const float* k, const float* v, int pitch, const float* o, const float* dout, const float* lse,
                         int N, int S, int C, float* dq, float* dk, float* dv, float* delta, cudaStream_t s) {
    PD_REQUIRE(attn8_mma_supported(S, C, pitch), "attn8_mma: sequence length must be a multiple of 128 (and fit shared memory)");
    PD_REQUIRE(dt == DT_BF16 || dt == DT_F16, "attn8_mma takes bf16 or fp16 operands");
    PD_DISPATCH_HALF(dt, T, { return attn8_mma_bwd<T>(q, k, v, pitch, o, dout, lse, N, S, C, dq, dk, dv, delta, s); });
    return 0;
}

}  // namespace pd
