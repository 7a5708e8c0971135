// GroupNorm apply arithmetic shared by the stand-alone pass (elementwise.cu gn_apply_kernel) and the conv kernel that
// applies the normalisation to its own input rows in shared memory (conv_kf.cu, APPLY): both must produce the same
// fp16 values bit for bit, so the statistics, the coefficient folding and the per-vector transform live here once.
// Oracle counterpart: oracle/unet.py RB (F.group_norm + FiLM + SiLU; the reference ships no code).
#pragma once
#include "act.cuh"
#include "gn_sums.cuh"
#include "ptx.cuh"

namespace cdc {

// x * sigmoid(x) = x * (0.5 + 0.5 * tanh(x / 2)): ONE MUFU op (tanh.approx.f32, max relative error 2^-11, below the
// fp16 rounding of the stored result) instead of ex2 + rcp -- a 25 M-element level-0 tensor costs 13 us of MUFU time
// chip-wide with two ops per element, which made the apply pass MUFU-bound rather than HBM-bound.
__device__ __forceinline__ float silu_f(float v) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * v));
    const float h = 0.5f * v;
    return fmaf(h, t, h);
}

// SiLU of 2h given h: with the coefficients (a, b) pre-multiplied by 0.5 (exact in binary floating point) the scaling
// multiply disappears and the result is bit-identical to silu_f(a*x + b)
__device__ __forceinline__ float silu_h(float h) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}

// y = SiLU(a*x + b) (+ r) on 8 channels (16 B); c = (a0, b0, a1, b1) per channel pair (SILU_HALF: (a/2, b/2))
template <bool SILU, bool RES, bool SILU_HALF = false>
__device__ __forceinline__ uint4 gn_apply_vec(const uint4 u, const uint4 rr, const float4 (&c)[4]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float v0 = fmaf(c[j].x, act_lo(w[j]), c[j].y);
        float v1 = fmaf(c[j].z, act_hi(w[j]), c[j].w);
        if (SILU) {
            v0 = SILU_HALF ? silu_h(v0) : silu_f(v0);
            v1 = SILU_HALF ? silu_h(v1) : silu_f(v1);
        }
        if (RES) {
            v0 += act_lo(rw[j]);
            v1 += act_hi(rw[j]);
        }
        // |SiLU(GN(x))| alone cannot reach the fp16 limit; with the residual added it can (trained weights): saturate
        o[j] = RES ? pack_act2(v0, v1) : pack_act2_nosat(v0, v1);
    }
    return make_uint4(o[0], o[1], o[2], o[3]);
}

// (mean, rstd) of one (image, group) from its fixed-point totals: exact integer totals -> double mean / variance
// (a handful of FP64 multiply-adds), rstd in fp32 (MUFU rsqrt + one Newton step, < 1 ulp) like the oracle's fp32 group_norm.
// inv_cnt = 1 / (channels per group * pixels)
__device__ __forceinline__ float2 gn_mean_rstd(const gn_sum_t* a, double inv_cnt, float eps) {
    double s, q;
    gn_sums_read(a, s, q);
    const double m = s * inv_cnt;
    const double var = q * inv_cnt - m * m;
    const float v = fmaxf(static_cast<float>(var), 0.0f) + eps;
    float r = rsqrtf(v);
    r = r * (1.5f - 0.5f * v * r * r);
    return make_float2(static_cast<float>(m), r);
}

// y = A*x + B with the GroupNorm affine and FiLM folded in: ((x - mean) * rstd * gamma + beta) * sc + sh, sc = 1 + s
__device__ __forceinline__ float2 gn_fold(float gamma, float beta, float sc, float sh, float2 mr) {
    const float a = gamma * mr.y;
    const float bb = fmaf(-mr.x, a, beta);
    return make_float2(a * sc, fmaf(bb, sc, sh));
}

}  // namespace cdc
