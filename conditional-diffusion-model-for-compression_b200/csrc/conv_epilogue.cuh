// Shared epilogue of the tcgen05 conv kernels: one 128-pixel x BN accumulator tile
// TMEM -> registers -> (+bias, GroupNorm sums, residual, DDIM update) -> global.
// Called by the 4 epilogue warps (128 threads); thread = TMEM lane = output pixel.
#pragma once
#include "kernels.cuh"
#include "conv_tc.cuh"
#include "gn_sums.cuh"
#include "ptx.cuh"
#include "sampler.cuh"

namespace cdc {

struct EpiArgs {
    act_t* out;
    const act_t* residual;
    int ldc;
    // EPI_DDIM
    float* x;
    act_t* xpad;
    float* x0_out;
    SamplerCoef sc;
    unsigned int* sat;  // saturation diagnostics counter (may be null)
    float act_slope;    // 0 = none; s in (0, 1): LeakyReLU(s) applied after the bias
};

template <int G>
__device__ __forceinline__ float warp_group_reduce(float (&s)[G], int lane) {
    // Butterfly reduce-scatter over the warp: on return lane L holds the warp total of group
    // L >> (5 - log2 G).  Fixed shuffle order => bitwise reproducible.
    constexpr int LOG2G = (G == 32) ? 5 : (G == 16) ? 4 : (G == 8) ? 3 : (G == 4) ? 2 : (G == 2) ? 1 : 0;
    static_assert((1 << LOG2G) == G, "G must be a power of two <= 32");
#pragma unroll
    for (int step = 0; step < LOG2G; ++step) {
        const int m = 16 >> step;
        const int half = G >> (step + 1);
        const bool up = (lane & m) != 0;
#pragma unroll
        for (int i = 0; i < G / 2; ++i) {
            if (i < half) {
                const float send = up ? s[i] : s[i + half];
                const float keep = up ? s[i + half] : s[i];
                s[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
            }
        }
    }
    float r = s[0];
#pragma unroll
    for (int m = (16 >> LOG2G); m >= 1; m >>= 1) r += __shfl_xor_sync(0xffffffffu, r, m);
    return r;
}

// Eight epilogue warps share one tile: warp (q, half) owns TMEM lanes 32q..32q+31 (rows) and the
// column range [half*BN/2, (half+1)*BN/2).  Two warps per SM sub-partition instead of one roughly
// halves the latency-bound epilogue time (a lone warp ran at IPC ~0.3 in the round-1 profile).
//
// taddr: TMEM address of lane quarter q of the accumulator; bar_tempty: mbarrier (256 arrivals, 128 for
// EPI_DDIM) that hands the accumulator back to the MMA warp; bs: bias of this N tile (shared memory);
// red: 2*4*16*2 floats of shared scratch (alternate between consecutive tiles);
// gn_dst: accumulator slot of this image, offset to the first group of this N tile (gn_sums.cuh), or unused.
constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;

template <int BN, int CPG, int EPI>
__device__ __forceinline__ void conv_epilogue_tile(const EpiArgs& e, uint32_t taddr, uint32_t bar_tempty,
                                                   const float* bs, float* red, int q, int half, int lane, bool valid,
                                                   size_t pix, int n0, gn_sum_t* gn_dst, bool arrive = true) {
    if constexpr (EPI == EPI_DDIM) {
        if (half != 0) return;
        uint32_t v[16];
        tmem_ld16(taddr, v);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(bar_tempty);
        if (valid) {
            const float ov[3] = {__uint_as_float(v[0]) + bs[0], __uint_as_float(v[1]) + bs[1], __uint_as_float(v[2]) + bs[2]};
            const float xt[3] = {e.x[pix * 3 + 0], e.x[pix * 3 + 1], e.x[pix * 3 + 2]};
            float x0[3], xn[3];
            sampler_update3(e.sc, ov, xt, pix, x0, xn);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                e.x[pix * 3 + c] = xn[c];
                e.xpad[pix * kXpadC + c] = to_act(xn[c]);
                if (e.x0_out) e.x0_out[pix * 3 + c] = x0[c];
            }
        }
    } else {
        constexpr int HC = BN / 2;                                 // columns per warp
        constexpr int NCH = HC / 32;                               // 32-column chunks per warp
        constexpr int GH = (EPI == EPI_STATS) ? HC / CPG : 1;      // groups per warp
        static_assert(HC % 32 == 0, "BN must be a multiple of 64");
        float gs[GH], gq[GH];
#pragma unroll
        for (int g = 0; g < GH; ++g) gs[g] = gq[g] = 0.0f;
        const int c0 = half * HC;
        act_t* orow = e.out + pix * e.ldc + n0 + c0;
        const act_t* rrow = e.residual ? e.residual + pix * e.ldc + n0 + c0 : nullptr;
        const float msk = valid ? 1.0f : 0.0f;
        uint32_t amax2 = 0u;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            uint32_t v[32];
            tmem_ld32(taddr + c0 + ch * 32, v);
            tmem_ld_wait();
            if (ch == NCH - 1 && arrive) {  // this warp's share of the accumulator (group) is drained
                tc_fence_before();
                mbar_arrive(bar_tempty);
            }
            float f[32];
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                const float4 b4 = *reinterpret_cast<const float4*>(bs + c0 + ch * 32 + j4 * 4);
                f[j4 * 4 + 0] = __uint_as_float(v[j4 * 4 + 0]) + b4.x;
                f[j4 * 4 + 1] = __uint_as_float(v[j4 * 4 + 1]) + b4.y;
                f[j4 * 4 + 2] = __uint_as_float(v[j4 * 4 + 2]) + b4.z;
                f[j4 * 4 + 3] = __uint_as_float(v[j4 * 4 + 3]) + b4.w;
            }
            if (e.act_slope != 0.0f) {  // LeakyReLU: max(x, s*x) for 0 < s < 1
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], e.act_slope * f[j]);
            }
            if constexpr (EPI == EPI_STATS) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int g = (ch * 32 + j) / CPG;
                    const float x = f[j] * msk;
                    gs[g] += x;
                    gq[g] = fmaf(x, x, gq[g]);
                }
            }
            if (valid) {
                uint4* dst = reinterpret_cast<uint4*>(orow + ch * 32);
#pragma unroll
                for (int s4 = 0; s4 < 4; ++s4) {
                    if (rrow) {
                        const uint4 r = *reinterpret_cast<const uint4*>(rrow + ch * 32 + s4 * 8);
                        f[s4 * 8 + 0] += act_lo(r.x);
                        f[s4 * 8 + 1] += act_hi(r.x);
                        f[s4 * 8 + 2] += act_lo(r.y);
                        f[s4 * 8 + 3] += act_hi(r.y);
                        f[s4 * 8 + 4] += act_lo(r.z);
                        f[s4 * 8 + 5] += act_hi(r.z);
                        f[s4 * 8 + 6] += act_lo(r.w);
                        f[s4 * 8 + 7] += act_hi(r.w);
                    }
                    uint4 o;
                    o.x = pack_act2(f[s4 * 8 + 0], f[s4 * 8 + 1]);
                    o.y = pack_act2(f[s4 * 8 + 2], f[s4 * 8 + 3]);
                    o.z = pack_act2(f[s4 * 8 + 4], f[s4 * 8 + 5]);
                    o.w = pack_act2(f[s4 * 8 + 6], f[s4 * 8 + 7]);
                    if constexpr (EPI != EPI_STATS) amax2 = act2_absmax(amax2, o);  // (EPI_STATS: from the sums of squares below)
                    dst[s4] = o;
                }
            }
        }
        {   // saturation diagnostics: exact from the packed outputs, or (EPI_STATS) conservative from the sums of squares
            // this thread already holds -- see conv_kf.cu
            bool sat = act2_is_sat(amax2);
            if constexpr (EPI == EPI_STATS) {
                float qm = gq[0];
#pragma unroll
                for (int g = 1; g < GH; ++g) qm = fmaxf(qm, gq[g]);
                sat = sat || qm >= kActMax * kActMax;
            }
            if (valid && sat && e.sat) atomicAdd(e.sat, 1u);
        }
        if constexpr (EPI == EPI_STATS) {
            // warp butterfly -> 8 warps through smem -> one (sum, sum of squares) per (tile, group) -> integer atomics
            const float ws = warp_group_reduce<GH>(gs, lane);
            const float wq = warp_group_reduce<GH>(gq, lane);
            constexpr int REP = 32 / GH;
            if ((lane & (REP - 1)) == 0) {
                const int g = lane / REP;
                red[((half * 4 + q) * 16 + g) * 2 + 0] = ws;
                red[((half * 4 + q) * 16 + g) * 2 + 1] = wq;
            }
            named_bar_sync(1, kEpiThreads);
            const int t = (half * 4 + q) * 32 + lane;
            if (t < 2 * GH) {
                const int hh = t / GH, gl = t % GH;
                const float* r0 = red + ((hh * 4) * 16 + gl) * 2;
                const float s = ((r0[0] + r0[32]) + r0[64]) + r0[96];
                const float s2 = ((r0[1] + r0[33]) + r0[65]) + r0[97];
                gn_sums_add(gn_dst, t, s, s2);
            }
        }
    }
}

}  // namespace cdc
