// K-conv: persistent, warp-specialised tcgen05 implicit-GEMM convolution for sm_100a.
//
//   M tile  = 128 output pixels forming a BH x BW rectangle of one image
//   N tile  = BN output channels (UMMA 128 x BN x 16, cta_group::1, fp32 accumulators in TMEM)
//   K block = 64 input channels of one filter tap: ONE 4-D TMA box {64 ch, BW, BH, 1} of the NHWC
//             activation tensor at the tap-shifted origin.  Out-of-image pixels are zero-filled by
//             TMA, which is exactly the conv zero padding, and the box lands in shared memory as
//             128 rows x 128 B with the 128-byte swizzle, i.e. already the K-major UMMA operand.
//
//   warp 0 : TMA producer (one elected lane)        smem ring: full[] / empty[] mbarriers
//   warp 1 : tcgen05.mma issuer (one elected lane)  TMEM ring: tfull[] / tempty[] (2 accumulators)
//   warp 2 : TMEM allocator
//   warps 4-11 : epilogue (tcgen05.ld -> +bias -> GroupNorm sums / residual / DDIM -> global)
//
// Oracle counterpart: oracle/unet.py `conv`, `Up`, `RB` (the reference ships no code).
#include <stdio.h>

#include "conv_epilogue.cuh"
#include "conv_tc.cuh"
#include "ptx.cuh"

namespace cdc {

template <int BN>
struct ConvCfg {
    static constexpr int A_BYTES = 128 * 128;
    static constexpr int B_BYTES = BN * 128;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int NS = (BN >= 256) ? 4 : (BN >= 192) ? 5 : (BN >= 128) ? 6 : 8;
    static constexpr int ACC_STRIDE = BN < 32 ? 32 : BN;
    static constexpr int TMEM_COLS = (2 * ACC_STRIDE <= 32)    ? 32
                                     : (2 * ACC_STRIDE <= 64)  ? 64
                                     : (2 * ACC_STRIDE <= 128) ? 128
                                     : (2 * ACC_STRIDE <= 256) ? 256
                                                               : 512;
    // aux region after the stage ring: barriers (8 B each), TMEM base, bias copy, stats scratch
    static constexpr int BAR_BYTES = 256;
    static constexpr int BIAS_BYTES = 768 * 4;
    static constexpr int RED_BYTES = 2 * 4 * 32 * 2 * 4;
    static constexpr int SMEM_BYTES = 1024 + NS * STAGE_BYTES + BAR_BYTES + BIAS_BYTES + RED_BYTES;
};

constexpr int kConvThreads = 128 + kEpiThreads;  // 4 control warps + 8 epilogue warps

template <int BN, int CPG, int EPI>
__global__ void __launch_bounds__(kConvThreads, 1) conv_tc_kernel(const __grid_constant__ ConvParams p) {
    using Cfg = ConvCfg<BN>;
    constexpr int NS = Cfg::NS;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_u32 = smem_u32(smem_raw);
    const uint32_t base = (raw_u32 + 1023u) & ~1023u;  // 128B-swizzle atoms need 1024 B alignment
    uint8_t* gen = smem_raw + (base - raw_u32);
    const uint32_t aux = base + NS * Cfg::STAGE_BYTES;
    uint8_t* aux_gen = gen + NS * Cfg::STAGE_BYTES;
    const uint32_t bar_full = aux, bar_empty = aux + 8 * NS, bar_tfull = aux + 16 * NS, bar_tempty = aux + 16 * NS + 16;
    volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(aux_gen + 16 * NS + 32);
    float* bias_s = reinterpret_cast<float*>(aux_gen + Cfg::BAR_BYTES);
    float* red_s = reinterpret_cast<float*>(aux_gen + Cfg::BAR_BYTES + Cfg::BIAS_BYTES);

    // logical roles: 0..3 control, 4..11 epilogue; the control warps are the LAST physical warps (the sub-partition
    // arbiter prefers high warp ids and the MMA issue stream must not queue behind the epilogue: see conv_kf.cu)
    const int pwarp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = pwarp >= 8 ? pwarp - 8 : pwarp + 4;
    const int BWl = p.bw_log2, BW = 1 << BWl, BH = 128 >> BWl;
    const int total_tiles = p.n_tiles * p.nphase * p.batch * p.tiles_h * p.tiles_w;
    if (threadIdx.x == 0) stamp_begin(p.stamp);

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&p.wmap);
        prefetch_tensormap(&p.amap[0]);
    }
    if (warp == 1) {  // (one barrier set per lane: the serial init loop sat on every launch's critical path)
        if (lane < NS) {
            mbar_init(bar_full + 8 * lane, 1);
            mbar_init(bar_empty + 8 * lane, 1);
        }
        if (lane < 2) {
            mbar_init(bar_tfull + 8 * lane, 1);
            mbar_init(bar_tempty + 8 * lane, EPI == EPI_DDIM ? 128 : kEpiThreads);
        }
        fence_mbar_init();
        __syncwarp();
    }
    if (warp == 2) {
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_holder)), Cfg::TMEM_COLS);
        tmem_relinquish();
    }
    for (int i = threadIdx.x; i < p.n_total; i += kConvThreads) bias_s[i] = p.bias[i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    auto decode = [&](int tile, int& nt, int& ph, int& b, int& th, int& tw) {
        nt = tile % p.n_tiles;
        int m = tile / p.n_tiles;
        tw = m % p.tiles_w;
        m /= p.tiles_w;
        th = m % p.tiles_h;
        m /= p.tiles_h;
        ph = m % p.nphase;
        b = m / p.nphase;
    };

    // Producer and issuer run warp-converged; only the async instruction is predicated on lane 0.
    const uint32_t leader = lane == 0 ? 1u : 0u;
    if (warp == 0) {
        // ---------------------------------------------------------------- TMA producer
        uint32_t stage = 0, phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            int nt, ph, b, th, tw;
            decode(tile, nt, ph, b, th, tw);
            const KBlock* tab = p.kb + ph * p.nkb;
            const int w0 = tw * BW, h0 = th * BH;
            for (int i = 0; i < p.nkb; ++i) {
                const KBlock e = tab[i];
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                const uint32_t sa = base + stage * Cfg::STAGE_BYTES;
                const uint32_t full = bar_full + 8 * stage;
                mbar_expect_tx_p(full, Cfg::STAGE_BYTES, leader);
                tma_load_4d_p(sa, &p.amap[e.map], full, e.c0, w0 + e.dw, h0 + e.dh, b, leader);
                tma_load_2d_p(sa + Cfg::A_BYTES, &p.wmap, full, e.wk, nt * BN, leader);
                if (++stage == NS) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    } else if (warp == 1) {
        // ---------------------------------------------------------------- MMA issuer
        // One elected thread.  The tensor pipe buffers about one MMA behind the running one (tools/exp_kf_interf.cu), so
        // the blocking barrier wait + fence + descriptor arithmetic that round 1 had in front of every K block's four MMAs
        // was a bubble per K block: the next stage's barrier is now probed right after the block's first MMA and its answer
        // used after the last one (also across tiles: the next tile's first K block does not depend on its accumulator).
        if (elect_one_sync()) {
            constexpr uint32_t idesc = make_idesc_f16(128, BN);
            const uint64_t desc_hi = make_sw128_desc(0) & 0xFFFFFFFF00000000ull;
            uint32_t stage = 0, phase = 0, it = 0;
            if (static_cast<int>(blockIdx.x) < total_tiles) {
                mbar_wait(bar_full + 8 * stage, phase);  // the CTA's first K block
                tc_fence_after();
            }
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
                const uint32_t as = it & 1, aphase = (it >> 1) & 1;
                mbar_wait(bar_tempty + 8 * as, aphase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + as * Cfg::ACC_STRIDE;
                const bool more_tiles = tile + static_cast<int>(gridDim.x) < total_tiles;
                for (int i = 0; i < p.nkb; ++i) {
                    const uint32_t sa = base + stage * Cfg::STAGE_BYTES;
                    const uint32_t alo = (sa >> 4) & 0x3FFFu, blo = ((sa + Cfg::A_BYTES) >> 4) & 0x3FFFu;
                    const uint32_t nstage = stage + 1 == NS ? 0u : stage + 1, nphase = nstage == 0 ? phase ^ 1 : phase;
                    const bool more = i + 1 < p.nkb || more_tiles;
                    umma_f16_ss(d_tmem, desc_hi | alo, desc_hi | blo, idesc, i != 0 ? 1u : 0u);
                    const uint32_t ready = more ? mbar_test_wait(bar_full + 8 * nstage, nphase) : 1u;
#pragma unroll
                    for (int k = 1; k < 4; ++k)  // 4 x (K = 16): +32 B inside the 128 B swizzle row
                        umma_f16_ss(d_tmem, desc_hi | (alo + 2 * k), desc_hi | (blo + 2 * k), idesc, 1u);
                    umma_commit(bar_empty + 8 * stage);  // frees the smem slot once these MMAs retire
                    if (i + 1 == p.nkb) umma_commit(bar_tfull + 8 * as);  // accumulator complete -> epilogue
                    if (!ready) mbar_wait(bar_full + 8 * nstage, nphase);
                    if (more) tc_fence_after();
                    stage = nstage;
                    phase = nphase;
                }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ---------------------------------------------------------------- epilogue (8 warps)
        const int q = warp & 3;            // TMEM sub-partition: lanes 32q .. 32q+31
        const int half = (warp - 4) >> 2;  // column half of the accumulator
        const int row = q * 32 + lane;
        const int ty = row >> BWl, tx = row & (BW - 1);
        const EpiArgs ea{p.out, p.residual, p.ldc, p.x, p.xpad, p.x0_out,
                         SamplerCoef{p.c0, p.c1, p.e0, p.e1, p.sg, p.seed, p.step, p.img_seeds, static_cast<unsigned int>(p.OH * p.OW)},
                         p.sat, p.act_slope};
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            int nt, ph, b, th, tw;
            decode(tile, nt, ph, b, th, tw);
            const uint32_t as = it & 1, aphase = (it >> 1) & 1;
            const int gy = th * BH + ty, gx = tw * BW + tx;
            const bool valid = (gy < p.gh) && (gx < p.gw);
            const int oy = gy * p.os + (ph >> 1), ox = gx * p.os + (ph & 1);
            const size_t pix = (static_cast<size_t>(b) * p.OH + oy) * p.OW + ox;

            mbar_wait(bar_tfull + 8 * as, aphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * Cfg::ACC_STRIDE;
            gn_sum_t* sdst = (EPI == EPI_STATS) ? p.gn_acc + (static_cast<size_t>(b) * 32 + nt * (BN / CPG)) * kGnVals : nullptr;
            conv_epilogue_tile<BN, CPG, EPI>(ea, taddr, bar_tempty + 8 * as, bias_s + nt * BN,
                                             red_s + (it & 1) * (2 * 4 * 16 * 2), q, half, lane, valid, pix, nt * BN, sdst);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) stamp_end(p.stamp);
    if (warp == 2) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

template <int BN, int CPG, int EPI>
static cudaError_t configure_one() {
    return cudaFuncSetAttribute(conv_tc_kernel<BN, CPG, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                ConvCfg<BN>::SMEM_BYTES);
}

template <int BN, int CPG, int EPI>
static cudaError_t launch_one(const ConvParams& p, int num_sms, cudaStream_t stream) {
    using Cfg = ConvCfg<BN>;
    auto kern = conv_tc_kernel<BN, CPG, EPI>;
    const int total = p.n_tiles * p.nphase * p.batch * p.tiles_h * p.tiles_w;
    const int grid = total < num_sms ? total : num_sms;
    kern<<<grid, kConvThreads, Cfg::SMEM_BYTES, stream>>>(p);
    return cudaGetLastError();
}

#define CDC_ALL_CASES()          \
    CDC_CASE(64, 1, EPI_STORE)   \
    CDC_CASE(128, 1, EPI_STORE)  \
    CDC_CASE(192, 1, EPI_STORE)  \
    CDC_CASE(256, 1, EPI_STORE)  \
    CDC_CASE(64, 2, EPI_STATS)   \
    CDC_CASE(64, 4, EPI_STATS)   \
    CDC_CASE(64, 8, EPI_STATS)   \
    CDC_CASE(128, 4, EPI_STATS)  \
    CDC_CASE(128, 8, EPI_STATS)  \
    CDC_CASE(192, 6, EPI_STATS)  \
    CDC_CASE(256, 8, EPI_STATS)  \
    CDC_CASE(16, 1, EPI_DDIM)

cudaError_t configure_conv_kernels() {
    cudaError_t e;
#define CDC_CASE(BN_, CPG_, EPI_) \
    if ((e = configure_one<BN_, CPG_, EPI_>()) != cudaSuccess) return e;
    CDC_ALL_CASES()
#undef CDC_CASE
    return cudaSuccess;
}

cudaError_t launch_conv(const ConvParams& p, int bn, int cpg, int epi, int num_sms, cudaStream_t stream) {
    if (epi != EPI_STATS) cpg = 1;
#define CDC_CASE(BN_, CPG_, EPI_) \
    if (bn == BN_ && cpg == CPG_ && epi == EPI_) return launch_one<BN_, CPG_, EPI_>(p, num_sms, stream);
    CDC_ALL_CASES()
#undef CDC_CASE
    return cudaErrorInvalidValue;
}


}  // namespace cdc
