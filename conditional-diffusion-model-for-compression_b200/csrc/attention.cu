// K-attn: fused flash-style softmax(Q K^T / 8) V for the 1/16-resolution mid block
// (4 heads x d = 64, N = HW/256 tokens).  Scores never touch HBM.
#include "kernels.cuh"
#include "ptx.cuh"

namespace cdc {

constexpr int kAttD = 64;

// =====================================================================================================================
// S = Q K^T and O_tile = P V run on the 5th-generation tensor cores (tcgen05) with TMEM accumulators.
//
//   CTA = 128 queries of one head; K/V tiles of 128 keys stream through a 2-deep TMA ring.
//   warp 0 : TMA producer (Q once, then K and V tiles; rows past N are zero-filled by the 3-D tensor map)
//   warp 1 : TMEM allocator + MMA issuer: S_b = Q K_b^T (M 128 x N 128 x K 64, both operands K-major), issued one tile
//            AHEAD of  O_b = P_b V_b  (M 128 x N 64 x K 128; A = P from shared memory, B = V as an MN-major operand:
//            the [key][d] tile exactly as TMA lands it, instruction-descriptor bit 16)
//   warps 2-5, 6-9 : two softmax warpgroups, thread = query row = TMEM lane; group g owns the tiles j = g (mod 2),
//            i.e. TMEM / P buffer g, and keeps its OWN online-softmax state (m, l, o) -- the two streams are merged
//            through shared memory at the end, so while one group does exp2 the tensor core serves the other.
//            Two passes over the S row in TMEM (row max, then exp2 / sum / fp16 P -> 128-byte-swizzled shared
//            memory) keep only 32 score registers live; the running output stays in REGISTERS
//            (o = o * scale + O_tile, O_tile read back with tcgen05.ld): no TMEM read-modify-write correction pass.
// Oracle counterpart: oracle/unet.py Attn.forward (softmax(q k^T / 8) v per head).
// =====================================================================================================================
constexpr int kTcThreads = 320;  // TMA warp, MMA warp, two softmax warpgroups
constexpr int kTcTile = 128 * 128;                               // bytes of one [128 rows][64 x 16-bit] tile
constexpr int kTcSmemBytes = 1024 + kTcTile * (1 + 2 + 2 + 4) + 256;  // Q, K[2], V[2], P[2][2 key blocks], barriers

__device__ __forceinline__ float ex2_approx(float x) {  // one MUFU op; ex2(-inf) = 0
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}

__global__ void __launch_bounds__(kTcThreads, 1) attention_tc_kernel(const __grid_constant__ AttnTcParams p) {
    extern __shared__ uint8_t att_raw[];
    const uint32_t raw = smem_u32(att_raw), base = (raw + 1023u) & ~1023u;
    uint8_t* gen = att_raw + (base - raw);
    const uint32_t sQ = base, sK = sQ + kTcTile, sV = sK + 2 * kTcTile, sP = sV + 2 * kTcTile, bars = sP + 4 * kTcTile;
    // barriers: q_full | k_full[2] k_empty[2] v_full[2] v_empty[2] | s_full[2] s_empty[2] p_full[2] o_full[2] o_empty[2]
    const uint32_t b_qf = bars, b_kf = bars + 8, b_ke = bars + 24, b_vf = bars + 40, b_ve = bars + 56;
    const uint32_t b_sf = bars + 72, b_se = bars + 88, b_pf = bars + 104, b_of = bars + 120, b_oe = bars + 136;
    volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(gen + 9 * kTcTile + 160);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int N = p.N, C = p.heads * kAttD;
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * 128;
    const int T = (N + 127) / 128;

    if (threadIdx.x == 0) {
        stamp_begin(p.stamp);
        prefetch_tensormap(&p.qkv_map);
        mbar_init(b_qf, 1);
    }
    if (warp == 0 && lane < 2) {  // (buffer i's barriers by lane i)
        const int i = lane;
        mbar_init(b_kf + 8 * i, 1);
        mbar_init(b_ke + 8 * i, 1);
        mbar_init(b_vf + 8 * i, 1);
        mbar_init(b_ve + 8 * i, 1);
        mbar_init(b_sf + 8 * i, 1);
        mbar_init(b_se + 8 * i, 128);
        mbar_init(b_pf + 8 * i, 128);
        mbar_init(b_of + 8 * i, 1);
        mbar_init(b_oe + 8 * i, 128);
    }
    if (warp == 0) {
        fence_mbar_init();
        __syncwarp();
    }
    if (warp == 1) {
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_holder)), 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_holder;

    if (warp == 0) {
        if (lane == 0) {
            mbar_expect_tx(b_qf, kTcTile);
            tma_load_3d(sQ, &p.qkv_map, b_qf, h * kAttD, q0, b);
            for (int j = 0; j < T; ++j) {
                const uint32_t buf = j & 1, ph = (j >> 1) & 1;
                mbar_wait(b_ke + 8 * buf, ph ^ 1);
                mbar_expect_tx(b_kf + 8 * buf, kTcTile);
                tma_load_3d(sK + buf * kTcTile, &p.qkv_map, b_kf + 8 * buf, C + h * kAttD, j * 128, b);
                mbar_wait(b_ve + 8 * buf, ph ^ 1);
                mbar_expect_tx(b_vf + 8 * buf, kTcTile);
                tma_load_3d(sV + buf * kTcTile, &p.qkv_map, b_vf + 8 * buf, 2 * C + h * kAttD, j * 128, b);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        constexpr uint32_t idesc_s = make_idesc_f16(128, 128);
        constexpr uint32_t idesc_o = make_idesc_f16(128, 64) | (1u << 16);  // B (= V) is MN-major
        const uint64_t desc_hi = make_sw128_desc(0) & 0xFFFFFFFF00000000ull;
        auto issue_s = [&](int t) {  // S_buf = Q K_t^T
            const uint32_t buf = t & 1, ph = (t >> 1) & 1;
            mbar_wait(b_kf + 8 * buf, ph);
            mbar_wait(b_se + 8 * buf, ph ^ 1);
            tc_fence_after();
            if (elect_one_sync()) {
                const uint32_t alo = sQ >> 4, blo = (sK + buf * kTcTile) >> 4;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    umma_f16_ss(tmem + buf * 128, desc_hi | (alo + 2 * k), desc_hi | (blo + 2 * k), idesc_s, k != 0 ? 1u : 0u);
                umma_commit(b_sf + 8 * buf);
                umma_commit(b_ke + 8 * buf);
            }
            __syncwarp();
        };
        mbar_wait(b_qf, 0);
        issue_s(0);
        for (int j = 0; j < T; ++j) {
            const uint32_t buf = j & 1, ph = (j >> 1) & 1;
            if (j + 1 < T) issue_s(j + 1);
            mbar_wait(b_pf + 8 * buf, ph);
            mbar_wait(b_vf + 8 * buf, ph);
            mbar_wait(b_oe + 8 * buf, ph ^ 1);
            tc_fence_after();
            if (elect_one_sync()) {  // O_buf = P_buf V_buf: two 64-key blocks of P x four 16-key steps
#pragma unroll
                for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t alo = ((sP + (buf * 2 + kb) * kTcTile) >> 4) + 2 * k;
                        const uint32_t blo = (sV + buf * kTcTile + (kb * 64 + k * 16) * 128) >> 4;  // 16 key rows further down
                        umma_f16_ss(tmem + 256 + buf * 64, desc_hi | alo, desc_hi | blo, idesc_o, (kb | k) != 0 ? 1u : 0u);
                    }
                umma_commit(b_of + 8 * buf);
                umma_commit(b_ve + 8 * buf);
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3, row = q * 32 + lane, grp = (warp - 2) >> 2;
        const uint32_t tq = tmem + (static_cast<uint32_t>(q * 32) << 16);
        const float sl2 = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
        float m = -INFINITY, l = 0.f;
        float o[64];
#pragma unroll
        for (int i = 0; i < 64; ++i) o[i] = 0.f;
        for (int j = grp; j < T; j += 2) {  // this group's tiles all use buffer `grp`
            const uint32_t buf = grp, ph = (j >> 1) & 1;
            mbar_wait(b_sf + 8 * buf, ph);
            tc_fence_after();
            const int key0 = j * 128;
            const int nkeys = N - key0 < 128 ? N - key0 : 128;  // valid keys of this tile (only the last tile is ragged)
            float mx = -INFINITY;
#pragma unroll
            for (int c = 0; c < 4; ++c) {  // pass 1: row maximum
                uint32_t v[32];
                tmem_ld32(tq + buf * 128 + c * 32, v);
                tmem_ld_wait();
                if (nkeys == 128) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(v[i]));
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (c * 32 + i < nkeys) mx = fmaxf(mx, __uint_as_float(v[i]));
                }
            }
            const float m_new = fmaxf(m, mx * sl2);  // every tile holds at least one valid key: finite
            const float sc = ex2_approx(m - m_new);
            float rs = 0.f;
            const uint32_t prow = sP + buf * 2 * kTcTile + row * 128;
#pragma unroll
            for (int c = 0; c < 4; ++c) {  // pass 2: p = exp2(s - m), row sum, fp16 P into the swizzled A-operand tile
                uint32_t v[32];
                tmem_ld32(tq + buf * 128 + c * 32, v);
                tmem_ld_wait();
                if (c == 3) {  // S_buf fully read: the issuer may overwrite it with tile j + 2
                    tc_fence_before();
                    mbar_arrive(b_se + 8 * buf);
                }
                float pv[32];
                if (nkeys == 128) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        pv[i] = ex2_approx(fmaf(__uint_as_float(v[i]), sl2, -m_new));
                        rs += pv[i];
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        pv[i] = c * 32 + i < nkeys ? ex2_approx(fmaf(__uint_as_float(v[i]), sl2, -m_new)) : 0.f;
                        rs += pv[i];
                    }
                }
#pragma unroll
                for (int s4 = 0; s4 < 4; ++s4) {
                    const int key = c * 32 + s4 * 8, kb = key >> 6, ck = (key & 63) >> 3;
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(prow + kb * kTcTile + ((ck ^ (row & 7)) << 4)),
                                 "r"(pack_act2(pv[s4 * 8 + 0], pv[s4 * 8 + 1])), "r"(pack_act2(pv[s4 * 8 + 2], pv[s4 * 8 + 3])),
                                 "r"(pack_act2(pv[s4 * 8 + 4], pv[s4 * 8 + 5])), "r"(pack_act2(pv[s4 * 8 + 6], pv[s4 * 8 + 7]))
                                 : "memory");
                }
            }
            fence_proxy_async_smem();
            mbar_arrive(b_pf + 8 * buf);
            l = fmaf(l, sc, rs);
            m = m_new;
            // o = o * scale + P_j V_j (the other group's softmax overlaps this wait)
            mbar_wait(b_of + 8 * buf, ph);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t v[32];
                tmem_ld32(tq + 256 + buf * 64 + c * 32, v);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) o[c * 32 + i] = fmaf(o[c * 32 + i], sc, __uint_as_float(v[i]));
            }
            tc_fence_before();
            mbar_arrive(b_oe + 8 * buf);
        }
        // merge the two groups' streams: group 1 -> shared memory (the K/V/P tiles are dead by now) -> group 0
        named_bar_sync(1, 256);
        float* scr = reinterpret_cast<float*>(gen + kTcTile) + row * 66;  // 128 rows x 66 floats = 33 KB over the K / V tiles
        if (grp == 1) {
#pragma unroll
            for (int i = 0; i < 64; ++i) scr[i] = o[i];
            scr[64] = m;
            scr[65] = l;
        }
        named_bar_sync(1, 256);
        if (grp == 0 && q0 + row < N) {
            const float mb = scr[64], lb = scr[65];
            const float mn = fmaxf(m, mb);  // group 0 always has a tile: finite
            const float sa = ex2_approx(m - mn), sb = ex2_approx(mb - mn);
            const float inv = 1.0f / (l * sa + lb * sb);
            const float wa = sa * inv, wb = sb * inv;
            uint4* dst = reinterpret_cast<uint4*>(p.out + (static_cast<size_t>(b) * N + q0 + row) * C + h * kAttD);
#pragma unroll
            for (int s8 = 0; s8 < 4; ++s8) {
                uint32_t w[8];
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    w[e] = pack_act2(o[s8 * 16 + 2 * e] * wa + scr[s8 * 16 + 2 * e] * wb, o[s8 * 16 + 2 * e + 1] * wa + scr[s8 * 16 + 2 * e + 1] * wb);
                st_global_v8(dst + 2 * s8, make_uint4(w[0], w[1], w[2], w[3]), make_uint4(w[4], w[5], w[6], w[7]));
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) stamp_end(p.stamp);
    if (warp == 1) tmem_dealloc(tmem, 512);
}

cudaError_t configure_attention_tc() {
    return cudaFuncSetAttribute(attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes);
}

cudaError_t launch_attention_tc(const AttnTcParams& p, int B, cudaStream_t s) {
    static const cudaError_t cfg = configure_attention_tc();
    if (cfg != cudaSuccess) return cfg;
    dim3 grid((p.N + 127) / 128, p.heads, B);
    attention_tc_kernel<<<grid, kTcThreads, kTcSmemBytes, s>>>(p);
    return cudaGetLastError();
}

}  // namespace cdc
