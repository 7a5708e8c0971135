// K-conv, kh-fused strip variant: 3x3 stride-1 convolution with the three vertical taps of an input row
// stacked along the MMA's N dimension.
//
// Why: tcgen05.mma (M = 128, K = 16, SS operands) costs max(~55, N/2) cycles (tools/exp_mma_n.cu on B200):
// below N = 128 the instruction is bound by the fetch of its 4 KB A tile, so a C_out = 64 layer issued as
// N = 64 MMAs cannot exceed ~56 % of the tensor pipe.  But input row r, shifted by kw, is the A operand of
// THREE taps: (kh = 0 -> output row r+1), (kh = 1 -> r), (kh = 2 -> r-1).  Their weights are stacked to a
// [3 * BN][64] B operand and the three output rows live in adjacent TMEM column blocks, so ONE N = 3*BN MMA
// does the work of three: N = 192 runs at the 96-cycle tensor floor (32 cycles per 64 columns, 100 %).
//
//   work unit : a vertical strip = 128 output columns x L output rows of one image, one N tile of BN channels
//   A operand : ring of input-row chunks in shared memory (TMA box {64 ch, 130 px, 1, 1}, zero fill = conv
//               padding); every (row, 64-channel chunk) is loaded once, consumed by its own 12 MMAs and released
//   B operand : the N tile's whole [kw][chunk][kh reversed][BN][64] weight block, resident in shared memory
//   D         : ring of 512 / BN (at most 16) accumulators (BN TMEM columns each); output row j of the running row counter g
//               lives in slot (g + j) % ring, so the window {r-1, r, r+1} is contiguous except when it wraps
//               (then the MMA is split in two).  BN = 64: six logical rows in eight physical slots, windows never wrap
//               (ALIAS below)
//   first use : every MMA accumulates; the epilogue re-arms an accumulator (tcgen05.st of the bias) right after
//               draining it, so the issue stream has no special first K step
//
//   logical warp 0 : input-row producer (TMA)   1 : barrier init + weight load (TMA, once), then tcgen05.mma issuer
//   logical warp 2 : TMEM allocator             4-11 : epilogue
//   logical warps 12-19 (APPLY only) : GroupNorm + FiLM + SiLU of the INPUT rows, in shared memory, two groups on
//   alternate chunks.  PHYSICALLY the control warps 0-3 are the CTA's LAST four warps (highest issue priority).
//
// Modes: 0 = 3x3 / stride 1 (optionally with the ResBlock's 1x1 residual conv riding along, RES1);
//        1 = nearest-x2 upsample + 3x3 as four parity 2x2 convs;  2 = 3x3 / stride 2 (even / odd pixel tiles).
//
// Epilogue: +bias, GroupNorm sums kept in registers over the whole strip and added once per strip to the
// fixed-point accumulators of gn_sums.cuh (integer atomics: bitwise reproducible), fp16 pack, then either a
// swizzled shared-memory tile + one TMA store per output row (coalesced 16 KB writes) or direct 32-byte stores;
// EPI_DDIM applies the sampler update.
//
// Oracle counterpart: oracle/unet.py `conv(k=3)` inside RB / stem / final (the reference ships no code).
#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

#include "conv_epilogue.cuh"
#include "conv_kf.cuh"
#include "kernels.cuh"
#include "gn_apply.cuh"
#include "ptx.cuh"
#include "sampler.cuh"

namespace cdc {

constexpr int kKfRowBytes = 17 * 1024;  // 130 pixels x 128 B = 16640, padded to a 1024 B multiple
constexpr int kKfRowTx = 130 * 128;
constexpr int kKfAccMax = 16;           // accumulator-ring barriers (the ring holds min(16, 512 / BN) output rows)
constexpr int kKfAux = 1024 + 2 * 8 * 16 * 2 * 4 + 2048 + 256 + 192;  // barriers + TMEM holder + bias, stats scratch, APPLY coefficients, ring barriers
constexpr int kKfMaxSlots = 8;          // input ring: at most 8 slots (4 unless the stride-2 mode has room for more)
// APPLY: eight input-transform warps in TWO groups of four (one warp of each group per SM sub-partition); the groups take
// alternate row chunks, so the load / arithmetic / store phases of consecutive chunks overlap and each group has two row
// periods for its chunk.  640 threads launch with 96 registers each; setmaxnreg then moves registers from warpgroup 0
// (producer / issuer: 48) and the transform warpgroups (64) to the two epilogue warpgroups (152): per sub-partition
// 48 + 2 * 152 + 2 * 64 = 480 registers per lane = the CTA's launch allocation (the pool setmaxnreg draws from).
constexpr int kKfXfGroups = 2;
constexpr int kKfXfExtra = kKfXfGroups * 128;  // threads beyond the 12 warps of the plain kernel
constexpr int kKfXfThreads = 128;              // per group
constexpr int kKfXfPix = kKfXfThreads / 8;     // pixels per pass (8 threads = one pixel's 128 bytes)

template <int BN, int CPG, int EPI, int CH, bool STAGE, bool XK16, int MODE, bool RES1, bool APPLY>
__global__ void __launch_bounds__(128 + kEpiThreads + (APPLY ? kKfXfExtra : 0), 1) conv_kf_kernel(const __grid_constant__ KfParams p) {
    constexpr int kThreads = 128 + kEpiThreads + (APPLY ? kKfXfExtra : 0);
    static_assert(!APPLY || (MODE == 0 && !XK16 && !RES1 && EPI == EPI_STATS && CH <= 2), "input GroupNorm: a 64/128-channel ResBlock's second conv");
    constexpr int WB = BN * 128;  // one (tap, chunk) weight block
    constexpr uint32_t WB16 = WB >> 4;
    // accumulator ring: as many output rows as TMEM holds (a window that wraps costs split MMAs: the longer the ring,
    // the rarer) -- 8 rows of 64 columns, 10 of 48, 16 of 32 or 16
    // RES1: the ResBlock's 1x1 residual conv of the same input rides along -- centre-tap MMAs into a second, short
    // ring of accumulators (its output row is complete one input row earlier than the 3x3's)
    constexpr uint32_t NRES = RES1 ? (BN == 64 ? 2 : 8) : 0;
    constexpr uint32_t NRESD = NRES ? NRES : 1;  // divisor (the fused-residual code is dead when NRES == 0)
    // ALIAS (64-column tiles without the fused residual conv): a ring of SIX logical accumulators in EIGHT physical slots.
    // The window of input row i starts at logical slot s = (first output row) % 6 and always covers the physical slots
    // s, s+1, s+2 <= 7 -- it never wraps, so no window is split into an N = 128 and an N = 64 MMA (119 instead of 96
    // cycles per K step on two rows in eight).  Physical slots 6 and 7 are second homes of logical rows 0 and 1 (what
    // they receive as the 2nd / 3rd row of a window that starts at slot 4 or 5); the epilogue adds the two homes.
    // The BN = 32 convs with the fused residual conv (whose 8 accumulators share TMEM) use the same ring: 6 + 2 + 8 slots
    // (43.0 / 58.2 -> 40.5 / 55.0 us for the two level-1 convs).  The BN = 64 one would be left with a four-row ring and
    // its epilogue, already at the register limit, spills on the second load: 47.6 -> 49.7 us; it keeps 6 + 2 residual slots.
    constexpr bool ALIAS = MODE == 0 && EPI != EPI_DDIM && ((BN == 64 && !RES1) || (BN == 32 && RES1));
    constexpr uint32_t NALIAS = ALIAS ? 2 : 0;
    // With ALIAS the logical slot of an output row is numerics, not just storage: rows in logical slots 0 and 1 receive
    // some taps in their second home, and the two partial sums are added in the epilogue.  So a strip's results depend on
    // (g mod NACC) at its start, i.e. on how many rows its CTA ran before it.  p.slot0 makes every strip start at slot 0:
    // between strips all three roles advance g to the next multiple of NACC through PHANTOM rows -- no MMA, no TMEM access,
    // but every barrier phase of a real row (the issuer waits "drained" and arrives "complete", the epilogue waits
    // "complete" and arrives "drained"; the producer, which waits "drained" only to reuse TMEM, just counts them), so
    // every (g / NACC) & 1 parity stays right.  Elsewhere the slot is storage only: a window that wraps is split along N,
    // and every output element still sums the same products in the same order.
    const bool slot0 = ALIAS && p.slot0 != 0;
    constexpr uint32_t NACC = RES1 ? 6 : ALIAS ? 6 : (512 / BN < kKfAccMax ? 512 / BN : kKfAccMax);
    constexpr int TMEM_COLS = (NACC + NALIAS + NRES) * BN <= 128 ? 128 : (NACC + NALIAS + NRES) * BN <= 256 ? 256 : 512;  // power of two
    static_assert(!RES1 || (MODE == 0 && !STAGE && EPI != EPI_DDIM && (BN == 64 || BN == 32)), "fused residual conv: 3x3 stats/store convs");
    constexpr int STAGE_BYTES = STAGE ? 2 * 128 * BN * 2 : 0;
    static_assert(!STAGE || BN == 64, "staged TMA store is built for 128-byte output rows");
    // MODE 0: 3x3 conv.  MODE 1: nearest-x2 upsample + 3x3 conv as four 2x2 convs on the low-resolution input, one
    // per output parity (py, px) with pre-summed weights (repack_weight_up2_kernel): N tile nt = (channel tile, parity),
    // taps kh in {py, py+1}, kw in {px, px+1} of the 3x3 window, output pixel (2h + py, 2w + px).
    // MODE 2: 3x3 conv with stride 2 (p.H, p.W = OUTPUT grid).  Every (input row, 64-channel chunk) lands as TWO tiles --
    // E = its even pixels 2x and O = its odd pixels 2x+1, through two pixel-stride-2 tensor maps -- so that the three
    // horizontal taps are again plain row offsets: kw=0 -> O[x-1], kw=1 -> E[x], kw=2 -> O[x].  Vertically, input row
    // 2h-1 feeds output rows h (kh=0) and h-1 (kh=2) with ONE N = 2*BN MMA, input row 2h feeds row h (kh=1) alone.
    constexpr int NKH = MODE == 1 ? 2 : 3, NKW = MODE == 1 ? 2 : 3;
    constexpr int NSUB = MODE == 2 ? 2 : 1;  // ring slots per (row, chunk)
    static_assert(MODE != 1 || (!STAGE && EPI == EPI_STORE && !XK16), "UP2 mode: plain scattered store only");
    static_assert(MODE != 2 || (EPI == EPI_STORE && !XK16 && !RES1 && !APPLY), "stride-2 mode: plain conv + store");

    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_u32 = smem_u32(smem_raw);
    const uint32_t base = (raw_u32 + 1023u) & ~1023u;
    uint8_t* gen = smem_raw + (base - raw_u32);
    const int NS = p.NS;
    const uint32_t ring = base;
    const uint32_t wbase = ring + NS * kKfRowBytes;
    const uint32_t wres1 = wbase + NKH * NKW * CH * WB;  // fused 1x1 weights [chunk][BN][64]
    const uint32_t stage = wres1 + (RES1 ? CH * WB : 0);
    const uint32_t aux = stage + STAGE_BYTES;
    uint8_t* aux_gen = gen + (aux - base);
    // barriers: tfull[16] tempty[16] wres xfull[8] xempty[8] (x = fused residual conv) ... row_full[8] row_empty[8]
    const uint32_t bar_rfull = aux + 5376, bar_rempty = aux + 5376 + 64, bar_tfull = aux + 64, bar_tempty = aux + 192, bar_wres = aux + 320;
    const uint32_t bar_xfull = aux + 328, bar_xempty = aux + 392;
    const uint32_t bar_rready = aux + 5376 + 128;  // APPLY: [8] row chunk transformed (one arrive per warp of the owning group)
    const uint32_t bar_afull = APPLY ? bar_rready : bar_rfull;  // what the MMA issuer waits for
    volatile uint32_t* tmem_holder = reinterpret_cast<volatile uint32_t*>(aux_gen + 456);
    float* bias_s = reinterpret_cast<float*>(aux_gen + 512);  // [BN] conv bias, then [BN] residual-conv bias
    float* red_s = reinterpret_cast<float*>(aux_gen + 1024);
    float2* coef_s = reinterpret_cast<float2*>(aux_gen + 3072);      // APPLY: [CH * 64] (a, b) of the current image

    // Roles by LOGICAL warp index: 0..3 control (producer, issuer, TMEM allocator, idle), 4..11 epilogue, 12..19 input
    // transform.  The control warps sit at the END of the CTA: a sub-partition's arbiter prefers its eligible warp with
    // the highest id, and the one-thread MMA issue stream must not queue behind the epilogue / transform warps it shares
    // a sub-partition with (the tensor pipe buffers ~1 MMA: every delayed issue is a bubble).  (w + 4) % 4 == w % 4: the
    // epilogue warps keep their TMEM lane quarter.
    constexpr int kCtrlWarp0 = kThreads / 32 - 4;
    const int pwarp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = pwarp >= kCtrlWarp0 ? pwarp - kCtrlWarp0 : pwarp + 4;
    const int nt = blockIdx.x / p.G1, cta = blockIdx.x % p.G1;
    const int py = MODE == 1 ? (nt & 3) >> 1 : 0, px = MODE == 1 ? nt & 1 : 0;  // output parity (UP2)
    const int cot = MODE == 1 ? nt >> 2 : nt;                                     // output-channel tile
    const int units = p.batch * p.nseg * p.S;
    if (threadIdx.x == 0) stamp_begin(p.stamp);

    if (warp == 0 && lane == 0) {
        prefetch_tensormap(&p.amap[0]);
        prefetch_tensormap(&p.wmap);
        if (STAGE) prefetch_tensormap(&p.omap);
    }
    if (warp == 1) {
        // Barrier initialisation and the weight loads are spread over the lanes of this warp: issued by one thread, the
        // ~60 mbarrier.init and up to 40 TMA instructions sat on the critical path of every launch (the issuer cannot
        // start before the weights are in; a ROLLED single-thread load loop measured -1.5 % images/s against the unrolled one).
        if (lane < kKfMaxSlots) {
            mbar_init(bar_rfull + 8 * lane, 1);
            mbar_init(bar_rempty + 8 * lane, 1);
            if (APPLY) mbar_init(bar_rready + 8 * lane, kKfXfThreads / 32);
        }
        if (lane < static_cast<int>(NACC)) {
            mbar_init(bar_tfull + 8 * lane, 1);
            mbar_init(bar_tempty + 8 * lane, EPI == EPI_DDIM ? 128 : kEpiThreads);
        }
        if (lane < static_cast<int>(NRES)) {
            mbar_init(bar_xfull + 8 * lane, 1);
            mbar_init(bar_xempty + 8 * lane, kEpiThreads);
        }
        if (lane == 0) mbar_init(bar_wres, 1);
        fence_mbar_init();
        __syncwarp();
        // The weight block starts loading right away, before the TMEM allocation and the CTA-wide sync (its barrier
        // was initialised by this warp).
        // smem block order [kw][chunk][2 - kh]: the kh taps of one (kw, chunk) form one contiguous B operand; the loads
        // are numbered in the order the MMAs consume them (chunk, horizontal tap, kh), load l by lane l % 32.
        // (Letting the issuer start on the first (chunk, kw) group while the rest is still landing was tried in round 2 --
        // one barrier per group, first input row issued group by group: the extra issue paths made every launch ~0.9 us
        // SLOWER (-3.5 % images/s), so: one barrier, one wait.)
        constexpr int NLW = NKH * NKW * CH, NL = NLW + (RES1 ? CH : 0);
        if (lane == 0) mbar_expect_tx(bar_wres, NL * WB);
        __syncwarp();
        for (int l = lane; l < NL; l += 32) {
            if (l < NLW) {
                const int e = l % NKH, kw = (l / NKH) % NKW, ch = l / (NKH * NKW);
                if constexpr (MODE == 2) {  // block order per (kw, chunk): kh = 2, 0 (the pair an odd input row feeds), then kh = 1
                    tma_load_2d(wbase + ((kw * CH + ch) * 3 + (e == 2 ? 0 : e == 0 ? 1 : 2)) * WB, &p.wmap, bar_wres,
                                ((e * 3 + kw) * CH + ch) * 64, cot * BN);
                } else if constexpr (MODE == 0) {
                    tma_load_2d(wbase + ((kw * CH + ch) * 3 + (2 - e)) * WB, &p.wmap, bar_wres,
                                ((p.tr ? kw * 3 + e : e * 3 + kw) * CH + ch) * 64, cot * BN);  // transposed walk: taps swap roles
                } else {  // pre-summed parity weights: K index ((parity * 4 + a * 2 + b) * CH + chunk) * 64; kw = b, e = a
                    tma_load_2d(wbase + ((kw * CH + ch) * 2 + (1 - e)) * WB, &p.wmap, bar_wres,
                                (((nt & 3) * 4 + e * 2 + kw) * CH + ch) * 64, cot * BN);
                }
            } else if constexpr (RES1) {
                const int ch = l - NLW;
                tma_load_2d(wres1 + ch * WB, &p.rmap, bar_wres, ch * 64, cot * BN);
            }
        }
        __syncwarp();
    }
    if (warp == 2) {  // (warp-collective)
        tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_holder)), TMEM_COLS);
        tmem_relinquish();
    }
    for (int i = threadIdx.x; i < BN; i += kThreads) {
        bias_s[i] = p.bias[cot * BN + i];
        if (RES1) bias_s[BN + i] = p.res_bias[cot * BN + i];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    auto decode = [&](int u, int& b, int& seg, int& si, int& h0, int& L) {
        si = u % p.S;
        const int t = u / p.S;
        seg = t % p.nseg;
        b = t / p.nseg;
        h0 = si * p.H / p.S;
        L = (si + 1) * p.H / p.S - h0;
    };

    // (role dispatch by warpgroup first: with APPLY each warpgroup re-sizes its register allocation at the top of its branch)
    if (warp < 4) {
    if constexpr (APPLY) setmaxnreg_dec<64>();
    if (warp == 0) {
        // ------------------------------------------------------------ input-row producer
        if (lane == 0) {
            uint32_t slot = 0, par = 0;  // ring position / fill parity (continues across strips)
            uint32_t g = 0;
            for (int u = cta; u < units; u += p.G1) {
                if (slot0) g = (g + NACC - 1) / NACC * NACC;  // phantom rows (see ALIAS): counted, not waited for
                int b, seg, si, h0, L;
                decode(u, b, seg, si, h0, L);
                const int w0 = seg * 128 - 1;
                const int nrows = MODE == 2 ? 2 * L + 1 : L + 2;  // input rows of the strip
                for (int i = 0; i < nrows; ++i) {
                    // input row i opens the accumulator of output row i (stride 2: of row i / 2, i even): drained and re-zeroed?
                    if (MODE == 2 ? ((i & 1) == 0 && (i >> 1) < L) : i < L) {
                        const uint32_t gi = g + (MODE == 2 ? (i >> 1) : i);
                        mbar_wait(bar_tempty + 8 * (gi % NACC), (gi / NACC) & 1);
                    }
                    // (the fused 1x1 conv's short accumulator ring is NOT waited for here: with only 2 slots that would tie
                    // the load of row i to the epilogue's progress three rows back -- measured 5300 instead of 2750 cycles per
                    // row; the issuer checks that ring itself, right before the residual MMAs)
#pragma unroll
                    for (int ch = 0; ch < CH; ++ch) {  // one ring slot per (row, 64-channel chunk) (stride 2: two, E then O)
#pragma unroll
                        for (int sub = 0; sub < NSUB; ++sub) {
                            mbar_wait(bar_rempty + 8 * slot, par ^ 1);
                            const uint32_t full = bar_rfull + 8 * slot;
                            mbar_expect_tx(full, kKfRowTx);
                            const bool s1 = ch >= p.chunks0;
                            const int cc = (s1 ? ch - p.chunks0 : ch) * 64;
                            if constexpr (MODE == 2)  // E tile: even pixels from output column w0+1; O tile: odd pixels from one earlier
                                tma_load_4d(ring + slot * kKfRowBytes, &p.amap[(s1 ? 2 : 0) + sub], full, cc, sub ? w0 : w0 + 1,
                                            2 * h0 - 1 + i, b);
                            else
                                tma_load_4d(ring + slot * kKfRowBytes, s1 ? &p.amap[1] : &p.amap[0], full, cc, w0, h0 - 1 + i, b);
                            if (++slot == static_cast<uint32_t>(NS)) {
                                slot = 0;
                                par ^= 1;
                            }
                        }
                    }
                }
                g += L;
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        // ONE elected thread runs the whole loop.  The tensor pipe queues very little: tools/exp_kf_interf.cu shows that an
        // issue pause of 50 cycles after every 6 MMAs already costs 17 cycles, 100 cost 37, 200 cost 83 (N = 192 MMAs of 96
        // cycles each) -- roughly one MMA is buffered behind the running one.  Round 1's issuer (warp-converged bookkeeping,
        // two elected regions per chunk, row parameters derived at the top of every row) left ~70 instructions between the
        // last MMA of a half chunk and the first of the next: 1305 cycles per 12-MMA row with an idle epilogue and 1570 with
        // a busy one (the issuer shares its SM sub-partition with two epilogue warps) against the 1152-cycle tensor floor.
        // So: everything a chunk needs (accumulator window, weight-block offsets, instruction descriptors, the ring slot's
        // address) is computed one chunk AHEAD, between the MMAs of the previous chunk, and the only instructions between
        // the last MMA of a chunk and the first of the next are the commits, the (already known) barrier answer and the
        // tcgen05 fence.  Every MMA accumulates (the epilogue re-zeroes slots).
        if (elect_one_sync()) {
            constexpr uint32_t idesc0 = make_idesc_f16(128, 0);
            constexpr uint32_t NB = static_cast<uint32_t>(BN >> 3) << 17;  // idesc increment per window slot
            constexpr int T = 4 * NKW;  // K steps per (input row, chunk)
            // (stride 2: the E slot carries kw = 1 (4 K steps), the O slot kw = 0 and kw = 2 (8 K steps))
            constexpr int TT = MODE == 2 ? 8 : T;
            constexpr int TH = 4;       // the next chunk's barrier is probed after this many K steps, its answer used after the last
            const uint64_t desc_hi = make_sw128_desc(0) & 0xFFFFFFFF00000000ull;
            const uint32_t wlo = wbase >> 4;
            uint32_t rslot = 0, rpar = 0;
            uint32_t g = 0;  // running output-row counter: row j of the current strip uses accumulator (g + j) % NACC
            mbar_wait(bar_wres, 0);
            // accumulator window of input row i: it feeds output rows j = i - py - e, e = 0 .. NKH-1 (kh = py + e), clipped to
            // the strip (stride 2: even i -> rows i/2 - 1 (kh = 2) and i/2 (kh = 0); odd i -> row i/2 (kh = 1)); a window
            // that wraps around the accumulator ring is issued as two pieces (A, then B)
            struct RowP {
                uint32_t cnt, nB, dA, dB, bA, bB, iA, iB;
                uint32_t tf;  // accumulator-complete barrier this row's last chunk commits to (0: none)
            };
            auto rowp = [&](int i, int L, uint32_t g_) {
                RowP r;
                const int jtop = MODE == 2 ? (i >> 1) : i - py;
                const int jspan = MODE == 2 ? ((i & 1) ? 0 : 1) : NKH - 1;
                const int jlo = jtop - jspan > 0 ? jtop - jspan : 0;
                const int jhi = jtop < L ? jtop : L - 1;
                r.cnt = jhi >= jlo ? static_cast<uint32_t>(jhi - jlo + 1) : 0u;  // 0: nothing to issue (UP2 edge rows)
                const uint32_t slo = (g_ + jlo) % NACC;
                // weight block of the first window slot (reversed kh; stride 2: blocks are ordered kh = 2, 0, 1)
                const uint32_t khp = MODE == 2 ? ((i & 1) ? 2u : static_cast<uint32_t>(1 - (jtop - jlo)))
                                               : static_cast<uint32_t>((NKH - 1) - (jtop - jlo));
                const uint32_t nA = ALIAS ? r.cnt : (r.cnt < NACC - slo ? r.cnt : NACC - slo);
                r.nB = r.cnt - nA;
                r.dA = tmem_base + slo * BN;
                r.dB = tmem_base;
                r.bA = khp * WB16;
                r.bB = (khp + nA) * WB16;
                r.iA = idesc0 + nA * NB;
                r.iB = idesc0 + r.nB * NB;
                // output row i-2 is complete after input row i (stride 2: row i/2 - 1 after the even-numbered input row i)
                if constexpr (MODE == 2)
                    r.tf = ((i & 1) == 0 && i >= 2) ? bar_tfull + 8 * ((g_ + (i >> 1) - 1) % NACC) : 0u;
                else
                    r.tf = i >= 2 ? bar_tfull + 8 * ((g_ + i - 2) % NACC) : 0u;
                return r;
            };
            // The scheduler sinks plain arithmetic to its first use, i.e. into the gap after a chunk's last MMA.  A (dead)
            // shared-memory store of the values pins their computation where the source has it: between the MMAs.
            const uint32_t pin_word = aux + 460;
            auto pin = [&](uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(pin_word), "r"(v) : "memory"); };
            for (int u = cta; u < units; u += p.G1) {
                // phantom rows up to the next multiple of NACC (see ALIAS).  "Drained" is waited for before "complete" is
                // arrived at, as for a real row, whose MMAs the producer only feeds after that wait: the epilogue has then
                // consumed the slot's previous "complete" phase.  (The first strip starts at g = 0: nothing to do.)
                if (slot0) {
                    for (; g % NACC != 0; ++g) {
                        mbar_wait(bar_tempty + 8 * (g % NACC), (g / NACC) & 1);
                        mbar_arrive(bar_tfull + 8 * (g % NACC));
                        if constexpr (RES1) {  // the fused 1x1 conv's ring is indexed by the same counter: its phases advance too
                            mbar_wait(bar_xempty + 8 * (g % NRESD), (g / NRESD) & 1);
                            mbar_arrive(bar_xfull + 8 * (g % NRESD));
                        }
                    }
                }
                int b, seg, si, h0, L;
                decode(u, b, seg, si, h0, L);
                const int nrows = MODE == 2 ? 2 * L + 1 : L + 2;
                RowP cur = rowp(0, L, g);
                uint32_t sfull = g % NACC;  // first accumulator slot of the next full window (input row 2: output rows 0 .. 2)
                uint32_t alo_base = (ring + rslot * kKfRowBytes) >> 4;
                mbar_wait(bar_afull + 8 * rslot, rpar);  // first chunk of the strip
                tc_fence_after();
                for (int i = 0; i < nrows; ++i) {
                    RowP nxt = cur;
#pragma unroll
                    for (int pc = 0; pc < CH * NSUB; ++pc) {
                        const int ch = pc / NSUB, sub = pc % NSUB;  // sub (stride 2 only): 0 = E tile, 1 = O tile
                        // K steps t = kw * 4 + k in [t0, t1) of one window piece
                        auto steps = [&](auto t0c, auto t1c, uint32_t d, uint32_t bo, uint32_t id) {
                            constexpr int t0 = decltype(t0c)::value, t1 = decltype(t1c)::value;
#pragma unroll
                            for (int t = t0; t < t1; ++t) {
                                const int k = t & 3;
                                // kw: horizontal tap; ashift: its pixel offset inside the slot's tile
                                const int kw = MODE == 2 ? (sub == 0 ? 1 : (t >> 2) * 2) : t >> 2;
                                const int ashift = MODE == 2 ? (sub == 1 && (t >> 2) == 1 ? 1 : 0) : kw + px;
                                if (MODE == 2 && sub == 0 && t >= 4) continue;  // E slot: kw = 1 only
                                if (XK16 && ch == 0 && k != 0) continue;  // stem: chunk 0 = x_t, channels 16..63 are zero
                                const uint32_t alo = alo_base + ashift * 8 + 2 * k;
                                const uint32_t blo = wlo + ((kw * CH + ch) * NKH) * WB16 + 2 * k;
                                umma_f16_ss(d, desc_hi | alo, desc_hi | (blo + bo), id, 1u);
                            }
                        };
                        const uint32_t nslot = rslot + 1 == static_cast<uint32_t>(NS) ? 0u : rslot + 1;
                        const uint32_t npar = nslot == 0 ? rpar ^ 1 : rpar;
                        const bool lastpc = pc == CH * NSUB - 1;
                        const bool more = !lastpc || i + 1 < nrows;  // (a new row's first chunk also certifies its accumulator)
                        if (cur.cnt != 0) steps(std::integral_constant<int, 0>{}, std::integral_constant<int, TH>{}, cur.dA, cur.bA, cur.iA);
                        // probe the next chunk's barrier now, use the answer after the last MMA of this chunk
                        const uint32_t ready = more ? mbar_test_wait(bar_afull + 8 * nslot, npar) : 1u;
                        // ... and derive what the next chunk's MMAs need while this chunk's are in the tensor pipe
                        const uint32_t alo_next = (ring + nslot * kKfRowBytes) >> 4;
                        const uint32_t rempty_bar = bar_rempty + 8 * rslot;
                        if (lastpc) {
                            const int i1 = i + 1;
                            if (MODE == 0 && i1 >= 2 && i1 < L) {
                                // full window (output rows i1-2 .. i1, all inside the strip): no clamps, slot counted up
                                const uint32_t nA = ALIAS ? 3u : (NACC - sfull < 3u ? NACC - sfull : 3u);
                                nxt.cnt = 3u;
                                nxt.nB = 3u - nA;
                                nxt.dA = tmem_base + sfull * BN;
                                nxt.dB = tmem_base;
                                nxt.bA = 0u;
                                nxt.bB = nA * WB16;
                                nxt.iA = idesc0 + nA * NB;
                                nxt.iB = idesc0 + nxt.nB * NB;
                                nxt.tf = bar_tfull + 8 * sfull;
                                sfull = sfull + 1 == NACC ? 0u : sfull + 1;
                            } else {
                                nxt = rowp(i1, L, g);
                            }
                            pin(nxt.cnt ^ nxt.nB ^ nxt.dA ^ nxt.bA ^ nxt.iA ^ nxt.bB ^ nxt.iB ^ nxt.tf ^ alo_next ^ rempty_bar);
                        } else {
                            pin(alo_next ^ rempty_bar);
                        }
                        if (cur.cnt != 0) steps(std::integral_constant<int, TH>{}, std::integral_constant<int, TT>{}, cur.dA, cur.bA, cur.iA);
                        if (cur.nB != 0) steps(std::integral_constant<int, 0>{}, std::integral_constant<int, TT>{}, cur.dB, cur.bB, cur.iB);
                        if (RES1 && i >= 1 && i <= L) {  // fused 1x1 residual conv: centre tap, its own accumulator ring
                            const uint32_t gr = g + i - 1;
                            const uint32_t dR = tmem_base + (NACC + NALIAS + gr % NRESD) * BN;
                            if (ch == 0) {  // slot drained and re-zeroed?  (two rows of MMAs ago: practically never blocks)
                                mbar_wait(bar_xempty + 8 * (gr % NRESD), (gr / NRESD) & 1);
                                tc_fence_after();
                            }
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                umma_f16_ss(dR, desc_hi | (alo_base + 8 + 2 * k), desc_hi | ((wres1 >> 4) + ch * WB16 + 2 * k), idesc0 + NB, 1u);
                            if (ch == CH - 1) umma_commit(bar_xfull + 8 * (gr % NRESD));
                        }
                        umma_commit(rempty_bar);                          // chunk consumed
                        if (lastpc && cur.tf != 0u) umma_commit(cur.tf);  // an output row is complete
                        if (!ready) mbar_wait(bar_afull + 8 * nslot, npar);
                        if (more) tc_fence_after();
                        rslot = nslot;
                        rpar = npar;
                        alo_base = alo_next;
                    }
                    cur = nxt;
                }
                g += L;
            }
        }
        __syncwarp();
    }
    } else if (warp < 12) {
        // ------------------------------------------------------------ epilogue (8 warps)
        if constexpr (APPLY) setmaxnreg_inc<144>();
        const int q = warp & 3;            // TMEM sub-partition: lanes 32q .. 32q+31
        const int half = (warp - 4) >> 2;  // column half of the accumulator
        const int row = q * 32 + lane;
        uint32_t g = 0, tile_ctr = 0, unit_ctr = 0;
        if constexpr (EPI == EPI_DDIM) {
            // 3 real output channels: thread = pixel.  The two warp groups (half 0 / 1) take alternate output rows.
            const float b0 = bias_s[0], b1 = bias_s[1], b2 = bias_s[2];
            const SamplerCoef sc{p.c0, p.c1, p.e0, p.e1, p.sg, p.seed, p.step, p.img_seeds,
                                 static_cast<unsigned int>(p.H * p.W)};
            const uint32_t tq = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
            if (half == 0) {
                // arm every accumulator: zero them all, ONE wait, then the first "drained" arrives
                for (int s_ = 0; s_ < static_cast<int>(NACC); ++s_) tmem_zero<16>(tq + s_ * BN);
                tmem_st_wait();
                tc_fence_before();
                for (int s_ = 0; s_ < static_cast<int>(NACC); ++s_) mbar_arrive(bar_tempty + 8 * s_);
            }
            for (int u = cta; u < units; u += p.G1) {
                int b, seg, si, h0, L;
                decode(u, b, seg, si, h0, L);
                const int gx = seg * 128 + row;
                const bool valid = gx < p.W;
                // x_t of this group's NEXT row is requested before the current row is processed: the accumulators are usually
                // ready when the group gets to them, so a load issued right before the wait would have its latency exposed
                float xt[3] = {0.f, 0.f, 0.f};
                if (valid && half < L) {
                    const size_t pix0 = (static_cast<size_t>(b) * p.H + (h0 + half)) * p.W + gx;
#pragma unroll
                    for (int c = 0; c < 3; ++c) xt[c] = p.x[pix0 * 3 + c];
                }
                for (int j = half; j < L; j += 2) {
                    const uint32_t gj = g + j, slot = gj % NACC;
                    const size_t pix = (static_cast<size_t>(b) * p.H + (h0 + j)) * p.W + gx;
                    float xnext[3] = {0.f, 0.f, 0.f};
                    if (valid && j + 2 < L) {
                        const size_t pix2 = pix + 2 * static_cast<size_t>(p.W);
#pragma unroll
                        for (int c = 0; c < 3; ++c) xnext[c] = p.x[pix2 * 3 + c];
                    }
                    mbar_wait(bar_tfull + 8 * slot, (gj / NACC) & 1);
                    tc_fence_after();
                    uint32_t v[16];
                    tmem_ld16(tq + slot * BN, v);
                    tmem_ld_wait();
                    tmem_zero<16>(tq + slot * BN);
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(bar_tempty + 8 * slot);
                    if (valid) {
                        const float ov[3] = {__uint_as_float(v[0]) + b0, __uint_as_float(v[1]) + b1, __uint_as_float(v[2]) + b2};
                        float x0[3], xn[3];
                        sampler_update3(sc, ov, xt, pix, x0, xn);
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            p.x[pix * 3 + c] = xn[c];
                            if (p.x0_out) p.x0_out[pix * 3 + c] = x0[c];
                        }
                        // the stem's x_t copy (kernels.cuh kXpadC = 16 channels per pixel, 3 real): one whole 32-byte sector
                        static_assert(kXpadC == 16, "one st.global.v8 per pixel");
                        st_global_v8(p.xpad + pix * kXpadC, make_uint4(pack_act2(xn[0], xn[1]), pack_act2(xn[2], 0.0f), 0u, 0u),
                                     make_uint4(0u, 0u, 0u, 0u));
                    }
#pragma unroll
                    for (int c = 0; c < 3; ++c) xt[c] = xnext[c];
                }
                g += L;
            }
        } else {
            constexpr int HC = BN / 2;                             // columns per thread
            constexpr int GH = (EPI == EPI_STATS) ? HC / CPG : 1;  // groups per thread
            static_assert(HC == 32 || HC == 24 || HC == 16, "BN must be 64, 48 or 32");
            // The accumulators are armed with the BIAS, not with zeros: every MMA accumulates on top of it and the drained
            // value needs no add (32 FADDs per thread and row less on an FMA pipe the kernel keeps busy).
            // (not with the fused residual conv: that epilogue is at the register limit, and the 32-register block the
            // tcgen05.st wants made it spill -- 48 -> 54 us for the level-0 128 -> 64 + res conv; there: zeros + an add)
            constexpr bool kBiasAcc = !RES1;
            uint32_t bias_r[HC];
#pragma unroll
            for (int c = 0; c < HC; ++c) bias_r[c] = __float_as_uint(bias_s[half * HC + c]);
            float rbias_r[RES1 ? HC : 1];
            if constexpr (RES1) {
#pragma unroll
                for (int c = 0; c < HC; ++c) rbias_r[c] = bias_s[BN + half * HC + c];
            }
            const bool store_leader = warp == 4 && lane == 0;
            // arm every accumulator, ONE wait, then the first "drained" arrives
            for (int s_ = 0; s_ < static_cast<int>(NACC); ++s_) {
                if constexpr (kBiasAcc)
                    tmem_st_cols<HC>(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + s_ * BN + half * HC, bias_r);
                else
                    tmem_zero<HC>(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + s_ * BN + half * HC);
            }
            if constexpr (RES1 || ALIAS) {  // residual-conv accumulators / second homes: zeros
                for (int s_ = static_cast<int>(NACC); s_ < static_cast<int>(NACC + NALIAS + NRES); ++s_)
                    tmem_zero<HC>(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + s_ * BN + half * HC);
            }
            tmem_st_wait();
            tc_fence_before();
            for (int s_ = 0; s_ < static_cast<int>(NACC + NRES); ++s_)
                mbar_arrive(s_ < static_cast<int>(NACC) ? bar_tempty + 8 * s_ : bar_xempty + 8 * (s_ - NACC));  // (barrier indices, not slots)
            for (int u = cta; u < units; u += p.G1, ++unit_ctr) {
                if (slot0) {  // phantom rows (see ALIAS and the issuer): the slot keeps its armed bias, its second home its zeros
                    for (; g % NACC != 0; ++g) {
                        if constexpr (RES1) {
                            mbar_wait(bar_xfull + 8 * (g % NRES), (g / NRES) & 1);
                            mbar_arrive(bar_xempty + 8 * (g % NRES));
                        }
                        mbar_wait(bar_tfull + 8 * (g % NACC), (g / NACC) & 1);
                        mbar_arrive(bar_tempty + 8 * (g % NACC));
                    }
                }
                int b, seg, si, h0, L;
                decode(u, b, seg, si, h0, L);
                const int gx = seg * 128 + row;
                const bool valid = gx < p.W;
                float gs[GH], gq[GH];
#pragma unroll
                for (int i = 0; i < GH; ++i) gs[i] = gq[i] = 0.0f;
                uint32_t amax2 = 0u;  // packed running max |output| of this thread over the strip (saturation diagnostics)
                for (int j = 0; j < L; ++j, ++tile_ctr) {
                    const uint32_t gj = g + j, slot = gj % NACC;
                    if constexpr (RES1) {  // the fused 1x1 conv's row j (complete one input row before the 3x3's)
                        const uint32_t xs = gj % NRES;
                        mbar_wait(bar_xfull + 8 * xs, (gj / NRES) & 1);
                        tc_fence_after();
                        const uint32_t xaddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (NACC + NALIAS + xs) * BN + half * HC;
                        uint32_t xv[HC];
                        tmem_ld_cols<HC>(xaddr, xv);
                        tmem_ld_wait();
                        tmem_zero<HC>(xaddr);
                        tmem_st_wait();
                        tc_fence_before();
                        mbar_arrive(bar_xempty + 8 * xs);
                        if (valid) {
                            uint4 xo[HC / 8];
#pragma unroll
                            for (int s4 = 0; s4 < HC / 8; ++s4) {
                                xo[s4].x = pack_act2(__uint_as_float(xv[s4 * 8 + 0]) + rbias_r[s4 * 8 + 0], __uint_as_float(xv[s4 * 8 + 1]) + rbias_r[s4 * 8 + 1]);
                                xo[s4].y = pack_act2(__uint_as_float(xv[s4 * 8 + 2]) + rbias_r[s4 * 8 + 2], __uint_as_float(xv[s4 * 8 + 3]) + rbias_r[s4 * 8 + 3]);
                                xo[s4].z = pack_act2(__uint_as_float(xv[s4 * 8 + 4]) + rbias_r[s4 * 8 + 4], __uint_as_float(xv[s4 * 8 + 5]) + rbias_r[s4 * 8 + 5]);
                                xo[s4].w = pack_act2(__uint_as_float(xv[s4 * 8 + 6]) + rbias_r[s4 * 8 + 6], __uint_as_float(xv[s4 * 8 + 7]) + rbias_r[s4 * 8 + 7]);
                                amax2 = act2_absmax(amax2, xo[s4]);
                            }
                            const size_t rpix = p.tr ? (static_cast<size_t>(b) * p.W + gx) * p.H + (h0 + j)
                                                     : (static_cast<size_t>(b) * p.H + (h0 + j)) * p.W + gx;
                            uint4* rdst = reinterpret_cast<uint4*>(p.res_out + rpix * p.res_ldc + cot * BN + half * HC);
#pragma unroll
                            for (int s8 = 0; s8 < HC / 16; ++s8) st_global_v8(rdst + 2 * s8, xo[2 * s8], xo[2 * s8 + 1]);
                        }
                    }
                    mbar_wait(bar_tfull + 8 * slot, (gj / NACC) & 1);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + slot * BN + half * HC;
                    uint32_t v[HC];
                    tmem_ld_cols<HC>(taddr, v);
                    tmem_ld_wait();
                    if constexpr (kBiasAcc)
                        tmem_st_cols<HC>(taddr, bias_r);  // re-arm the slot (with the bias): every MMA accumulates
                    else
                        tmem_zero<HC>(taddr);
                    if (ALIAS && slot < NALIAS) {  // logical rows 0 and 1: add what landed in the second home
                        const uint32_t t2 = taddr + NACC * BN;
                        uint32_t v2[HC];
                        tmem_ld_cols<HC>(t2, v2);
                        tmem_ld_wait();
                        tmem_zero<HC>(t2);
#pragma unroll
                        for (int c = 0; c < HC; ++c) v[c] = __float_as_uint(__uint_as_float(v[c]) + __uint_as_float(v2[c]));
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    mbar_arrive(bar_tempty + 8 * slot);
                    float f[HC];
#pragma unroll
                    for (int c = 0; c < HC; ++c) f[c] = kBiasAcc ? __uint_as_float(v[c]) : __uint_as_float(v[c]) + __uint_as_float(bias_r[c]);
                    if constexpr (EPI == EPI_STATS) {
                        if (valid) {  // (pixels past the image edge hold bias + 0: not part of the statistics)
                            // (packed fp32 pairs -- FADD2 / FFMA2 with (even, odd) lane accumulators -- measured no
                            // faster and doubled the accumulator registers: scalar)
#pragma unroll
                            for (int c = 0; c < HC; ++c) {
                                gs[c / CPG] += f[c];
                                gq[c / CPG] = fmaf(f[c], f[c], gq[c / CPG]);
                            }
                        }
                    }
                    uint4 o[HC / 8];
#pragma unroll
                    for (int s4 = 0; s4 < HC / 8; ++s4) {
                        o[s4].x = pack_act2(f[s4 * 8 + 0], f[s4 * 8 + 1]);
                        o[s4].y = pack_act2(f[s4 * 8 + 2], f[s4 * 8 + 3]);
                        o[s4].z = pack_act2(f[s4 * 8 + 4], f[s4 * 8 + 5]);
                        o[s4].w = pack_act2(f[s4 * 8 + 6], f[s4 * 8 + 7]);
                        if constexpr (EPI != EPI_STATS) amax2 = act2_absmax(amax2, o[s4]);  // (EPI_STATS: see below)
                    }
                    if constexpr (STAGE) {
                        // 128 pixel rows x 128 B, 128-byte swizzle: 16-byte chunk c of row r sits at chunk c ^ (r & 7)
                        const uint32_t sb = stage + (tile_ctr & 1) * (128 * BN * 2) + row * 128;
#pragma unroll
                        for (int s4 = 0; s4 < HC / 8; ++s4) {
                            const uint32_t c = half * (HC / 8) + s4;
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sb + ((c ^ (row & 7)) << 4)), "r"(o[s4].x),
                                         "r"(o[s4].y), "r"(o[s4].z), "r"(o[s4].w)
                                         : "memory");
                        }
                        fence_proxy_async_smem();
                        if (store_leader) bulk_wait_group_read<0>();  // the previous row's store has left its buffer
                        named_bar_sync(1, kEpiThreads);
                        if (store_leader) {
                            tma_store_4d(&p.omap, stage + (tile_ctr & 1) * (128 * BN * 2), cot * BN, seg * 128, h0 + j, b);
                            bulk_commit_group();
                        }
                    } else if (valid) {
                        const size_t pix = MODE == 1 ? (static_cast<size_t>(b) * 2 * p.H + 2 * (h0 + j) + py) * (2 * p.W) + 2 * gx + px
                                           : p.tr ? (static_cast<size_t>(b) * p.W + gx) * p.H + (h0 + j)
                                                  : (static_cast<size_t>(b) * p.H + (h0 + j)) * p.W + gx;
                        uint4* dst = reinterpret_cast<uint4*>(p.out + pix * p.ldc + cot * BN + half * HC);
                        // thread = pixel: its channels are contiguous, lanes are a pixel pitch apart.  32-byte stores fill
                        // whole sectors and halve the store instructions (each costs ~1 cycle per distinct line)
                        if constexpr (HC % 16 == 0) {
#pragma unroll
                            for (int s8 = 0; s8 < HC / 16; ++s8) st_global_v8(dst + 2 * s8, o[2 * s8], o[2 * s8 + 1]);
                        } else {
#pragma unroll
                            for (int s4 = 0; s4 < HC / 8; ++s4) dst[s4] = o[s4];
                        }
                    }
                }
                g += L;
                // Saturation diagnostics.  Without statistics: exact, from the packed outputs.  With GroupNorm statistics the
                // per-row tracking (32 more instructions per row: -0.7 % images/s) is replaced by a test on the sums of
                // squares this thread already holds: one saturated value makes its group's partial >= 65504^2.  That test
                // is conservative the safe way -- it also fires when a pixel column's squares add up to 65504^2 over the
                // strip (rms beyond ~5000: within one order of magnitude of the fp16 limit, worth reporting all the same).
                bool sat = act2_is_sat(amax2);
                if constexpr (EPI == EPI_STATS) {
                    float qm = gq[0];
#pragma unroll
                    for (int i = 1; i < GH; ++i) qm = fmaxf(qm, gq[i]);
                    sat = sat || qm >= kActMax * kActMax;
                }
                if (valid && sat && p.sat) atomicAdd(p.sat, 1u);
                if constexpr (EPI == EPI_STATS) {
                    // one (sum, sum of squares) per (strip, group): warp butterfly -> 4 lane quarters through smem -> integer atomics
                    const float ws = warp_group_reduce<GH>(gs, lane);
                    const float wq = warp_group_reduce<GH>(gq, lane);
                    constexpr int REP = 32 / GH;
                    float* red = red_s + (unit_ctr & 1) * (8 * 16 * 2);
                    if ((lane & (REP - 1)) == 0) {
                        const int gl = lane / REP;
                        red[((half * 4 + q) * 16 + gl) * 2 + 0] = ws;
                        red[((half * 4 + q) * 16 + gl) * 2 + 1] = wq;
                    }
                    named_bar_sync(2, kEpiThreads);
                    const int t = (half * 4 + q) * 32 + lane;
                    if (t < 2 * GH) {
                        const int hh = t / GH, gl = t % GH;
                        const float* r0 = red + ((hh * 4) * 16 + gl) * 2;
                        const float s = ((r0[0] + r0[32]) + r0[64]) + r0[96];
                        const float s2 = ((r0[1] + r0[33]) + r0[65]) + r0[97];
                        gn_sums_add(p.gn_acc + static_cast<size_t>(b) * kGnImgStride, cot * (BN / CPG) + t, s, s2);
                    }
                }
            }
            if (STAGE && store_leader) bulk_wait_group<0>();

        }
    } else if constexpr (APPLY) {
        // ------------------------------------------------------------ input transform (warps 12 .. 19, two groups)
        // y = SiLU(a*x + b) on every landed row chunk, in place, before the MMAs read it: the arithmetic of
        // gn_apply_kernel (gn_apply.cuh), bit for bit.  Thread = (16-byte channel vector c, pixel lane pl): its 8 channels'
        // (a, b) pairs stay in registers.  Pixels and rows outside the image are left as TMA zero-filled them: the conv
        // pads with zeros AFTER the activation.  Group g takes the chunks n = g, g + 2, ... of this CTA's sequence (ring
        // slot n % NS: with an even ring a slot always belongs to the same group).
        setmaxnreg_dec<64>();
        const int grp = (warp - 12) >> 2;
        const int xt = ((warp - 12) & 3) * 32 + lane;
        const int c = xt & 7, pl = xt >> 3;
        const uint32_t toff = static_cast<uint32_t>(pl) * 128u + (static_cast<uint32_t>(c ^ (pl & 7)) << 4);  // 128-byte swizzle
        constexpr int NIT = (130 + kKfXfPix - 1) / kKfXfPix;  // 9 passes of 16 pixels, done as 3 x 3 (64-register budget)
        static_assert(kKfXfPix % 8 == 0 && NIT == 9, "a pixel's swizzle phase must not depend on the pass");
        constexpr int cpg_in = CH * 2;  // channels per group of the input (C_in / 32)
        const double inv_n = 1.0 / (static_cast<double>(cpg_in) * p.H * p.W);
        float2* coef_g = coef_s + grp * (CH * 64);  // each group keeps its own table: no cross-group barrier
        uint32_t n = 0;  // chunk counter of the CTA (all chunks; this group handles n % 2 == grp)
        int cur_b = -1;
        float4 cf[4];
        for (int u = cta; u < units; u += p.G1) {
            int b, seg, si, h0, L;
            decode(u, b, seg, si, h0, L);
            if (b != cur_b) {  // coefficient table of image b (once per CTA when the batch is 1)
                named_bar_sync(3 + grp, kKfXfThreads);
                if (xt < CH * 64) {  // (every thread derives its channel's group statistics itself: a few FP64 operations)
                    const float2 mr = gn_mean_rstd(p.in_acc + (static_cast<size_t>(b) * 32 + xt / cpg_in) * kGnVals, inv_n, p.in_eps);
                    const float sc = p.in_film ? 1.0f + p.in_film[xt] : 1.0f, sh = p.in_film ? p.in_film[CH * 64 + xt] : 0.0f;
                    const float2 ab = gn_fold(p.in_gamma[xt], p.in_beta[xt], sc, sh, mr);
                    coef_g[xt] = make_float2(0.5f * ab.x, 0.5f * ab.y);  // (a/2, b/2): see silu_h
                }
                named_bar_sync(3 + grp, kKfXfThreads);
                cur_b = b;
                // with two chunks per row the groups' alternation pins group g to chunk g: one coefficient set either way
#pragma unroll
                for (int j = 0; j < 4; ++j) cf[j] = reinterpret_cast<const float4*>(coef_g + (CH == 2 ? grp * 64 : 0) + c * 8)[j];
            }
            const int w0 = seg * 128 - 1;
            for (int ic = 0; ic < (L + 2) * CH; ++ic, ++n) {
                const int i = ic / CH;
                if ((n & 1u) != static_cast<uint32_t>(grp)) continue;
                const uint32_t slot = n % static_cast<uint32_t>(NS), par = (n / static_cast<uint32_t>(NS)) & 1u;
                const int h = h0 - 1 + i;
                const bool row_in = h >= 0 && h < p.H;
                mbar_wait(bar_rfull + 8 * slot, par);
                if (row_in) {
                    const uint32_t sb = ring + slot * kKfRowBytes + toff;
                    // per half: all loads, all arithmetic, all stores, with distinct registers per vector -- a store that
                    // has to leave the (busy) shared-memory queue before its registers are reused costs ~150 cycles
                    auto part = [&](auto k0c, auto k1c) {
                        constexpr int K0 = decltype(k0c)::value, K1 = decltype(k1c)::value;
                        uint4 v[K1 - K0];
                        bool ok[K1 - K0];
#pragma unroll
                        for (int k = K0; k < K1; ++k) {
                            const int pxl = pl + kKfXfPix * k, gx = w0 + pxl;
                            ok[k - K0] = pxl < 130 && gx >= 0 && gx < p.W;
                            v[k - K0] = make_uint4(0u, 0u, 0u, 0u);
                            if (ok[k - K0])
                                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                                             : "=r"(v[k - K0].x), "=r"(v[k - K0].y), "=r"(v[k - K0].z), "=r"(v[k - K0].w)
                                             : "r"(sb + k * (kKfXfPix * 128)));
                        }
#pragma unroll
                        for (int k = 0; k < K1 - K0; ++k) v[k] = gn_apply_vec<true, false, true>(v[k], v[k], cf);
#pragma unroll
                        for (int k = K0; k < K1; ++k) {
                            if (ok[k - K0])
                                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sb + k * (kKfXfPix * 128)), "r"(v[k - K0].x),
                                             "r"(v[k - K0].y), "r"(v[k - K0].z), "r"(v[k - K0].w)
                                             : "memory");
                        }
                    };
                    part(std::integral_constant<int, 0>{}, std::integral_constant<int, 3>{});
                    part(std::integral_constant<int, 3>{}, std::integral_constant<int, 6>{});
                    part(std::integral_constant<int, 6>{}, std::integral_constant<int, 9>{});
                }
                fence_proxy_async_smem();  // generic-proxy writes -> visible to the MMA's async-proxy reads
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_rready + 8 * slot);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) stamp_end(p.stamp);
    if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------ host
// (BN, CPG, EPI, CH, STAGED, XK16, MODE, RES1) instantiations: the layer shapes of the UNet / context net this variant serves.
#define KF_ALL_CASES()                                            \
    KF_CASE(64, 2, EPI_STATS, 1, true, false, 0, false, false)    \
    KF_CASE(64, 2, EPI_STATS, 2, false, false, 0, false, false)   \
    KF_CASE(64, 4, EPI_STATS, 1, true, false, 0, false, false)    \
    KF_CASE(64, 4, EPI_STATS, 2, false, false, 0, false, false)   \
    KF_CASE(64, 1, EPI_STORE, 1, true, false, 0, false, false)    \
    KF_CASE(64, 1, EPI_STORE, 2, false, false, 0, false, false)   \
    KF_CASE(64, 1, EPI_STORE, 2, false, true, 0, false, false)    \
    KF_CASE(32, 4, EPI_STATS, 3, false, false, 0, false, false)   \
    KF_CASE(32, 4, EPI_STATS, 4, false, false, 0, false, false)   \
    KF_CASE(48, 6, EPI_STATS, 3, false, false, 0, false, false)   \
    KF_CASE(32, 8, EPI_STATS, 4, false, false, 0, false, false)   \
    KF_CASE(16, 1, EPI_DDIM, 1, false, false, 0, false, false)    \
    KF_CASE(64, 1, EPI_STORE, 2, false, false, 1, false, false)   \
    KF_CASE(64, 1, EPI_STORE, 3, false, false, 1, false, false)   \
    KF_CASE(64, 1, EPI_STORE, 4, false, false, 1, false, false)   \
    KF_CASE(64, 2, EPI_STATS, 2, false, false, 0, true, false)    \
    KF_CASE(32, 4, EPI_STATS, 3, false, false, 0, true, false)    \
    KF_CASE(32, 4, EPI_STATS, 4, false, false, 0, true, false)    \
    KF_CASE(64, 2, EPI_STATS, 1, true, false, 0, false, true)     \
    KF_CASE(64, 4, EPI_STATS, 2, false, false, 0, false, true)    \
    KF_CASE(64, 1, EPI_STORE, 1, true, false, 2, false, false)      \
    KF_CASE(64, 1, EPI_STORE, 2, false, false, 2, false, false)


int kf_smem_bytes(int bn, int CH, int NS, bool staged, int mode, bool res) {
    return 1024 + NS * kKfRowBytes + ((mode == 1 ? 4 : 9) + (res ? 1 : 0)) * CH * bn * 128 + (staged ? 2 * 128 * bn * 2 : 0) + kKfAux;
}

bool kf_plan(int bn, int CH, int mode, bool res, int* NS, bool* staged) {
    const int limit = 227 * 1024;
    for (int st = (mode == 1 || res) ? 0 : 1; st >= 0; --st) {  // NS = ring slots of one (row, chunk) each
        if (st && bn != 64) continue;
        // (a single staging buffer + a 3-slot ring for the two-chunk store-only stem was tried: 35 -> 43 us)
        // (stride 2: two slots per (row, chunk); one-chunk convs: a deeper ring where shared memory allows -- the input
        // transform adds a pipeline stage)
        for (int ns = mode == 2 ? kKfMaxSlots : CH == 1 ? 6 : 4; ns >= (mode == 2 ? 4 : 3); --ns)
            if (kf_smem_bytes(bn, CH, ns, st != 0, mode, res) <= limit) {
                *NS = ns;
                *staged = st != 0;
                return true;
            }
    }
    return false;
}

bool kf_inst_ok(int bn, int cpg, int epi, int CH, int mode, bool res, bool apply) {
    int ns;
    bool st;
    if (!kf_plan(bn, CH, mode, res, &ns, &st)) return false;
    // APPLY: transform group g owns the chunks n = g (mod 2) and waits on ring slot n % NS by parity -- sound only when
    // a slot always belongs to the same group, i.e. for an EVEN ring (ADVICE r1)
    if (apply && (ns & 1)) return false;
#define KF_CASE(BN_, CPG_, EPI_, CH_, ST_, X_, M_, R_, A_) \
    if (bn == BN_ && (EPI_ != EPI_STATS || cpg == CPG_) && epi == EPI_ && CH == CH_ && st == ST_ && mode == M_ && res == R_ && apply == A_) return true;
    KF_ALL_CASES()
#undef KF_CASE
    return false;
}

cudaError_t configure_kf_kernels() {
    cudaError_t e;
#define KF_CASE(BN_, CPG_, EPI_, CH_, ST_, X_, M_, R_, A_)                                                  \
    if ((e = cudaFuncSetAttribute(conv_kf_kernel<BN_, CPG_, EPI_, CH_, ST_, X_, M_, R_, A_>,                  \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) \
        return e;
    KF_ALL_CASES()
#undef KF_CASE
    return cudaSuccess;
}

cudaError_t launch_conv_kf(const KfParams& p, int bn, int cpg, int epi, int CH, bool xk16, int mode, bool res, bool apply,
                           bool st, cudaStream_t stream) {
    if (p.NS < 3 || p.NS > kKfMaxSlots || (apply && (p.NS & 1))) return cudaErrorInvalidValue;
    const dim3 grid(p.n_tiles * p.G1), block(128 + kEpiThreads + (apply ? kKfXfExtra : 0));
    const size_t smem = kf_smem_bytes(bn, CH, p.NS, st, mode, res);
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
#define KF_CASE(BN_, CPG_, EPI_, CH_, ST_, X_, M_, R_, A_)                                                                                \
    if (bn == BN_ && (EPI_ != EPI_STATS || cpg == CPG_) && epi == EPI_ && CH == CH_ && st == ST_ && xk16 == X_ && mode == M_ && res == R_ && \
        apply == A_) {                                                                                                                       \
        conv_kf_kernel<BN_, CPG_, EPI_, CH_, ST_, X_, M_, R_, A_><<<grid, block, smem, stream>>>(p);                                         \
        return cudaGetLastError();                                                                                                           \
    }
    KF_ALL_CASES()
#undef KF_CASE
    return cudaErrorInvalidValue;
}

}  // namespace cdc
