// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05
// (alloc / mma / commit / ld / fences).  Hand-written; nothing here links CUTLASS.
#pragma once
#include "act.cuh"
#include <stdint.h>
#include <stdio.h>

namespace cdc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// try_wait with a suspend-time hint: the hardware parks the thread until the phase completes (or the
// hint expires) instead of letting it spin.  Spinning waiters share the SM sub-partition's issue slots
// with the single-thread MMA issue stream; the round-1 timeline showed 115 instead of 64 cycles per
// tcgen05.mma with default (short) try_wait polling.
__device__ __forceinline__ bool mbar_try_wait_suspend(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(hint_ns)
        : "memory");
    return ok != 0;
}
// Non-blocking probe.  Issued EARLY and consumed late, its ~140-cycle latency overlaps whatever is issued in between
// (the kf conv issuer puts half a chunk's MMAs there).
__device__ __forceinline__ uint32_t mbar_test_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
// Bounded wait: a protocol bug must trap (sticky launch failure), never hang the GPU box.  The tools build also says
// which barrier (printf's argument buffer, inlined at every wait site, costs the 48..64-register producer / issuer warps
// of the APPLY kernels spills, so the product build only traps).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 8000000000LL) {  // ~4 s at 2 GHz
#ifdef CDC_TOOLS
            printf("cdc: mbarrier timeout block %d thread %d bar 0x%x parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
#endif
            __trap();
        }
    }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const void* desc) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(desc)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// 256-bit global store (sm_100: STG.256): one full 32-byte sector per lane.  p must be 32-byte aligned.
__device__ __forceinline__ void st_global_v8(void* p, const uint4& a, const uint4& b) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x),
                 "r"(b.y), "r"(b.z), "r"(b.w)
                 : "memory");
}
// TMA store of one 4-D box shared -> global (bulk async-group completion).  Pixels of the box that fall
// outside the tensor are clipped by the hardware.
__device__ __forceinline__ void tma_store_4d(const void* desc, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(desc)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the source shared memory of all but the N most recent bulk groups has been read
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_f16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// mbarrier arrive when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// Predicated forms.  The producer / issuer warps run warp-converged (all 32 lanes execute the loop,
// addresses and descriptors are warp-uniform) and only the asynchronous instruction itself is
// predicated on the leader lane.
__device__ __forceinline__ void umma_f16_ss_p(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void umma_commit_p(uint32_t bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(bar), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_p(uint32_t bar, uint32_t bytes, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
        ::"r"(bar), "r"(bytes), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_p(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1,
                                              uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %5, 0;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d_p(uint32_t dst, const void* desc, uint32_t bar, int c0, int c1, int c2,
                                              int c3, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %7, 0;\n\t"
        "@q cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(leader)
        : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (rows of 128 B, 8-row atoms 1024 B apart).
// bits [0,14) start>>4, [16,30) LBO>>4 (unused for swizzled K-major), [32,46) SBO>>4,
// [46,48) version = 1 (sm_100), [49,52) base offset, [61,64) layout type (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr, uint32_t base_offset = 0) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(base_offset & 7) << 49;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// kind::f16 instruction descriptor: fp32 accumulate, act_t (fp16 or bf16) A/B, both K-major, M x N tile.
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | (kUmmaFormat << 7) | (kUmmaFormat << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread = lane = row).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
// this warp's 32 lanes x NCOL consecutive fp32 columns (NCOL = 32, 24 or 16); follow with tmem_ld_wait()
template <int NCOL>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t (&v)[NCOL]) {
    static_assert(NCOL == 32 || NCOL == 24 || NCOL == 16, "32, 24 or 16 columns");
    if constexpr (NCOL == 32) {
        tmem_ld32(taddr, v);
    } else {
        uint32_t(&lo)[16] = reinterpret_cast<uint32_t(&)[16]>(v);
        tmem_ld16(taddr, lo);
        if constexpr (NCOL == 24) tmem_ld8(taddr + 16, &v[16]);
    }
}
// registers -> TMEM: zero this warp's 32 lanes x NCOL consecutive columns (re-arms an accumulator so that every
// MMA into it can run with accumulate = 1)
template <int NCOL>
__device__ __forceinline__ void tmem_zero(uint32_t taddr) {
    static_assert(NCOL == 16 || NCOL == 24 || NCOL == 32, "16, 24 or 32 columns");
    const uint32_t z = 0;
    if constexpr (NCOL == 24) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr + 16), "r"(z) : "memory");
    }
    if constexpr (NCOL == 32) {
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
            "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
            "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z)
            : "memory");
    } else {  // 16, and the first 16 of 24
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
            "{%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z)
            : "memory");
    }
}
// registers -> TMEM: this warp's 32 lanes x NCOL consecutive columns from v (re-arms an accumulator with the conv bias)
template <int NCOL>
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&v)[NCOL]) {
    static_assert(NCOL == 16 || NCOL == 24 || NCOL == 32, "16, 24 or 32 columns");
    if constexpr (NCOL == 32) {
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
            "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
            "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
            "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
            "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]),
            "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
            : "memory");
    } else {
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
            "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
            "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]),
            "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
            : "memory");
        if constexpr (NCOL == 24) {
            asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr + 16), "r"(v[16]), "r"(v[17]),
                         "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23])
                         : "memory");
        }
    }
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t elect_one_sync() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Warpgroup register reallocation (all 4 warps of a warpgroup, converged): dec releases registers to the CTA's pool,
// inc blocks until the pool holds enough.  Counts are multiples of 8 in [24, 256].  The pool is what the CTA was
// launched with (threads x launch registers), not the SM's unallocated remainder.
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
// In-graph timing stamps (diagnostics): slot[0] = earliest CTA start, slot[1] = latest CTA end of a launch, in
// globaltimer nanoseconds; the host initialises the slot to (~0, 0).  One thread per CTA calls each, so the cost is two
// atomics per CTA -- and nothing when the pointer is null (the product's decode graph).
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void stamp_begin(long long* slot) {
    if (slot) atomicMin(reinterpret_cast<unsigned long long*>(slot), globaltimer_ns());
}
__device__ __forceinline__ void stamp_end(long long* slot) {
    if (slot) atomicMax(reinterpret_cast<unsigned long long*>(slot) + 1, globaltimer_ns());
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace cdc
