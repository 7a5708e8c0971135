// rANS bitstream of the quantised latents (SURVEY.md section 8 row f3): byte-exact with oracle/rans.py, which pins
// the format (32-bit state, 16-bit precision, 16-bit words; every channel row cut into `spc` interleaved streams so that
// the lanes of a warp read consecutive symbols; escapes carry raw + 1 as a 5-bit length and uniform bits; container
// "CDCR" | version | n_chan | hw | spc | 0 | u32 size[streams] | streams).
//
// Integer / byte work, inherently serial inside a stream: one thread per stream, n_chan * spc streams per call (8192 for
// a 2048 x 2048 image's y), coalesced symbol reads (stream j of a row reads symbols j, j + spc, ...), 2-byte word
// writes into a per-stream scratch region (filled backwards, so the stream comes out in decode order), then a
// device-side exclusive scan of the stream sizes and a packing pass into the container.  No tensor cores, no shared-memory
// staging worth having: the bound is the dependent-instruction chain per symbol (a 32-bit divide), not bandwidth.
// Oracle counterpart: oracle/rans.py encode / decode (the reference ships no code).
#include "kernels.cuh"

namespace cdc {

constexpr uint32_t kRansL = 1u << 16;
constexpr int kRansHeader = 24;  // magic, version, n_chan, hw, spc, reserved

__host__ __device__ inline long long rans_stream_stride(long long hw, int spc) {  // bytes of scratch per stream
    const long long kmax = (hw + spc - 1) / spc;
    return ((4 + 2 * 4 * kmax) + 7) & ~7LL;  // final state + at most one word per (sub-)symbol, four per element
}

__device__ __forceinline__ void rans_put(uint32_t& x, uint16_t*& wp, uint32_t start, uint32_t freq) {
    if (static_cast<unsigned long long>(x) >= (static_cast<unsigned long long>(freq) << 16)) {
        *--wp = static_cast<uint16_t>(x & 0xFFFFu);
        x >>= 16;
    }
    x = ((x / freq) << 16) + (x % freq) + start;
}

// one thread per stream
__global__ void __launch_bounds__(128) rans_encode_kernel(const int32_t* __restrict__ idx, const int32_t* __restrict__ v,
                                                          const int32_t* __restrict__ lo, const int32_t* __restrict__ hi,
                                                          const int32_t* __restrict__ raw, const int32_t* __restrict__ cdf_length,
                                                          long long n_chan, long long hw, int spc, uint8_t* scratch,
                                                          uint32_t* sizes, uint32_t* begin) {
    const long long t = blockIdx.x * 128LL + threadIdx.x;
    if (t >= n_chan * spc) return;
    const long long chan = t / spc;
    const int j = static_cast<int>(t % spc);
    const long long stride = rans_stream_stride(hw, spc);
    uint16_t* const base = reinterpret_cast<uint16_t*>(scratch + t * stride);
    uint16_t* wp = base + stride / 2;
    uint32_t x = kRansL;
    const long long kmax = (hw + spc - 1) / spc;
    for (long long k = kmax - 1; k >= 0; --k) {
        const long long i = j + k * spc;
        if (i >= hw) continue;
        const long long e = chan * hw + i;
        const int l = lo[e], h = hi[e];
        if (v[e] == cdf_length[idx[e]] - 2) {  // escape: payload first (symbols are pushed in reverse decode order)
            const uint32_t r1 = static_cast<uint32_t>(raw[e]) + 1u;
            const int nb = 31 - __clz(r1);
            const uint32_t bits = r1 - (1u << nb);
            if (nb > 0) {
                const int lo_n = nb < 16 ? nb : 16;
                rans_put(x, wp, (bits & ((1u << lo_n) - 1u)) << (16 - lo_n), 1u << (16 - lo_n));
            }
            if (nb > 16) {
                const int hi_n = nb - 16;
                rans_put(x, wp, (bits >> 16) << (16 - hi_n), 1u << (16 - hi_n));
            }
            rans_put(x, wp, static_cast<uint32_t>(nb) << 11, 1u << 11);
        }
        rans_put(x, wp, static_cast<uint32_t>(l), static_cast<uint32_t>(h - l));
    }
    *--wp = static_cast<uint16_t>(x >> 16);  // u32 state, little endian, in front of the words
    *--wp = static_cast<uint16_t>(x & 0xFFFFu);
    sizes[t] = static_cast<uint32_t>((base + stride / 2 - wp) * 2);
    begin[t] = static_cast<uint32_t>((wp - base) * 2);
}

// exclusive scan of the stream sizes (single block; a few thousand to a few hundred thousand entries), and the header
__global__ void __launch_bounds__(1024) rans_scan_kernel(const uint32_t* __restrict__ sizes, unsigned long long* __restrict__ offs,
                                                         long long ns, unsigned long long first, unsigned long long* total) {
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = first;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (long long b0 = 0; b0 < ns; b0 += 1024) {
        const long long i = b0 + threadIdx.x;
        const unsigned long long val = i < ns ? sizes[i] : 0ull;
        unsigned long long inc = val;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long o = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += o;
        }
        if (lane == 31) warp_tot[w] = inc;
        __syncthreads();
        if (w == 0) {
            unsigned long long tinc = warp_tot[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned long long o = __shfl_up_sync(0xffffffffu, tinc, d);
                if (lane >= d) tinc += o;
            }
            warp_tot[lane] = tinc;
        }
        __syncthreads();
        const unsigned long long before = carry + (w ? warp_tot[w - 1] : 0ull) + inc - val;
        if (i < ns) offs[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + val;
        __syncthreads();
    }
    if (threadIdx.x == 0 && total) *total = carry;
}

__global__ void rans_header_kernel(uint8_t* out, const uint32_t* __restrict__ sizes, long long n_chan, long long hw, int spc) {
    const long long ns = n_chan * spc;
    uint32_t* o32 = reinterpret_cast<uint32_t*>(out);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        o32[0] = 0x52434443u;  // "CDCR"
        o32[1] = 1u;
        o32[2] = static_cast<uint32_t>(n_chan);
        o32[3] = static_cast<uint32_t>(hw);
        o32[4] = static_cast<uint32_t>(spc);
        o32[5] = 0u;
    }
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < ns; i += gridDim.x * 256LL) o32[6 + i] = sizes[i];
}

// one warp per stream: scratch -> its place in the container (2-byte units; offsets are even)
__global__ void __launch_bounds__(256) rans_pack_kernel(const uint8_t* __restrict__ scratch, const uint32_t* __restrict__ sizes,
                                                        const uint32_t* __restrict__ begin, const unsigned long long* __restrict__ offs,
                                                        long long ns, long long stride, uint8_t* out) {
    const long long s = (blockIdx.x * 256LL + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (s >= ns) return;
    const uint16_t* src = reinterpret_cast<const uint16_t*>(scratch + s * stride + begin[s]);
    uint16_t* dst = reinterpret_cast<uint16_t*>(out + offs[s]);
    const uint32_t n = sizes[s] / 2;
    for (uint32_t i = lane; i < n; i += 32) dst[i] = src[i];
}

long long rans_scratch_bytes(long long n_chan, long long hw, int spc) {
    const long long ns = n_chan * spc;
    return ns * rans_stream_stride(hw, spc) + ns * (4 + 4 + 8) + 64;  // regions, sizes, begin, offsets
}
long long rans_max_bytes(long long n_chan, long long hw, int spc) {
    const long long ns = n_chan * spc;
    return kRansHeader + 4 * ns + ns * rans_stream_stride(hw, spc);
}

cudaError_t launch_rans_encode(const int32_t* idx, const int32_t* v, const int32_t* lo, const int32_t* hi, const int32_t* raw,
                               const int32_t* cdf_length, long long n_chan, long long hw, int spc, void* scratch, uint8_t* out,
                               unsigned long long* out_bytes, cudaStream_t s) {
    const long long ns = n_chan * spc;
    if (ns <= 0) return cudaErrorInvalidValue;
    if (reinterpret_cast<uintptr_t>(out) & 3u) return cudaErrorMisalignedAddress;  // the header and size table are u32 stores
    const long long stride = rans_stream_stride(hw, spc);
    uint8_t* sc = static_cast<uint8_t*>(scratch);
    uint32_t* sizes = reinterpret_cast<uint32_t*>(sc + ns * stride);
    uint32_t* begin = sizes + ns;
    unsigned long long* offs = reinterpret_cast<unsigned long long*>((reinterpret_cast<uintptr_t>(begin + ns) + 7) & ~uintptr_t(7));
    rans_encode_kernel<<<static_cast<unsigned>((ns + 127) / 128), 128, 0, s>>>(idx, v, lo, hi, raw, cdf_length, n_chan, hw, spc, sc, sizes, begin);
    rans_scan_kernel<<<1, 1024, 0, s>>>(sizes, offs, ns, static_cast<unsigned long long>(kRansHeader + 4 * ns), out_bytes);
    rans_header_kernel<<<static_cast<unsigned>((ns + 255) / 256 < 256 ? (ns + 255) / 256 : 256), 256, 0, s>>>(out, sizes, n_chan, hw, spc);
    rans_pack_kernel<<<static_cast<unsigned>((ns * 32 + 255) / 256), 256, 0, s>>>(sc, sizes, begin, offs, ns, stride, out);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------- decode
__device__ __forceinline__ uint32_t rans_pop(uint32_t& x, const uint16_t*& rp, const uint16_t* end, uint32_t start, uint32_t freq, int& bad) {
    const uint32_t c = x & 0xFFFFu;
    x = freq * (x >> 16) + c - start;
    if (x < kRansL) {
        if (rp < end) {
            x = (x << 16) | *rp++;
        } else {
            bad = 1;
        }
    }
    return c;
}

__global__ void __launch_bounds__(128) rans_decode_kernel(const uint8_t* __restrict__ data, const unsigned long long* __restrict__ offs,
                                                          const int32_t* __restrict__ idx, CdfTables t, long long n_chan, long long hw,
                                                          int spc, long long data_bytes, int32_t* __restrict__ q, int32_t* status) {
    const long long tt = blockIdx.x * 128LL + threadIdx.x;
    if (tt >= n_chan * spc) return;
    const long long chan = tt / spc;
    const int j = static_cast<int>(tt % spc);
    const uint32_t* sizes = reinterpret_cast<const uint32_t*>(data + kRansHeader);
    if (sizes[tt] < 4 || (sizes[tt] & 1) || offs[tt] + sizes[tt] > static_cast<unsigned long long>(data_bytes)) {
        atomicExch(status, 1);  // the size table points outside the buffer: corrupt container
        return;
    }
    const uint16_t* rp = reinterpret_cast<const uint16_t*>(data + offs[tt]);
    const uint16_t* end = rp + sizes[tt] / 2;
    int bad = 0;
    uint32_t x = static_cast<uint32_t>(rp[0]) | (static_cast<uint32_t>(rp[1]) << 16);
    rp += 2;
    const long long kmax = (hw + spc - 1) / spc;
    for (long long k = 0; k < kmax && !bad; ++k) {
        const long long i = j + k * spc;
        if (i >= hw) break;
        const long long e = chan * hw + i;
        const int r = idx[e];
        const int32_t* row = t.cdf + t.row_start[r];
        const int max_v = t.cdf_length[r] - 2;
        const int c = static_cast<int>(x & 0xFFFFu);
        int a = 0, b = max_v;  // largest vv in [0, max_v] with row[vv] <= c
        while (a < b) {
            const int m = (a + b + 1) >> 1;
            if (__ldg(row + m) <= c) a = m; else b = m - 1;
        }
        const int start = __ldg(row + a), fr = __ldg(row + a + 1) - start;
        if (fr <= 0) {
            bad = 1;
            break;
        }
        rans_pop(x, rp, end, static_cast<uint32_t>(start), static_cast<uint32_t>(fr), bad);
        int vv = a;
        if (a == max_v) {  // escape payload: 5-bit length, then the low bits of raw + 1
            const int nb = static_cast<int>((x & 0xFFFFu) >> 11);
            rans_pop(x, rp, end, static_cast<uint32_t>(nb) << 11, 1u << 11, bad);
            uint32_t bits = 0;
            if (nb > 16) {
                const int hi_n = nb - 16;
                const uint32_t hv = (x & 0xFFFFu) >> (16 - hi_n);
                rans_pop(x, rp, end, hv << (16 - hi_n), 1u << (16 - hi_n), bad);
                bits = hv << 16;
            }
            if (nb > 0) {
                const int lo_n = nb < 16 ? nb : 16;
                const uint32_t lv = (x & 0xFFFFu) >> (16 - lo_n);
                rans_pop(x, rp, end, lv << (16 - lo_n), 1u << (16 - lo_n), bad);
                bits |= lv;
            }
            const long long rawv = static_cast<long long>((1u << nb) + bits) - 1;
            vv = (rawv & 1) ? static_cast<int>(-((rawv + 1) / 2)) : static_cast<int>(rawv / 2 + max_v);
        }
        q[e] = vv + t.offset[r];
    }
    if (bad || x != kRansL || rp != end) atomicExch(status, 1);  // truncated / corrupt / not consumed exactly
}

cudaError_t launch_rans_decode(const uint8_t* data, long long data_bytes, const int32_t* idx, CdfTables t, long long n_chan, long long hw,
                               int spc, void* scratch, int32_t* q, int32_t* status, cudaStream_t s) {
    const long long ns = n_chan * spc;
    if (ns <= 0) return cudaErrorInvalidValue;
    // the size table is read as u32 (a container that starts at an offset of 2 mod 4 in a larger buffer must be copied)
    if (reinterpret_cast<uintptr_t>(data) & 3u) return cudaErrorMisalignedAddress;
    if (data_bytes < kRansHeader + 4 * ns) return cudaErrorInvalidValue;  // before any launch reads the size table
    unsigned long long* offs = static_cast<unsigned long long*>(scratch);  // ns entries
    cudaError_t e = cudaMemsetAsync(status, 0, 4, s);
    if (e != cudaSuccess) return e;
    rans_scan_kernel<<<1, 1024, 0, s>>>(reinterpret_cast<const uint32_t*>(data + kRansHeader), offs, ns,
                                        static_cast<unsigned long long>(kRansHeader + 4 * ns), nullptr);
    rans_decode_kernel<<<static_cast<unsigned>((ns + 127) / 128), 128, 0, s>>>(data, offs, idx, t, n_chan, hw, spc, data_bytes, q, status);
    return cudaGetLastError();
}

}  // namespace cdc
