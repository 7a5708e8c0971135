// Integer kernels of the codec path (SURVEY.md 2.2 C10, section 8 rows a8/a9), bit-exact with
// oracle/entropy.py quantize_symbols / build_indexes / lookup_rows.  HBM-bound: 16 B/symbol
// (rounding) and 28 B/symbol (lookup); the 109 KB CDF table stays in L1/L2.
// Every global access of the streaming arrays is a 16-byte vector (four symbols per thread-iteration, grid-stride over
// one resident wave); a scalar tail covers n % 4 and unaligned callers.
#include "kernels.cuh"

namespace cdc {

// q = rint(y - mu) (round-half-even), y_hat = q + mu.  mu is elementwise (mu_mod == 0) or a
// per-channel vector indexed by (i / mu_inner) % mu_mod (factorised-prior medians).
__device__ __forceinline__ void quantize_one(float y, float m, int32_t& q, float& yh) {
    const float r = rintf(__fsub_rn(y, m));
    q = static_cast<int32_t>(r);
    yh = __fadd_rn(r, m);
}

// Block b owns the kVPT * 256 consecutive vectors starting at b * kVPT * 256; thread t takes vectors t, t + 256, ...:
// every load of the thread is issued before the first result is needed (kVPT x 2 independent 16-byte loads in flight),
// every access is coalesced, and the grid is one wave for the sizes this path sees (1025 blocks for 4 M symbols).
constexpr int kVPT = 4;

__global__ void __launch_bounds__(256) quantize_kernel(const float* __restrict__ y, const float* __restrict__ mu,
                                                       int32_t* __restrict__ q, float* __restrict__ yhat, long long n,
                                                       long long mu_inner, long long mu_mod, int vec) {
    const long long n4 = vec ? n / 4 : 0;
    const long long v0 = blockIdx.x * static_cast<long long>(kVPT * 256) + threadIdx.x;
    float4 yy[kVPT], mm[kVPT];
#pragma unroll
    for (int k = 0; k < kVPT; ++k) {
        const long long v = v0 + k * 256;
        if (v < n4) {
            yy[k] = reinterpret_cast<const float4*>(y)[v];
            if (!mu_mod) mm[k] = reinterpret_cast<const float4*>(mu)[v];
        }
    }
#pragma unroll
    for (int k = 0; k < kVPT; ++k) {
        const long long v = v0 + k * 256;
        if (v >= n4) continue;
        if (mu_mod) {
            const long long i = v * 4;
            mm[k].x = mu[(i / mu_inner) % mu_mod];
            mm[k].y = mu[((i + 1) / mu_inner) % mu_mod];
            mm[k].z = mu[((i + 2) / mu_inner) % mu_mod];
            mm[k].w = mu[((i + 3) / mu_inner) % mu_mod];
        }
        int4 qq;
        float4 hh;
        quantize_one(yy[k].x, mm[k].x, qq.x, hh.x);
        quantize_one(yy[k].y, mm[k].y, qq.y, hh.y);
        quantize_one(yy[k].z, mm[k].z, qq.z, hh.z);
        quantize_one(yy[k].w, mm[k].w, qq.w, hh.w);
        reinterpret_cast<int4*>(q)[v] = qq;
        if (yhat) reinterpret_cast<float4*>(yhat)[v] = hh;
    }
    // tail (or everything, for unaligned buffers): grid-stride scalars
    for (long long i = n4 * 4 + blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
        const float m = mu_mod ? mu[(i / mu_inner) % mu_mod] : mu[i];
        int32_t qi;
        float hi;
        quantize_one(y[i], m, qi, hi);
        q[i] = qi;
        if (yhat) yhat[i] = hi;
    }
}

static int int_grid(long long n, int vec, int num_sms) {
    if (vec) {
        const long long b = (n / 4 + kVPT * 256 - 1) / (kVPT * 256);
        return static_cast<int>(b < 1 ? 1 : b);
    }
    const long long want = (n + 255) / 256, cap = static_cast<long long>(num_sms) * 8;
    return static_cast<int>(want < cap ? want : cap);
}

cudaError_t launch_quantize(const float* y, const float* mu, int32_t* q, float* yhat, int64_t n, int64_t mu_inner,
                            int64_t mu_mod, int num_sms, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const int vec = al(y) && al(q) && (!yhat || al(yhat)) && (mu_mod || al(mu)) ? 1 : 0;
    quantize_kernel<<<int_grid(n, vec, num_sms), 256, 0, s>>>(y, mu, q, yhat, n, mu_inner, mu_mod, vec);
    return cudaGetLastError();
}

// idx = 63 - #{j in [0,62] : max(sigma, table[0]) <= table[j]}  (or the channel when sigma == null);
// v = q - offset[idx]; outside [0, max_v) -> escape; (lo, hi) = cdf[idx][v], cdf[idx][v+1].
struct ScaleSmem {
    float tab[64];
    float lg0, inv_step;  // log2(tab[0]), 63 / (log2(tab[63]) - log2(tab[0]))
};
struct CdfSmem {
    ScaleSmem sc;
    int32_t start[256], len[256], off[256];
};

__device__ __forceinline__ void load_scale_smem(ScaleSmem& sc, const float* __restrict__ scale_table) {  // (the caller syncs)
    if (threadIdx.x < 64) sc.tab[threadIdx.x] = scale_table[threadIdx.x];
    if (threadIdx.x == 0) {
        sc.lg0 = log2f(scale_table[0]);
        sc.inv_step = 63.0f / (log2f(scale_table[63]) - sc.lg0);
    }
}

// The CDF row of a Gaussian symbol: idx = 63 - #{j <= 62 : sg <= tab[j]} = #{j <= 62 : tab[j] < sg} on the ascending
// table.  The table is log-spaced, so a logarithm lands within one entry of the answer and two exact fix-up loops
// (comparisons against the table itself) make it exact: 63 compares + 63 adds per symbol had made the lookup ALU-bound
// (2.6 TB/s).  The encoder's lookup and the decoder's index kernel both call this, so they agree bit for bit.
__device__ __forceinline__ int scale_index(const ScaleSmem& sc, float sg_in) {
    const float sg = fmaxf(sg_in, sc.tab[0]);
    int g = static_cast<int>((__log2f(sg) - sc.lg0) * sc.inv_step) + 1;
    g = g < 0 ? 0 : (g > 63 ? 63 : g);
    while (g > 0 && !(sc.tab[g - 1] < sg)) --g;
    while (g < 63 && sc.tab[g] < sg) ++g;
    return g;
}

__device__ __forceinline__ void cdf_one(const CdfSmem& sm, const int32_t* __restrict__ cdf, int rows, bool has_sigma, float sg_in,
                                        int qv, long long i, long long inner, int32_t& idx_o, int32_t& v_o, int32_t& lo_o,
                                        int32_t& hi_o, int32_t& raw_o) {
    const int idx = has_sigma ? scale_index(sm.sc, sg_in) : static_cast<int>((i / inner) % rows);
    const int max_v = sm.len[idx] - 2;
    int v = qv - sm.off[idx];
    int raw = 0;
    if (v < 0) {
        raw = -2 * v - 1;
        v = max_v;
    } else if (v >= max_v) {
        raw = 2 * (v - max_v);
        v = max_v;
    }
    const int32_t* row = cdf + sm.start[idx];
    idx_o = idx;
    v_o = v;
    lo_o = __ldg(row + v);
    hi_o = __ldg(row + v + 1);
    raw_o = raw;
}

__global__ void __launch_bounds__(256) cdf_lookup_kernel(const int32_t* __restrict__ q, const float* __restrict__ sigma,
                                                         CdfTables t, long long inner, int32_t* __restrict__ idx_o,
                                                         int32_t* __restrict__ v_o, int32_t* __restrict__ lo_o,
                                                         int32_t* __restrict__ hi_o, int32_t* __restrict__ raw_o,
                                                         long long n, int vec) {
    __shared__ CdfSmem sm;
    if (t.scale_table) load_scale_smem(sm.sc, t.scale_table);
    for (int r = threadIdx.x; r < t.rows && r < 256; r += 256) {
        sm.start[r] = t.row_start[r];
        sm.len[r] = t.cdf_length[r];
        sm.off[r] = t.offset[r];
    }
    __syncthreads();
    const long long tid = blockIdx.x * 256LL + threadIdx.x, nthr = gridDim.x * 256LL;
    const long long n4 = vec ? n / 4 : 0;
    const bool hs = sigma != nullptr;
    const long long w0 = blockIdx.x * static_cast<long long>(kVPT * 256) + threadIdx.x;  // (see quantize_kernel)
    int4 qv[kVPT];
    float4 sv[kVPT];
#pragma unroll
    for (int k = 0; k < kVPT; ++k) {
        const long long w = w0 + k * 256;
        sv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (w < n4) {
            qv[k] = reinterpret_cast<const int4*>(q)[w];
            if (hs) sv[k] = reinterpret_cast<const float4*>(sigma)[w];
        }
    }
#pragma unroll
    for (int k = 0; k < kVPT; ++k) {
        const long long w = w0 + k * 256;
        if (w >= n4) continue;
        const int4 qq = qv[k];
        const float4 ss = sv[k];
        int4 a, b, c, d, e;
        const long long i = w * 4;
        cdf_one(sm, t.cdf, t.rows, hs, ss.x, qq.x, i, inner, a.x, b.x, c.x, d.x, e.x);
        cdf_one(sm, t.cdf, t.rows, hs, ss.y, qq.y, i + 1, inner, a.y, b.y, c.y, d.y, e.y);
        cdf_one(sm, t.cdf, t.rows, hs, ss.z, qq.z, i + 2, inner, a.z, b.z, c.z, d.z, e.z);
        cdf_one(sm, t.cdf, t.rows, hs, ss.w, qq.w, i + 3, inner, a.w, b.w, c.w, d.w, e.w);
        reinterpret_cast<int4*>(idx_o)[w] = a;
        reinterpret_cast<int4*>(v_o)[w] = b;
        reinterpret_cast<int4*>(lo_o)[w] = c;
        reinterpret_cast<int4*>(hi_o)[w] = d;
        reinterpret_cast<int4*>(raw_o)[w] = e;
    }
    for (long long i = n4 * 4 + tid; i < n; i += nthr)
        cdf_one(sm, t.cdf, t.rows, hs, hs ? sigma[i] : 0.f, q[i], i, inner, idx_o[i], v_o[i], lo_o[i], hi_o[i], raw_o[i]);
}

cudaError_t launch_cdf_lookup(const int32_t* q, const float* sigma, CdfTables t, int64_t inner, int32_t* idx,
                              int32_t* v, int32_t* lo, int32_t* hi, int32_t* raw, int64_t n, int num_sms,
                              cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    if (t.rows > 256 || (sigma && !t.scale_table)) return cudaErrorInvalidValue;
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const int vec = al(q) && (!sigma || al(sigma)) && al(idx) && al(v) && al(lo) && al(hi) && al(raw) ? 1 : 0;
    cdf_lookup_kernel<<<int_grid(n, vec, num_sms), 256, 0, s>>>(q, sigma, t, inner, idx, v, lo, hi, raw, n, vec);
    return cudaGetLastError();
}

// The decoder's CDF rows of y: idx NCHW int32 [B][C][HW] = scale_index(max(sigma, min_sigma)) with sigma channels
// [c_off, c_off + C) of an NHWC act_t tensor (the hyper-decoder's output), through a 32 x 32 shared tile as
// nhwc_slice_to_nchw_kernel transposes.  Gives the idx of cdf_lookup on the NCHW fp32 sigma of cdc_hyper_decode without
// the fp32 round trip.
__global__ void __launch_bounds__(256) scale_rows_kernel(const act_t* __restrict__ src, const float* __restrict__ scale_table,
                                                         int32_t* __restrict__ idx, int C, int HW, int ldc, int c_off, float min_sigma) {
    __shared__ ScaleSmem sc;
    __shared__ float tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    load_scale_smem(sc, scale_table);
    for (int j = ty; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + tx;
        tile[j][tx] = (c < C && p < HW) ? from_act(src[(static_cast<size_t>(b) * HW + p) * ldc + c_off + c]) : 0.f;
    }
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + tx;
        if (p < HW && c < C) idx[(static_cast<size_t>(b) * C + c) * HW + p] = scale_index(sc, fmaxf(tile[tx][j], min_sigma));
    }
}

cudaError_t launch_scale_rows(const act_t* src, int ldc, int c_off, float min_sigma, const float* scale_table, int32_t* idx, int B,
                              int C, int HW, cudaStream_t s) {
    if (!scale_table) return cudaErrorInvalidValue;
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    scale_rows_kernel<<<grid, 256, 0, s>>>(src, scale_table, idx, C, HW, ldc, c_off, min_sigma);
    return cudaGetLastError();
}

}  // namespace cdc
