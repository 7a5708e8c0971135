// HBM-/latency-bound kernels around K-conv: GroupNorm statistics / apply(+SiLU,+residual),
// time-embedding MLP + FiLM vectors, layout conversion at the API boundary, weight repack.
// Oracle counterparts: oracle/unet.py RB, Attn.gn, TimeEmbed; SURVEY.md 2.2 C5, C6, C8.
#include "gn_apply.cuh"
#include "gn_sums.cuh"
#include "kernels.cuh"
#include "ptx.cuh"
#include "sampler.cuh"

namespace cdc {

// ------------------------------------------------------------------------------------------------
// Standalone GN statistics (used where the producer is not a conv epilogue: attention input).
// One CTA per (image, 64-pixel chunk); fixed-order reductions only.
constexpr int kStatsPix = 64;

__global__ void __launch_bounds__(256) gn_stats_kernel(const act_t* x, gn_sum_t* acc, int HW, int C, long long* stamp) {
    __shared__ float s_sum[8][512], s_sq[8][512];  // [row-in-pass][channel] (C <= 512)
    if (threadIdx.x == 0) stamp_begin(stamp);
    const int b = blockIdx.y, pt = blockIdx.x;
    const int vecs = C / 8;                 // uint4 per pixel
    const int rows = (256 / vecs) < 8 ? (256 / vecs) : 8;  // pixels per pass (smem rows)
    const int t = threadIdx.x, cv = t % vecs, pr = t / vecs;
    float s[8], q[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
    const int p0 = pt * kStatsPix;
    if (pr < rows) {
        for (int pp = pr; pp < kStatsPix && p0 + pp < HW; pp += rows) {
            const uint4 u = *reinterpret_cast<const uint4*>(x + (static_cast<size_t>(b) * HW + p0 + pp) * C + cv * 8);
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float a = act_lo(w[j]), c = act_hi(w[j]);
                s[2 * j] += a;
                q[2 * j] += a * a;
                s[2 * j + 1] += c;
                q[2 * j + 1] += c * c;
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            s_sum[pr][cv * 8 + j] = s[j];
            s_sq[pr][cv * 8 + j] = q[j];
        }
    }
    __syncthreads();
    // per-channel totals over the pass rows, then per-group totals, all in fixed order
    __shared__ float c_sum[512], c_sq[512];
    for (int c = t; c < C; c += 256) {
        float a = 0.f, d = 0.f;
        for (int r = 0; r < rows && r < 8; ++r) {
            a += s_sum[r][c];
            d += s_sq[r][c];
        }
        c_sum[c] = a;
        c_sq[c] = d;
    }
    __syncthreads();
    if (t < 32) {
        const int cpg = C / 32;
        float a = 0.f, d = 0.f;
        for (int j = 0; j < cpg; ++j) {
            a += c_sum[t * cpg + j];
            d += c_sq[t * cpg + j];
        }
        gn_sums_add(acc + static_cast<size_t>(b) * kGnImgStride, t, a, d);
    }
    if (threadIdx.x == 0) stamp_end(stamp);
}

cudaError_t launch_gn_stats(const act_t* x, gn_sum_t* acc, int B, int HW, int C, cudaStream_t s, long long* stamp) {
    if (C % 32 != 0 || C > 512 || C < 32) return cudaErrorInvalidValue;
    const int PT = (HW + kStatsPix - 1) / kStatsPix;
    gn_stats_kernel<<<dim3(PT, B), 256, 0, s>>>(x, acc, HW, C, stamp);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Apply: y = SiLU(a*x + b) (+ r), 8 channels (16 B) per thread, grid-stride.
// GroupNorm coefficients of this thread's 8 channels, y = a*x + b with the affine and FiLM (1 + s, sh) folded in, from
// the fixed-point (sum, sum of squares) accumulators of the image (gn_sums.cuh).  Same arithmetic as the oracle's
// F.group_norm + FiLM (oracle/unet.py RB): mean / variance in double, rstd = 1 / sqrt(var + eps).
struct GnCoef {
    const gn_sum_t* acc;   // [B][32][2]; written by the preceding kernel: plain (coherent) loads only
    const float* gamma;
    const float* beta;
    const float* film;     // [2C] (scale | shift) of this step, or null
    int C, HW;
    float eps;
    long long* stamp;   // diagnostics, may be null
    unsigned int* sat;  // counts threads that stored a saturated value (residual path), may be null
};
// (mean, rstd) of every (image, group), once per CTA: exact integer totals -> double mean / variance (a handful of
// FP64 multiply-adds), rstd in fp32 (MUFU rsqrt + one Newton step, < 1 ulp) like the oracle's fp32 group_norm.
__device__ __forceinline__ void gn_group_stats(const GnCoef& g, int B, float2* s_mr) {
    const int cpg = g.C / 32;
    const double inv_n = 1.0 / (static_cast<double>(cpg) * g.HW);
    for (int i = threadIdx.x; i < B * 32; i += blockDim.x) {
        s_mr[i] = gn_mean_rstd(g.acc + static_cast<size_t>(i) * kGnVals, inv_n, g.eps);
    }
    __syncthreads();
}
// This thread's 8 channels: GroupNorm affine and FiLM, loaded once (they do not depend on the statistics, so the
// loads are issued before the statistics phase and overlap it)
struct GnChan {
    float gamma[8], beta[8], sc[8], sh[8];
};
__device__ __forceinline__ void gn_load_chan(const GnCoef& g, int c0, GnChan& k) {
    const float4* ga = reinterpret_cast<const float4*>(g.gamma + c0);
    const float4* be = reinterpret_cast<const float4*>(g.beta + c0);
    const float4 g0 = ga[0], g1 = ga[1], b0 = be[0], b1 = be[1];
    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0, h0 = s0, h1 = s0;
    if (g.film) {
        const float4* fs = reinterpret_cast<const float4*>(g.film + c0);
        const float4* fh = reinterpret_cast<const float4*>(g.film + g.C + c0);
        s0 = fs[0], s1 = fs[1], h0 = fh[0], h1 = fh[1];
    }
    const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w}, bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
    const float ss[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w}, hh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        k.gamma[j] = gg[j];
        k.beta[j] = bb[j];
        k.sc[j] = 1.0f + ss[j];
        k.sh[j] = hh[j];
    }
}
__device__ __forceinline__ void gn_coef(const GnChan& k, const float2* s_mr, int b, int c0, int cpg, float4 (&c)[4]) {
    float ab[16];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float2 f = gn_fold(k.gamma[j], k.beta[j], k.sc[j], k.sh[j], s_mr[b * 32 + (c0 + j) / cpg]);  // (s = sh = 0 without FiLM)
        ab[2 * j] = f.x;
        ab[2 * j + 1] = f.y;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) c[j] = make_float4(ab[4 * j], ab[4 * j + 1], ab[4 * j + 2], ab[4 * j + 3]);
}

// The grid stride is a multiple of the vectors per pixel, so a thread always owns the same 8 channels:
// its (a, b) pairs live in registers and are recomputed only when the image index changes.  64 registers at most:
// 4 CTAs per SM, and the grid is exactly one resident wave (the statistics prologue is paid once per CTA).
template <bool SILU, bool RES>
__global__ void __launch_bounds__(256, 4) gn_apply_kernel(const uint4* x, const uint4* r, uint4* y, long long nvec, int vecs_per_pix,
                                                          long long vecs_per_img, const GnCoef g, int B) {
    extern __shared__ float2 s_mr[];  // [B][32] (mean, rstd)
    if (threadIdx.x == 0) stamp_begin(g.stamp);
    const long long stride = gridDim.x * 256LL;
    long long i = blockIdx.x * 256LL + threadIdx.x;
    const int cv = static_cast<int>(i % vecs_per_pix), cpg = g.C / 32;
    const bool single = vecs_per_img >= nvec;  // one image: skip the 64-bit divide
    float4 c[4];
    int cur_b;
    {   // channel constants and the first vectors are in flight before the statistics phase (none depends on it)
        GnChan k;
        gn_load_chan(g, cv * 8, k);
        gn_group_stats(g, B, s_mr);
        cur_b = (single || i >= nvec) ? 0 : static_cast<int>(i / vecs_per_img);
        gn_coef(k, s_mr, cur_b, cv * 8, cpg, c);
    }
    uint32_t satm = 0u;
    for (; i < nvec; i += 2 * stride) {
        const long long i2 = i + stride;
        const bool has2 = i2 < nvec;
        const uint4 u0 = x[i];
        uint4 u1 = make_uint4(0, 0, 0, 0), r0 = u1, r1 = u1;
        if (has2) u1 = x[i2];
        if (RES) {
            r0 = r[i];
            if (has2) r1 = r[i2];
        }
        int b = single ? 0 : static_cast<int>(i / vecs_per_img);
        if (b != cur_b) {  // (batch > 1 only) reload this thread's channel constants: L2 hits
            GnChan k;
            gn_load_chan(g, cv * 8, k);
            gn_coef(k, s_mr, b, cv * 8, cpg, c);
            cur_b = b;
        }
        const uint4 y0 = gn_apply_vec<SILU, RES>(u0, r0, c);
        y[i] = y0;
        if (RES) satm = act2_absmax(satm, y0);
        if (has2) {
            b = single ? 0 : static_cast<int>(i2 / vecs_per_img);
            if (b != cur_b) {
                GnChan k;
                gn_load_chan(g, cv * 8, k);
                gn_coef(k, s_mr, b, cv * 8, cpg, c);
                cur_b = b;
            }
            const uint4 y1 = gn_apply_vec<SILU, RES>(u1, r1, c);
            y[i2] = y1;
            if (RES) satm = act2_absmax(satm, y1);
        }
    }
    if (RES && act2_is_sat(satm) && g.sat) atomicAdd(g.sat, 1u);
    if (threadIdx.x == 0) stamp_end(g.stamp);
}

cudaError_t launch_gn_apply(const act_t* x, const gn_sum_t* acc, const float* gamma, const float* beta, const float* film,
                            float eps, const act_t* r, act_t* y, int B, int HW, int C, int silu, int num_sms, cudaStream_t s,
                            long long* stamp, unsigned int* sat) {
    const long long nvec = static_cast<long long>(B) * HW * C / 8;
    const int vpp = C / 8;
    const long long vpi = static_cast<long long>(HW) * vpp;
    long long want = (nvec + 511) / 512;
    const long long cap = static_cast<long long>(num_sms) * 4;  // one resident wave (__launch_bounds__(256, 4))
    long long grid = want < cap ? want : cap;
    // (grid * 256) % vpp == 0  <=>  the per-thread channel vector is loop-invariant
    const int need = vpp % 3 == 0 ? 3 : 1;  // 256 covers the power-of-two part of vpp (8, 16, 32, 64)
    grid = (grid + need - 1) / need * need;
    if ((grid * 256) % vpp != 0 || C % 32 != 0) return cudaErrorInvalidValue;
    const uint4* xv = reinterpret_cast<const uint4*>(x);
    const uint4* rv = reinterpret_cast<const uint4*>(r);
    uint4* yv = reinterpret_cast<uint4*>(y);
    const dim3 g(static_cast<unsigned>(grid)), blk(256);
    const GnCoef gc{acc, gamma, beta, film, C, HW, eps, stamp, sat};
    const size_t sm = static_cast<size_t>(B) * 32 * sizeof(float2);
    if (sm > 48 * 1024) return cudaErrorInvalidValue;
    auto kern = silu ? (r ? gn_apply_kernel<true, true> : gn_apply_kernel<true, false>)
                     : (r ? gn_apply_kernel<false, true> : gn_apply_kernel<false, false>);
    kern<<<g, blk, sm, s>>>(xv, rv, yv, nvec, vpp, vpi, gc, B);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Time embedding + all FiLM vectors for every step of the schedule (runs once per set_schedule).
// One CTA per step.  fp32 throughout, accurate expf (the oracle is fp32 eager).
__device__ __forceinline__ float silu_acc(float v) { return v / (1.0f + expf(-v)); }

__global__ void __launch_bounds__(256) temb_film_kernel(const __grid_constant__ FilmParams p) {
    __shared__ float e[64], h1[256], te[256];
    const int k = blockIdx.x, t = threadIdx.x;
    if (t < 64) e[t] = p.sinus[k * 64 + t];
    __syncthreads();
    for (int o = t; o < p.temb; o += 256) {
        float acc = p.b1[o];
        for (int i = 0; i < 64; ++i) acc = fmaf(p.w1[o * 64 + i], e[i], acc);
        h1[o] = silu_acc(acc);
    }
    __syncthreads();
    for (int o = t; o < p.temb; o += 256) {
        float acc = p.b2[o];
        for (int i = 0; i < p.temb; ++i) acc = fmaf(p.w2[o * p.temb + i], h1[i], acc);
        te[o] = silu_acc(acc);  // every consumer applies SiLU(te) first
    }
    __syncthreads();
    const int warp = t >> 5, lane = t & 31;
    for (int l = 0; l < p.nlayers; ++l) {
        const FilmLayer L = p.layer[l];
        for (int o = warp; o < L.c2; o += 8) {
            float acc = 0.f;
            for (int i = lane; i < p.temb; i += 32) acc = fmaf(L.w[o * p.temb + i], te[i], acc);
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m);
            if (lane == 0) p.out[static_cast<size_t>(k) * p.total + L.offset + o] = acc + L.b[o];
        }
    }
}

cudaError_t launch_temb_film(const FilmParams& p, int K, cudaStream_t s) {
    if (p.temb > 256) return cudaErrorInvalidValue;
    temb_film_kernel<<<K, 256, 0, s>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Layout conversion (API boundary: NCHW fp32 tensors <-> device NHWC act_t / fp32).
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, act_t* __restrict__ dst, int C, int HW,
                                    int ldc) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + threadIdx.x;
        tile[j][threadIdx.x] = (c < C && p < HW) ? src[(static_cast<size_t>(b) * C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + threadIdx.x;
        if (p < HW && c < C) dst[(static_cast<size_t>(b) * HW + p) * ldc + c] = to_act(tile[threadIdx.x][j]);
    }
}
cudaError_t launch_nchw_f32_to_nhwc_act(const float* src, act_t* dst, int B, int C, int HW, int ldc,
                                         cudaStream_t s) {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    nchw_to_nhwc_kernel<<<grid, dim3(32, 8), 0, s>>>(src, dst, C, HW, ldc);
    return cudaGetLastError();
}

__global__ void nhwc_to_nchw_kernel(const act_t* __restrict__ src, float* __restrict__ dst, int C, int HW) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + threadIdx.x;
        tile[j][threadIdx.x] = (c < C && p < HW) ? from_act(src[(static_cast<size_t>(b) * HW + p) * C + c]) : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + threadIdx.x;
        if (p < HW && c < C) dst[(static_cast<size_t>(b) * C + c) * HW + p] = tile[threadIdx.x][j];
    }
}
cudaError_t launch_nhwc_act_to_nchw_f32(const act_t* src, float* dst, int B, int C, int HW, cudaStream_t s) {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    nhwc_to_nchw_kernel<<<grid, dim3(32, 8), 0, s>>>(src, dst, C, HW);
    return cudaGetLastError();
}

__global__ void x_in_kernel(const float* __restrict__ x, float* __restrict__ xs, act_t* __restrict__ xpad,
                            long long n, int HW) {
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
        const long long b = i / HW, p = i % HW;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float v = x[(b * 3 + c) * HW + p];
            xs[i * 3 + c] = v;
            xpad[i * kXpadC + c] = to_act(v);
        }
    }
}
cudaError_t launch_x_in(const float* x_nchw, float* xs, act_t* xpad, int B, int HW, cudaStream_t s) {
    const long long n = static_cast<long long>(B) * HW;
    x_in_kernel<<<static_cast<int>((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, s>>>(x_nchw, xs, xpad, n, HW);
    return cudaGetLastError();
}

// x_T = gamma * z of every image from its own seed (sampler.cuh, counter (pixel within the image, 0, 1)), written where
// launch_x_in would put it: xs through shared memory as whole float4s, xpad as one 32-byte sector per pixel (channels
// 3..15 zero, as the DDIM epilogue stores them).
constexpr int kInitPix = 256;
__global__ void __launch_bounds__(kInitPix) init_noise_kernel(const unsigned long long* __restrict__ seeds, float* __restrict__ xs,
                                                              act_t* __restrict__ xpad, float gamma, long long n, int HW) {
    __shared__ __align__(16) float tile[kInitPix * 3];
    for (long long i0 = static_cast<long long>(blockIdx.x) * kInitPix; i0 < n; i0 += static_cast<long long>(gridDim.x) * kInitPix) {
        const long long i = i0 + threadIdx.x;
        if (i < n) {
            const long long b = i / HW;
            float z[3];
            philox_normal3(seeds[1 + b], static_cast<unsigned long long>(i - b * HW), 0u, 1u, z);
            const float v0 = gamma * z[0], v1 = gamma * z[1], v2 = gamma * z[2];
            tile[threadIdx.x * 3 + 0] = v0;
            tile[threadIdx.x * 3 + 1] = v1;
            tile[threadIdx.x * 3 + 2] = v2;
            st_global_v8(xpad + i * kXpadC, make_uint4(pack_act2(v0, v1), pack_act2(v2, 0.0f), 0u, 0u), make_uint4(0u, 0u, 0u, 0u));
        }
        __syncthreads();
        const long long m = (n - i0 < kInitPix ? n - i0 : kInitPix) * 3;  // floats of this chunk
        if (m == kInitPix * 3) {
            if (threadIdx.x < kInitPix * 3 / 4)
                reinterpret_cast<float4*>(xs + i0 * 3)[threadIdx.x] = reinterpret_cast<const float4*>(tile)[threadIdx.x];
        } else {
            for (int j = threadIdx.x; j < m; j += kInitPix) xs[i0 * 3 + j] = tile[j];
        }
        __syncthreads();
    }
}
cudaError_t launch_init_noise(const unsigned long long* seeds, float* xs, act_t* xpad, float gamma, int B, int HW, cudaStream_t s) {
    const long long n = static_cast<long long>(B) * HW;
    const long long blocks = (n + kInitPix - 1) / kInitPix;
    init_noise_kernel<<<static_cast<int>(blocks < 8192 ? blocks : 8192), kInitPix, 0, s>>>(seeds, xs, xpad, gamma, n, HW);
    return cudaGetLastError();
}

// The sampler state as an image value in [0, 1]; cdc_get_x(to_image) and the 8-bit output both map through it.
__device__ __forceinline__ float image01(float v) { return (fminf(fmaxf(v, -1.0f), 1.0f) + 1.0f) / 2.0f; }

// Pixel i of xs (NHWC, 3 fp32 channels) -> its three NCHW planes: consecutive threads store consecutive pixels of a plane.
__device__ __forceinline__ void x_out_pixel(const float* __restrict__ xs, float* __restrict__ x, long long i, int HW, int to_image) {
    const long long b = i / HW, p = i % HW;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float v = xs[i * 3 + c];
        if (to_image) v = image01(v);
        x[(b * 3 + c) * HW + p] = v;
    }
}
__global__ void x_out_kernel(const float* __restrict__ xs, float* __restrict__ x, long long n, int HW, int to_image) {
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) x_out_pixel(xs, x, i, HW, to_image);
}
static int x_out_grid(long long n) { return static_cast<int>((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096); }
cudaError_t launch_x_out(const float* xs, float* x_nchw, int B, int HW, int to_image, cudaStream_t s) {
    const long long n = static_cast<long long>(B) * HW;
    x_out_kernel<<<x_out_grid(n), 256, 0, s>>>(xs, x_nchw, n, HW, to_image);
    return cudaGetLastError();
}

// Trajectory store: the slot pointers are read from `dst` when the kernel runs, so a captured graph serves any buffers.
__global__ void traj_store_kernel(const float* __restrict__ xs, const float* __restrict__ x0s, const TrajPtrs* dst,
                                  long long slot_x, long long slot_x0, long long n, int HW) {
    float* x = slot_x >= 0 && dst->x ? dst->x + slot_x * n * 3 : nullptr;
    float* x0 = slot_x0 >= 0 && dst->x0 ? dst->x0 + slot_x0 * n * 3 : nullptr;
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
        if (x) x_out_pixel(xs, x, i, HW, 0);
        if (x0) x_out_pixel(x0s, x0, i, HW, 0);
    }
}
cudaError_t launch_traj_store(const float* xs, const float* x0s, const TrajPtrs* dst, int slot_x, int slot_x0, int B, int HW,
                              cudaStream_t s) {
    const long long n = static_cast<long long>(B) * HW;
    traj_store_kernel<<<x_out_grid(n), 256, 0, s>>>(xs, x0s, dst, slot_x, slot_x0, n, HW);
    return cudaGetLastError();
}

__global__ void traj_set_ptrs_kernel(TrajPtrs* dst, float* x, float* x0) {
    dst->x = x;
    dst->x0 = x0;
}
cudaError_t launch_traj_set_ptrs(TrajPtrs* dst, float* x, float* x0, cudaStream_t s) {
    traj_set_ptrs_kernel<<<1, 1, 0, s>>>(dst, x, x0);
    return cudaGetLastError();
}

// OIHW fp32 -> [O_pad][taps][I_pad] bf16; input channel i < split keeps slot i, i >= split moves to
// split_pad + (i - split); everything else is zero.
__global__ void repack_weight_kernel(const float* __restrict__ src, act_t* __restrict__ dst, int O, int I,
                                     int taps, int O_pad, int I_pad, int split, int split_pad) {
    const long long n = static_cast<long long>(O_pad) * taps * I_pad;
    for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < n; idx += gridDim.x * 256LL) {
        const int slot = static_cast<int>(idx % I_pad);
        const int tap = static_cast<int>((idx / I_pad) % taps);
        const int o = static_cast<int>(idx / (static_cast<long long>(I_pad) * taps));
        int i = -1;
        if (slot < split) i = slot;
        else if (slot >= split_pad && slot - split_pad + split < I) i = slot - split_pad + split;
        float v = 0.f;
        if (o < O && i >= 0 && i < I) v = src[(static_cast<size_t>(o) * I + i) * taps + tap];
        dst[idx] = to_act(v);
    }
}
cudaError_t launch_repack_weight(const float* src, act_t* dst, int O, int I, int taps, int O_pad, int I_pad,
                                 int split, int split_pad, cudaStream_t s) {
    const long long n = static_cast<long long>(O_pad) * taps * I_pad;
    repack_weight_kernel<<<static_cast<int>((n + 255) / 256 < 2048 ? (n + 255) / 256 : 2048), 256, 0, s>>>(
        src, dst, O, I, taps, O_pad, I_pad, split, split_pad);
    return cudaGetLastError();
}

// Nearest-x2-then-conv3x3 == four 2x2 convolutions on the low-resolution input, one per output parity
// (py, px), with phase weights that are sums of the original taps:
//   rows:  py = 0 -> {dh -1: kh 0 | dh 0: kh 1+2},   py = 1 -> {dh 0: kh 0+1 | dh +1: kh 2}   (same for columns)
// dst: [O_pad][16 = (ph, a, b)][I_pad], summed in fp32 and rounded once (the originals are bf16-exact, so
// the sums are almost always exact in fp16).  2.25x fewer MMAs than evaluating the 9 taps per parity.
__global__ void repack_weight_up2_kernel(const float* __restrict__ src, act_t* __restrict__ dst, int O, int I,
                                         int O_pad, int I_pad) {
    const long long n = static_cast<long long>(O_pad) * 16 * I_pad;
    for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < n; idx += gridDim.x * 256LL) {
        const int i = static_cast<int>(idx % I_pad);
        const int t = static_cast<int>((idx / I_pad) % 16);
        const int o = static_cast<int>(idx / (static_cast<long long>(I_pad) * 16));
        const int ph = t >> 2, a = (t >> 1) & 1, b = t & 1, py = ph >> 1, px = ph & 1;
        const int kh0 = py == 0 ? (a == 0 ? 0 : 1) : (a == 0 ? 0 : 2), kh1 = py == 0 ? (a == 0 ? 0 : 2) : (a == 0 ? 1 : 2);
        const int kw0 = px == 0 ? (b == 0 ? 0 : 1) : (b == 0 ? 0 : 2), kw1 = px == 0 ? (b == 0 ? 0 : 2) : (b == 0 ? 1 : 2);
        float v = 0.f;
        if (o < O && i < I)
            for (int kh = kh0; kh <= kh1; ++kh)
                for (int kw = kw0; kw <= kw1; ++kw) v += src[(static_cast<size_t>(o) * I + i) * 9 + kh * 3 + kw];
        dst[idx] = to_act(v);
    }
}
cudaError_t launch_repack_weight_up2(const float* src, act_t* dst, int O, int I, int O_pad, int I_pad, cudaStream_t s) {
    const long long n = static_cast<long long>(O_pad) * 16 * I_pad;
    repack_weight_up2_kernel<<<static_cast<int>((n + 255) / 256 < 2048 ? (n + 255) / 256 : 2048), 256, 0, s>>>(src, dst, O, I,
                                                                                                            O_pad, I_pad);
    return cudaGetLastError();
}

// ConvTranspose2d(5, stride 2, padding 2, output_padding 1): out[2h+py][2w+px] = sum over taps ky = py + 2a', kx = px + 2b'
// of in[h + 1 - a'][w + 1 - b'] * W[ci][co][ky][kx]  (ky <= 4).  Parity 0 has three taps per axis (ky 0, 2, 4 -> rows
// h+1, h, h-1), parity 1 two (ky 1, 3 -> rows h+1, h).  dst tap index = parity * 9 + a * 3 + b with row offset 1 - a.
__global__ void repack_weight_convt5_kernel(const float* __restrict__ src, act_t* __restrict__ dst, int O, int I, int O_pad, int I_pad) {
    const long long n = static_cast<long long>(O_pad) * 36 * I_pad;
    for (long long idx = blockIdx.x * 256LL + threadIdx.x; idx < n; idx += gridDim.x * 256LL) {
        const int i = static_cast<int>(idx % I_pad);
        const int t = static_cast<int>((idx / I_pad) % 36);
        const int o = static_cast<int>(idx / (static_cast<long long>(I_pad) * 36));
        const int ph = t / 9, a = (t % 9) / 3, b = t % 3, py = ph >> 1, px = ph & 1;
        const int ky = py + 2 * a, kx = px + 2 * b;
        float v = 0.f;
        if (o < O && i < I && ky <= 4 && kx <= 4) v = src[((static_cast<size_t>(i) * O + o) * 5 + ky) * 5 + kx];
        dst[idx] = to_act(v);
    }
}
cudaError_t launch_repack_weight_convt5(const float* src, act_t* dst, int O, int I, int O_pad, int I_pad, cudaStream_t s) {
    const long long n = static_cast<long long>(O_pad) * 36 * I_pad;
    repack_weight_convt5_kernel<<<static_cast<int>((n + 255) / 256 < 2048 ? (n + 255) / 256 : 2048), 256, 0, s>>>(src, dst, O, I, O_pad, I_pad);
    return cudaGetLastError();
}

__global__ void img_in_kernel(const float* __restrict__ img, act_t* __restrict__ dst, long long n, int HW) {
    for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
        const long long b = i / HW, p = i % HW;
#pragma unroll
        for (int c = 0; c < 3; ++c) dst[i * 64 + c] = to_act(2.0f * img[(b * 3 + c) * HW + p] - 1.0f);
    }
}
cudaError_t launch_img_in(const float* img_nchw, act_t* dst64, int B, int HW, cudaStream_t s) {
    const long long n = static_cast<long long>(B) * HW;
    img_in_kernel<<<static_cast<int>((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, s>>>(img_nchw, dst64, n, HW);
    return cudaGetLastError();
}

// 8-bit interleaved RGB [n][3] -> img64 channels 0..2 (channel 3 written zero, as it already is), 16 pixels = three 16-byte
// loads per thread.  2 * (v / 255) - 1 with the division IEEE-rounded as the host's u8 / 255 in fp32 is, so the
// analysis encoder sees exactly the values launch_img_in makes of that fp32 image.
__global__ void __launch_bounds__(256) rgb8_in_kernel(const uint8_t* __restrict__ rgb, act_t* __restrict__ dst, long long n16) {
    for (long long g = blockIdx.x * 256LL + threadIdx.x; g < n16; g += gridDim.x * 256LL) {
        const uint4* src = reinterpret_cast<const uint4*>(rgb + g * 48);
        uint4 raw[3] = {src[0], src[1], src[2]};
        const uint8_t* v = reinterpret_cast<const uint8_t*>(raw);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            uint2 w;
            act_t* px = reinterpret_cast<act_t*>(&w);
#pragma unroll
            for (int c = 0; c < 3; ++c) px[c] = to_act(2.0f * (static_cast<float>(v[k * 3 + c]) / 255.0f) - 1.0f);
            px[3] = to_act(0.0f);
            *reinterpret_cast<uint2*>(dst + (g * 16 + k) * 64) = w;
        }
    }
}
cudaError_t launch_rgb8_in(const uint8_t* rgb, act_t* dst64, long long npix, cudaStream_t s) {
    if (npix % 16 || (reinterpret_cast<uintptr_t>(rgb) & 15u)) return cudaErrorInvalidValue;
    const long long n16 = npix / 16;
    rgb8_in_kernel<<<static_cast<int>((n16 + 255) / 256 < 4096 ? (n16 + 255) / 256 : 4096), 256, 0, s>>>(rgb, dst64, n16);
    return cudaGetLastError();
}

// xs [n][3] fp32 -> 8-bit interleaved RGB: round_half_even(255 * image01(x)), 16 pixels = twelve 16-byte loads and three
// 16-byte stores per thread.
__global__ void __launch_bounds__(256) rgb8_out_kernel(const float* __restrict__ xs, uint8_t* __restrict__ rgb, long long n16) {
    for (long long g = blockIdx.x * 256LL + threadIdx.x; g < n16; g += gridDim.x * 256LL) {
        const float4* src = reinterpret_cast<const float4*>(xs + g * 48);
        uint4 out[3];
        uint32_t* o = reinterpret_cast<uint32_t*>(out);
#pragma unroll
        for (int k = 0; k < 12; ++k) {
            const float4 f = src[k];
            const float e[4] = {f.x, f.y, f.z, f.w};
            uint32_t w = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) w |= static_cast<uint32_t>(static_cast<uint8_t>(rintf(__fmul_rn(image01(e[j]), 255.0f)))) << (8 * j);
            o[k] = w;
        }
        uint4* dst = reinterpret_cast<uint4*>(rgb + g * 48);
        dst[0] = out[0];
        dst[1] = out[1];
        dst[2] = out[2];
    }
}
cudaError_t launch_rgb8_out(const float* xs, uint8_t* rgb, long long npix, cudaStream_t s) {
    if (npix % 16 || (reinterpret_cast<uintptr_t>(rgb) & 15u) || (reinterpret_cast<uintptr_t>(xs) & 15u)) return cudaErrorInvalidValue;
    const long long n16 = npix / 16;
    rgb8_out_kernel<<<static_cast<int>((n16 + 255) / 256 < 4096 ? (n16 + 255) / 256 : 4096), 256, 0, s>>>(xs, rgb, n16);
    return cudaGetLastError();
}

// q NCHW int32 [B][C][HW] -> dst NHWC act_t [B][HW][C] = to_act(float(q) + mu), mu = mu_vec[c] or channel c of the NHWC
// act_t mu_act (ldc channels per pixel).  The same fp32 add and rounding as q.float() + mu on the NCHW fp32 mu, then
// launch_nchw_f32_to_nhwc_act; the 32 x 32 tile transposes as nchw_to_nhwc_kernel does.
__global__ void dequant_to_act_kernel(const int32_t* __restrict__ q, const float* __restrict__ mu_vec, const act_t* __restrict__ mu_act,
                                      int mu_ldc, act_t* __restrict__ dst, int C, int HW) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + threadIdx.x;
        tile[j][threadIdx.x] = (c < C && p < HW) ? static_cast<float>(q[(static_cast<size_t>(b) * C + c) * HW + p]) : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + threadIdx.x;
        if (p < HW && c < C) {
            const size_t px = static_cast<size_t>(b) * HW + p;
            const float m = mu_vec ? mu_vec[c] : from_act(mu_act[px * mu_ldc + c]);
            dst[px * C + c] = to_act(__fadd_rn(tile[threadIdx.x][j], m));
        }
    }
}
cudaError_t launch_dequant_to_act(const int32_t* q, const float* mu_vec, const act_t* mu_act, int mu_ldc, act_t* dst, int B, int C,
                                  int HW, cudaStream_t s) {
    if (!mu_vec == !mu_act) return cudaErrorInvalidValue;
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    dequant_to_act_kernel<<<grid, dim3(32, 8), 0, s>>>(q, mu_vec, mu_act, mu_ldc, dst, C, HW);
    return cudaGetLastError();
}

__global__ void nhwc_slice_to_nchw_kernel(const act_t* __restrict__ src, float* __restrict__ dst, int C, int HW, int ldc, int c_off,
                                          float min_clamp, int use_clamp) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z, c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int p = p0 + j, c = c0 + threadIdx.x;
        tile[j][threadIdx.x] = (c < C && p < HW) ? from_act(src[(static_cast<size_t>(b) * HW + p) * ldc + c_off + c]) : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += 8) {
        const int c = c0 + j, p = p0 + threadIdx.x;
        if (p < HW && c < C) {
            float v = tile[threadIdx.x][j];
            if (use_clamp) v = fmaxf(v, min_clamp);
            dst[(static_cast<size_t>(b) * C + c) * HW + p] = v;
        }
    }
}
cudaError_t launch_nhwc_slice_to_nchw_f32(const act_t* src, float* dst, int B, int C, int HW, int ldc, int c_off, float min_clamp,
                                          int use_clamp, cudaStream_t s) {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    nhwc_slice_to_nchw_kernel<<<grid, dim3(32, 8), 0, s>>>(src, dst, C, HW, ldc, c_off, min_clamp, use_clamp);
    return cudaGetLastError();
}

}  // namespace cdc
