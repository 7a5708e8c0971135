// Host runtime of the decode hot path: weight store, schedule, workspace arena, per-layer TMA
// tensor maps, the launch plan of one denoise step (and of the context net), CUDA-graph capture
// of the K-step loop, and the extern "C" ABI declared in include/cdc_b200.h.
//
// Oracle counterparts (the reference ships no code): oracle/unet.py UNet.forward,
// oracle/sampler.py make_schedule / denoise_step / decode, oracle/codec.py ContextNet.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/cdc_b200_tools.h"
#include "codec_io.cuh"
#include "conv_kf.cuh"
#include "conv_tc.cuh"
#include "kernels.cuh"

namespace cdc {

static std::string g_create_err;

// Planner decisions that tests / tools A/B through cdc_set_plan_option (include/cdc_b200_tools.h).
struct PlanOpts {
    int v[CDC_OPT_COUNT] = {2, 1, 0};
    int fuse_apply_max_tiles() const { return v[CDC_OPT_FUSE_APPLY]; }
    bool kf() const { return v[CDC_OPT_KF] != 0; }
    // SMs the plan lays its grids out for: the device's count unless CDC_OPT_PLAN_SMS asks for fewer
    int plan_sms(int device_sms) const { return v[CDC_OPT_PLAN_SMS] > 0 && v[CDC_OPT_PLAN_SMS] < device_sms ? v[CDC_OPT_PLAN_SMS] : device_sms; }
    // cdc_set_batch_invariant: every op is laid out per image as for a batch of 1 (strip lengths, walk direction, N tiles),
    // and the strip conv starts every strip at accumulator slot 0, so an image's bits do not depend on its batch
    bool batch_invariant = false;
    // the batch the geometry decisions are made for (the launch still covers all B images)
    int plan_batch(int B) const { return batch_invariant ? 1 : B; }
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

struct Act {  // NHWC act_t activation, batch implied by the plan
    act_t* p = nullptr;
    int C = 0, H = 0, W = 0;
    int Cphys = 0;  // channels actually stored per pixel (0: C).  The stem's x_t copy stores kXpadC of its 64 logical
                    // channels: tensor maps get this extent and pitch, TMA zero-fills the rest of the 64-channel box
    int cs() const { return Cphys ? Cphys : C; }
};

struct ConvW {  // repacked conv weights: act_t [n_pad][taps][c_pad], fp32 bias [n_pad]
    act_t* w = nullptr;
    float* bias = nullptr;
    int n_true = 0, n_pad = 0, taps = 0, c_pad = 0, c_true = 0;
    bool up2 = false;  // taps == 16: parity-specific pre-summed 2x2 weights for nearest-x2-input convs
    bool convt = false;  // taps == 36: ConvTranspose2d(5, stride 2) as four output-parity 3x3 convs (missing taps zero)
};

struct Op {
    std::string name;
    double flops = 0, bytes = 0;
    // (stream, sampler step k, timing slot or null): see ptx.cuh stamp_begin / stamp_end
    std::function<cudaError_t(cudaStream_t, int, long long*)> run;
    cdc_step_op_desc desc{};  // what the op computes and with which kernel (cdc_step_op_describe); never read by run
};

static cdc_tensor_desc tensor_desc(const Act& a) {
    cdc_tensor_desc d;
    d.p = a.p;
    d.C = a.C;
    d.Cphys = a.cs();
    d.H = a.H;
    d.W = a.W;
    return d;
}
static void set_desc_name(char (&dst)[64], const std::string& s) { snprintf(dst, sizeof dst, "%s", s.c_str()); }

// per-step sampler coefficients (host copies; oracle/sampler.py make_schedule)
struct SamplerTab {
    std::vector<float> c0, c1, e0, e1, sg;
    unsigned long long seed = 0;
};

enum ConvMode { MODE_S1 = 0, MODE_S2 = 1, MODE_UP2 = 2, MODE_CONVT = 3 };  // MODE_CONVT: ConvTranspose2d(5, 2, 2, 1), output 2H x 2W

static bool stats_inst_ok(int bn, int cpg) {
    return (bn == 64 && (cpg == 2 || cpg == 4 || cpg == 8)) || (bn == 128 && (cpg == 4 || cpg == 8)) ||
           (bn == 192 && cpg == 6) || (bn == 256 && cpg == 8);
}

struct Arena {
    std::vector<void*> ptrs;
    size_t total = 0;
    cudaError_t alloc(void** p, size_t bytes) {
        bytes = (bytes + 255) & ~size_t(255);
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) {
            ptrs.push_back(*p);
            total += bytes;
        }
        return e;
    }
    void release() {
        for (void* p : ptrs) cudaFree(p);
        ptrs.clear();
        total = 0;
    }
};

struct ConvBuild {
    std::string name;
    std::vector<Act> srcs;
    const ConvW* w = nullptr;
    int mode = MODE_S1;
    int ksize = 3;
    Act out;
    int epi = EPI_STORE;
    int cpg = 1;
    gn_sum_t* gn_acc = nullptr;  // EPI_STATS: this GroupNorm's accumulator slot [B][32][2]
    const act_t* residual = nullptr;
    int force_bn = 0;   // > 0: force the N tile of conv_tc.cu; -1: force conv_tc.cu with its own choice
    float act_slope = 0.0f;  // LeakyReLU slope applied after the bias (0 = none); general kernel only
    // DDIM
    float* x = nullptr;
    act_t* xpad = nullptr;
    float* x0_out = nullptr;
    const SamplerTab* samp = nullptr;  // per-step sampler coefficients (host)
    const unsigned long long* img_seeds = nullptr;  // per-image seed block (kernels.cuh), or null
    unsigned int* sat = nullptr;       // saturation diagnostics counter (device)
    // offered: fused 1x1 residual conv of the same input (kf path only; op->desc.res1 says whether it was taken)
    const ConvW* res_w = nullptr;
    Act res_out;
    bool x16 = false;          // source 0 carries at most 16 non-zero channels (the stem's x_t copy)
    // offered: input GroupNorm (+FiLM) + SiLU applied inside the conv (kf path only; op->desc.apply says whether it is
    // taken): the source is the RAW output of the preceding conv, in_acc that conv's statistics slot
    const gn_sum_t* in_acc = nullptr;
    const float* in_gamma = nullptr;
    const float* in_beta = nullptr;
    int in_film_off = -1;      // offset into the step's FiLM vector, or -1
    std::string in_gn;         // parameter prefix of that GroupNorm (op description only)
    float in_eps = 1e-5f;
    float* const* film_base = nullptr;  // -> ctx->film: [steps][*film_total] FiLM vectors of the schedule (set later)
    const int* film_total = nullptr;
};

// 16-bit tensor of `rank` dimensions (innermost first; byte_strides of dimensions 1 .. rank-1), 128-byte swizzle
static int encode_map(CUtensorMap* m, const act_t* base, int rank, const cuuint64_t* dims, const cuuint64_t* byte_strides,
                      const cuuint32_t* box) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return -1;
    const cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(m, CDC_TMA_DTYPE, rank, const_cast<act_t*>(base), dims, byte_strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

// An activation as a 4-D tensor {C, W, H, B}, box {64, BW, BH, 1}: every sx-th pixel of every sy-th row, starting at
// pixel (x0, y0); tr swaps image rows and columns ({C, H, W, B}).
static int encode_act_map(CUtensorMap* m, const Act& a, int B, int BW, int BH, int sx = 1, int sy = 1, int x0 = 0,
                          int y0 = 0, bool tr = false) {
    const cuuint64_t px = 2 * static_cast<cuuint64_t>(a.cs()), row = px * a.W;
    cuuint64_t dims[4] = {static_cast<cuuint64_t>(a.cs()), static_cast<cuuint64_t>(a.W / sx),
                          static_cast<cuuint64_t>(a.H / sy), static_cast<cuuint64_t>(B)};
    cuuint64_t strides[3] = {px * sx, row * sy, row * a.H};
    if (tr) {
        std::swap(dims[1], dims[2]);
        std::swap(strides[0], strides[1]);
    }
    const cuuint32_t box[4] = {64, static_cast<cuuint32_t>(BW), static_cast<cuuint32_t>(BH), 1};
    return encode_map(m, a.p + (static_cast<size_t>(y0) * a.W + x0) * a.cs(), 4, dims, strides, box);
}

// qkv [B][N][cols] viewed as a 3-D tensor {cols, N, B}, box {64, 128, 1}: one head's Q / K / V slice of 128 tokens
static int encode_qkv_map(CUtensorMap* m, const act_t* qkv, int cols, int N, int B) {
    const cuuint64_t dims[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(B)};
    const cuuint64_t strides[2] = {static_cast<cuuint64_t>(cols) * 2, static_cast<cuuint64_t>(N) * cols * 2};
    const cuuint32_t box[3] = {64, 128, 1};
    return encode_map(m, qkv, 3, dims, strides, box);
}

// repacked weights as the [n_pad][taps * c_pad] K-major matrix, box {64, BN}
static int encode_w_map(CUtensorMap* m, const ConvW& w, int BN) {
    const cuuint64_t K = static_cast<cuuint64_t>(w.taps) * w.c_pad;
    const cuuint64_t dims[2] = {K, static_cast<cuuint64_t>(w.n_pad)};
    const cuuint64_t strides[1] = {K * 2};
    const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(BN)};
    return encode_map(m, w.w, 2, dims, strides, box);
}


// ---- kh-fused strip variant (conv_kf.cu): 3x3, stride 1, resident weights, N tiles of 64 (16 for the final conv) ----
struct KfGeom {
    int bn, CH, n_tiles, nseg, S, G1, NS, mode;
    bool staged, res;
    bool apply;  // the input GroupNorm + SiLU runs inside the kernel
    bool tr;  // transposed walk: strips run along image columns (less padding / halo for e.g. a 128 x 192 level)
};
static bool conv_uses_kf(const ConvBuild& cb, int B, int num_sms, const PlanOpts& po, KfGeom* g) {
    if (!po.kf() || cb.ksize != 3 || cb.force_bn != 0 || cb.residual || cb.act_slope != 0.0f || cb.mode == MODE_CONVT) return false;
    g->mode = cb.mode == MODE_UP2 ? 1 : cb.mode == MODE_S2 ? 2 : 0;
    if (g->mode == 1 && (!cb.w->up2 || cb.epi != EPI_STORE)) return false;
    if (g->mode == 2 && (cb.epi != EPI_STORE || cb.res_w || cb.in_acc || ((cb.srcs[0].W | cb.srcs[0].H) & 1))) return false;
    // (only the 64- and 128-channel downsampling convs have stride-2 kf instantiations: with 32-channel N tiles (192 / 256
    // channels, 64x96 outputs and below) the strip form measured 3 us per step SLOWER than the general kernel)
    // strip geometry lives on the grid the kernel walks: the input grid (mode 1 writes 2x2 outputs per pixel), for the
    // stride-2 mode the OUTPUT grid
    int gw = cb.srcs[0].W >> (g->mode == 2 ? 1 : 0), gh = cb.srcs[0].H >> (g->mode == 2 ? 1 : 0);
    g->tr = false;
    g->nseg = (gw + 127) / 128;
    // segments are 128 pixels wide: too much of the tile would be padding (measured break-even against conv_tc.cu:
    // 3x3 convs down to 48 of 128 columns; the upsampling convs need 96)
    const bool wide_ok = gw * 100 >= g->nseg * 128 * (cb.mode == MODE_UP2 ? 50 : 35);
    const bool tall_ok = cb.mode == MODE_S1 && cb.epi != EPI_DDIM && gh * 100 >= ((gh + 127) / 128) * 128 * 35;
    if (!wide_ok && !tall_ok) return false;
    int ctot = 0;
    for (const Act& a : cb.srcs) ctot += a.C;
    g->CH = ctot / 64;
    // largest N tile whose whole weight block stays resident in shared memory (and holds whole GroupNorm groups)
    g->bn = 0;
    const int cands[3] = {64, 48, 32};
    for (int c : cands) {
        const int bn = cb.epi == EPI_DDIM ? 16 : c;
        if (cb.w->n_pad % bn || (cb.epi == EPI_STATS && bn % cb.cpg)) continue;
        // with the ResBlock's 1x1 residual conv riding along when that fits, else without
        g->res = cb.res_w != nullptr && g->mode == 0 && cb.res_w->n_pad == cb.w->n_pad && cb.res_w->taps == 1 &&
                 cb.res_w->c_pad == ctot && kf_inst_ok(bn, cb.cpg, cb.epi, g->CH, g->mode, true) &&
                 kf_plan(bn, g->CH, g->mode, true, &g->NS, &g->staged);
        if (!g->res && (!kf_inst_ok(bn, cb.cpg, cb.epi, g->CH, g->mode, false) ||
                        !kf_plan(bn, g->CH, g->mode, false, &g->NS, &g->staged)))
            continue;
        g->bn = bn;
        break;
    }
    if (!g->bn) return false;
    // (every N tile's CTAs transform the same rows: levels 0 and 1 -- one and two N tiles, instantiated for 64 and 128
    // channels -- gain 2.4 % and 0.8 % images/s; with 3+ tiles the redundant MUFU work costs more than the pass it replaces)
    g->apply = cb.in_acc != nullptr && !g->res && cb.srcs.size() == 1 && cb.cpg == g->CH * 2 &&
               cb.w->n_pad / g->bn <= po.fuse_apply_max_tiles() &&
               kf_inst_ok(g->bn, cb.cpg, cb.epi, g->CH, g->mode, false, true);
    g->n_tiles = cb.w->n_pad / g->bn * (g->mode == 1 ? 4 : 1);
    if (cb.epi == EPI_DDIM && g->n_tiles != 1) return false;
    // strip geometry for a walk along image rows (tr = 0) or image columns (tr = 1): relative cost = padding of the
    // 128-pixel segments x halo rows per strip; the transposed walk is used for unstaged kernels when it is >10 % cheaper
    // (S is chosen for the plan batch; with a plan batch of 1 and B > 1 a CTA runs several strips, of any images)
    auto plan = [&](int w_, int h_, int* nseg, int* S, int* G1) {
        *nseg = (w_ + 127) / 128;
        const int cols = po.plan_batch(B) * *nseg;  // independent strip columns per N tile
        int g1 = num_sms / g->n_tiles;
        if (g1 < 1) g1 = 1;
        int s_ = g1 / cols;
        if (s_ < 1) s_ = 1;
        if (s_ > h_) s_ = h_;
        *S = s_;
        const int units = B * *nseg * s_;
        *G1 = units < g1 ? units : g1;
        const double L = static_cast<double>(h_) / s_;
        return (*nseg * 128.0 / w_) * (L + 2.0) / L;
    };
    int nsegT, ST, G1T;
    const double c0 = wide_ok ? plan(gw, gh, &g->nseg, &g->S, &g->G1) : 1e30;
    const double c1 = (tall_ok && !g->staged && g->mode == 0) ? plan(gh, gw, &nsegT, &ST, &G1T) : 1e30;
    if (c1 < 0.9 * c0) {
        g->tr = true;
        g->nseg = nsegT;
        g->S = ST;
        g->G1 = G1T;
    } else if (!wide_ok) {
        return false;
    }
    return true;
}

// This step's sampler coefficients into the params block of either conv kernel (KfParams, ConvParams); false when k is
// outside the schedule.
template <class P>
static bool set_sampler_step(P* q, const SamplerTab* samp, int k) {
    if (!samp || k < 0 || k >= static_cast<int>(samp->c0.size())) return false;
    q->c0 = samp->c0[k];
    q->c1 = samp->c1[k];
    q->e0 = samp->e0[k];
    q->e1 = samp->e1[k];
    q->sg = samp->sg[k];
    q->seed = samp->seed;
    q->step = k;
    return true;
}

// What a kf op's run needs besides its params block: the instantiation, and where the per-step inputs come from.
struct KfLaunch {
    int bn, cpg, epi, ch, mode;
    bool xk16, res, apply, staged;
    const SamplerTab* samp;   // EPI_DDIM
    float* const* film_base;  // input GroupNorm with FiLM: ConvBuild::film_base / film_total / in_film_off
    const int* film_total;
    int film_off;
};

// The kh-fused strip kernel (conv_kf.cu) in geometry kg.  Returns an error message, or null.
static const char* plan_conv_kf(const ConvBuild& cb, const KfGeom& kg, int B, const PlanOpts& po, int gw, int gh, Op* op) {
    const ConvW& w = *cb.w;
    auto kp = std::shared_ptr<KfParams>(new KfParams());
    memset(kp.get(), 0, sizeof(KfParams));
    for (size_t s = 0; s < cb.srcs.size(); ++s) {
        const Act& a = cb.srcs[s];
        if (kg.mode == 2) {  // even-pixel and odd-pixel views of the source: pixel stride 2, W/2 pixels each
            for (int eo = 0; eo < 2; ++eo)
                if (encode_act_map(&kp->amap[2 * s + eo], a, B, 130, 1, 2, 1, eo))
                    return "cuTensorMapEncodeTiled (kf stride-2 activation) failed";
        } else if (encode_act_map(&kp->amap[s], a, B, 130, 1, 1, 1, 0, 0, kg.tr)) {
            return "cuTensorMapEncodeTiled (kf activation) failed";
        }
    }
    if (encode_w_map(&kp->wmap, w, kg.bn)) return "cuTensorMapEncodeTiled (weights) failed";
    if (kg.res) {
        if (encode_w_map(&kp->rmap, *cb.res_w, kg.bn)) return "cuTensorMapEncodeTiled (residual-conv weights) failed";
        kp->res_out = cb.res_out.p;
        kp->res_ldc = cb.res_out.C;
        kp->res_bias = cb.res_w->bias;
    }
    if (kg.staged && encode_act_map(&kp->omap, cb.out, B, 128, 1)) return "cuTensorMapEncodeTiled (kf output) failed";
    kp->chunks0 = cb.srcs[0].C / 64;
    kp->tr = kg.tr ? 1 : 0;
    kp->H = kg.tr ? gw : gh;  // kernel-space rows / pixels per row
    kp->W = kg.tr ? gh : gw;
    kp->batch = B;
    kp->nseg = kg.nseg;
    kp->S = kg.S;
    kp->slot0 = po.batch_invariant ? 1 : 0;
    kp->NS = kg.NS;
    kp->n_tiles = kg.n_tiles;
    kp->G1 = kg.G1;
    kp->ldc = cb.epi == EPI_DDIM ? 3 : cb.out.C;
    kp->out = cb.out.p;
    kp->bias = w.bias;
    kp->gn_acc = cb.gn_acc;
    if (kg.apply) {
        kp->in_acc = cb.in_acc;
        kp->in_gamma = cb.in_gamma;
        kp->in_beta = cb.in_beta;
        kp->in_eps = cb.in_eps;
    }
    kp->x = cb.x;
    kp->xpad = cb.xpad;
    kp->x0_out = cb.x0_out;
    kp->img_seeds = cb.img_seeds;
    kp->sat = cb.sat;
    kp->e1 = 1.0f;
    if (kg.apply) op->name += "+gn_in";  // the GroupNorm apply pass no longer touches HBM; its arithmetic rides along
    if (kg.res) {  // the 1x1 residual conv's algorithmic work moves into this launch
        const double Ms = static_cast<double>(B) * gh * gw;
        op->flops += 2.0 * Ms * cb.res_w->n_true * cb.res_w->c_true;
        op->bytes += 2.0 * (Ms * cb.res_w->n_true + static_cast<double>(cb.res_w->c_true) * cb.res_w->n_true);
        op->name += "+res";
    }
    const bool xk16 = cb.x16 && cb.epi == EPI_STORE && kg.bn == 64 && kg.CH == 2 && cb.srcs[0].C == 64 && kg.mode == 0;
    const KfLaunch L{kg.bn, cb.cpg, cb.epi, kg.CH, kg.mode, xk16, kg.res, kg.apply, kg.staged,
                     cb.samp, cb.film_base, cb.film_total, cb.in_film_off};
    cdc_step_op_desc& d = op->desc;
    d.kernel = 2;
    d.bn = kg.bn;
    d.staged = kg.staged;
    d.xk16 = xk16;
    d.tr = kg.tr;
    d.res1 = kg.res;
    d.apply = kg.apply;
    d.n_tiles = kg.n_tiles;
    d.g1 = kg.G1;
    d.nseg = kg.nseg;
    d.strips = kg.S;
    d.rows = kp->H;
    d.grid = kg.n_tiles * kg.G1;
    if (kg.res) d.res_out = tensor_desc(cb.res_out);
    if (kg.apply) {
        d.gn_in_acc = const_cast<gn_sum_t*>(cb.in_acc);
        d.film_off = cb.in_film_off;
        set_desc_name(d.in_gn, cb.in_gn);
    }
    op->run = [kp, L](cudaStream_t s, int k, long long* stamp) -> cudaError_t {
        KfParams q = *kp;
        q.stamp = stamp;
        if (L.epi == EPI_DDIM && !set_sampler_step(&q, L.samp, k)) return cudaErrorInvalidValue;
        if (L.apply && L.film_off >= 0)  // this step's FiLM (scale | shift) of the input GroupNorm
            q.in_film = *L.film_base + static_cast<size_t>(k) * *L.film_total + L.film_off;
        return launch_conv_kf(q, L.bn, L.cpg, L.epi, L.ch, L.xk16, L.mode, L.res, L.apply, L.staged, s);
    };
    return nullptr;
}

// The general implicit-GEMM kernel (conv_tc.cu).  Returns an error message, or null.
static const char* plan_conv_tc(const ConvBuild& cb, int B, int num_sms, const PlanOpts& po, int gw, int gh, Op* op) {
    const ConvW& w = *cb.w;
    const int ctot = w.c_pad;
    const bool x2 = cb.mode == MODE_UP2 || cb.mode == MODE_CONVT;  // four output phases, each on the input grid
    const int nphase = x2 ? 4 : 1, os = x2 ? 2 : 1;
    // tile of (128 >> bwl) rows x (1 << bwl) columns: the shape that needs the fewest tiles
    int bwl = 7;
    long best_tiles = -1;
    for (int l = 7; l >= 2; --l) {
        const int BW = 1 << l, BH = 128 >> l;
        const long t = static_cast<long>((gw + BW - 1) / BW) * ((gh + BH - 1) / BH);
        if (best_tiles < 0 || t < best_tiles) {
            best_tiles = t;
            bwl = l;
        }
    }
    const int BW = 1 << bwl, BH = 128 >> bwl;
    const int tiles_w = (gw + BW - 1) / BW, tiles_h = (gh + BH - 1) / BH;

    // N tile (chosen for the plan batch; the grid covers all B images)
    const long m_tiles = static_cast<long>(nphase) * B * tiles_w * tiles_h;
    const long m_tiles_plan = static_cast<long>(nphase) * po.plan_batch(B) * tiles_w * tiles_h;
    int bn = 0;
    if (cb.epi == EPI_DDIM) {
        bn = 16;
    } else if (cb.force_bn > 0) {
        bn = cb.force_bn;
    } else {
        // Cost model from the round-1 per-layer measurements: a CTA ingests ~33 B/cycle from L2 through
        // TMA when all SMs stream, a K-block costs max(MMA cycles, bytes / 33), and whole waves count.
        const int cands[4] = {256, 192, 128, 64};
        double best = 0;
        for (int c : cands) {
            if (w.n_pad % c) continue;
            if (cb.epi == EPI_STATS && !stats_inst_ok(c, cb.cpg)) continue;
            const long tiles = m_tiles_plan * (w.n_pad / c);
            const long waves = (tiles + num_sms - 1) / num_sms;
            const double mma = 4.0 * (c / 2.0), mem = (16384.0 + c * 128.0) / 33.0;
            const double cost = static_cast<double>(waves) * (mma > mem ? mma : mem);
            if (!bn || cost < best) {
                bn = c;
                best = cost;
            }
        }
    }
    if (!bn || w.n_pad % bn) return "no N tile for C_out";
    if (w.n_pad > 768) return "C_out beyond the general kernel's 768-entry bias table";
    if (cb.epi == EPI_STATS && !stats_inst_ok(bn, cb.cpg)) return "no stats instantiation for (BN, cpg)";

    // tensor maps
    auto cp = std::shared_ptr<ConvParams>(new ConvParams());
    memset(cp.get(), 0, sizeof(ConvParams));
    int nmaps = 0;
    for (const Act& a : cb.srcs) {
        if (cb.mode == MODE_S2) {  // the four (row, column) parity views of the source: pixel stride 2 both ways
            for (int py = 0; py < 2; ++py)
                for (int px = 0; px < 2; ++px)
                    if (encode_act_map(&cp->amap[nmaps++], a, B, BW, BH, 2, 2, px, py))
                        return "cuTensorMapEncodeTiled (stride-2 view) failed";
        } else if (encode_act_map(&cp->amap[nmaps++], a, B, BW, BH)) {
            return "cuTensorMapEncodeTiled (activation) failed";
        }
    }
    if (encode_w_map(&cp->wmap, w, bn)) return "cuTensorMapEncodeTiled (weights) failed";

    // K-block table: for every output phase, the taps {row / column shift, phase view, weight tap} in K order, each
    // split into the 64-channel chunks of every source
    const int ntap = w.convt ? 9 : w.up2 ? 4 : cb.ksize * cb.ksize;  // taps per output phase
    const int nkb = ntap * (ctot / 64);
    if (nkb * nphase > kMaxKBlocks) return "K-block table overflow";
    const int pad = cb.ksize / 2;
    KBlock* e = cp->kb;
    for (int ph = 0; ph < nphase; ++ph) {
        const int py = ph >> 1, px = ph & 1;
        for (int t = 0; t < ntap; ++t) {
            int dh, dw, msel = 0, wt;  // wt: the tap's ctot-wide slice of a weight row
            if (w.convt) {  // transposed conv: 3x3 taps (a, b) per output parity (zero weights where the parity has two),
                            // row offset 1 - a, column offset 1 - b
                dh = 1 - t / 3;
                dw = 1 - t % 3;
                wt = ph * 9 + t;
            } else if (w.up2) {  // pre-summed parity weights: 2x2 taps (a, b), K index = ((ph*4 + a*2 + b) * ctot + channel)
                dh = t / 2 - (py == 0);
                dw = t % 2 - (px == 0);
                wt = ph * 4 + t;
            } else {
                dh = t / cb.ksize - pad;
                dw = t % cb.ksize - pad;
                wt = t;
                if (cb.mode == MODE_S2) {  // the parity of the source row / column picks one of the four phase views
                    const int qy = dh & 1, qx = dw & 1;
                    msel = qy * 2 + qx;
                    dh = (dh - qy) / 2;
                    dw = (dw - qx) / 2;
                }
            }
            int soff = 0;
            for (size_t s = 0; s < cb.srcs.size(); ++s) {
                for (int c = 0; c < cb.srcs[s].C; c += 64)
                    *e++ = KBlock{static_cast<int8_t>(s * (cb.mode == MODE_S2 ? 4 : 1) + msel), static_cast<int8_t>(dw),
                                  static_cast<int8_t>(dh), 0, static_cast<uint16_t>(c),
                                  static_cast<uint16_t>(wt * ctot + soff + c)};
                soff += cb.srcs[s].C;
            }
        }
    }
    cp->nkb = nkb;
    cp->nphase = nphase;
    cp->tiles_w = tiles_w;
    cp->tiles_h = tiles_h;
    cp->batch = B;
    cp->bw_log2 = bwl;
    cp->gw = gw;
    cp->gh = gh;
    cp->OH = gh * os;
    cp->OW = gw * os;
    cp->os = os;
    cp->ldc = cb.epi == EPI_DDIM ? 3 : cb.out.C;
    cp->n_total = w.n_pad;
    cp->n_tiles = w.n_pad / bn;
    cp->out = cb.out.p;
    cp->bias = w.bias;
    cp->residual = cb.residual;
    cp->gn_acc = cb.gn_acc;
    cp->x = cb.x;
    cp->xpad = cb.xpad;
    cp->x0_out = cb.x0_out;
    cp->img_seeds = cb.img_seeds;
    cp->sat = cb.sat;
    cp->e1 = 1.0f;
    cp->act_slope = cb.act_slope;

    const int epi = cb.epi, cpg = cb.cpg;
    const SamplerTab* samp = cb.samp;
    op->desc.kernel = 1;
    op->desc.bn = bn;
    const long total = m_tiles * (w.n_pad / bn);  // (launch_conv's grid: conv_tc.cu launch_one)
    op->desc.n_tiles = static_cast<int>(total);
    op->desc.grid = static_cast<int>(total < num_sms ? total : num_sms);
    op->run = [cp, bn, cpg, epi, num_sms, samp](cudaStream_t s, int k, long long* stamp) -> cudaError_t {
        ConvParams q = *cp;
        q.stamp = stamp;
        if (epi == EPI_DDIM && !set_sampler_step(&q, samp, k)) return cudaErrorInvalidValue;
        return launch_conv(q, bn, cpg, epi, num_sms, s);
    };
    return nullptr;
}

// Builds the op of one conv: the kh-fused strip kernel when it can run the conv, with those of the offered fusions it
// takes (op->desc.res1: the 1x1 residual conv, op->desc.apply: the input GroupNorm), else the general kernel, which
// takes neither.
static int build_conv(const ConvBuild& cb, int B, int num_sms, const PlanOpts& po, Op* op, std::string* err) {
    auto fail = [&](const std::string& m) {
        *err = "conv " + cb.name + ": " + m;
        return CDC_ERR_SHAPE;
    };
    if (cb.srcs.empty() || cb.srcs.size() > 2) return fail("1 or 2 sources required");
    int ctot = 0;
    for (const Act& a : cb.srcs) {
        if (a.C % 64) return fail("source channels must be a multiple of 64");
        if (a.H != cb.srcs[0].H || a.W != cb.srcs[0].W) return fail("sources differ in size");
        ctot += a.C;
    }
    const ConvW& w = *cb.w;
    const int taps = cb.ksize * cb.ksize;
    // (nearest-x2 convs run on pre-summed parity weights, which are repacked from 3x3 weights only)
    if (ctot != w.c_pad || (w.convt ? (cb.mode != MODE_CONVT || cb.ksize != 5)
                            : w.up2  ? (cb.mode != MODE_UP2 || cb.ksize != 3)
                                     : (taps != w.taps || cb.mode == MODE_UP2 || cb.mode == MODE_CONVT)))
        return fail("weight layout does not match the sources");
    const Act& in = cb.srcs[0];
    if (cb.mode == MODE_S2 && ((in.W | in.H) & 1)) return fail("stride 2 needs even H, W");
    // the grid the kernels walk: the output grid of a stride-2 conv, else the input grid (2x2 outputs per pixel when
    // upsampling)
    const int gw = cb.mode == MODE_S2 ? in.W / 2 : in.W, gh = cb.mode == MODE_S2 ? in.H / 2 : in.H;
    const bool x2 = cb.mode == MODE_UP2 || cb.mode == MODE_CONVT;
    const int OH = x2 ? 2 * gh : gh, OW = x2 ? 2 * gw : gw;
    if (cb.epi != EPI_DDIM && (cb.out.H != OH || cb.out.W != OW || cb.out.C != w.n_pad))
        return fail("output tensor shape mismatch");
    cdc_step_op_desc& d = op->desc;
    d = cdc_step_op_desc{};
    d.kind = CDC_OPK_CONV;
    d.film_off = -1;
    d.mode = cb.mode;
    d.ksize = cb.ksize;
    d.epi = cb.epi;
    d.cpg = cb.cpg;
    d.ch = ctot / 64;
    for (size_t s = 0; s < cb.srcs.size(); ++s) d.src[s] = tensor_desc(cb.srcs[s]);
    d.out = tensor_desc(cb.out);
    if (cb.residual) {
        d.residual = d.out;
        d.residual.p = const_cast<act_t*>(cb.residual);
    }
    d.gn_out_acc = cb.gn_acc;
    d.act_slope = cb.act_slope;
    d.x = cb.x;
    d.x0_out = cb.x0_out;
    d.xpad = cb.xpad;
    op->name = cb.name;
    const double m_in = static_cast<double>(B) * in.H * in.W, M = static_cast<double>(B) * OH * OW;
    op->flops = w.convt ? 2.0 * m_in * w.n_true * (25.0 * w.c_true)  // every input pixel meets every tap once
                        : 2.0 * M * w.n_true * (static_cast<double>(taps) * w.c_true);
    op->bytes = 2.0 * (m_in * w.c_true + M * w.n_true + static_cast<double>(taps) * w.c_true * w.n_true);
    KfGeom kg;
    const char* m = conv_uses_kf(cb, B, num_sms, po, &kg) ? plan_conv_kf(cb, kg, B, po, gw, gh, op)
                                                          : plan_conv_tc(cb, B, num_sms, po, gw, gh, op);
    return m ? fail(m) : CDC_OK;
}

}  // namespace cdc

using namespace cdc;

struct WeightT {
    float* p = nullptr;
    std::vector<int64_t> shape;
    size_t numel = 0;
};

constexpr int kMaxGnSlots = 64;  // GroupNorms per sequence (37 in a denoise step, 8 in the context net)
// Largest batch a plan can run: gn_apply_kernel keeps every image's 32 (mean, rstd) float2 pairs in dynamic shared
// memory without the opt-in beyond 48 KB (launch_gn_apply refuses more).  Nothing else limits the batch below this.
constexpr int kMaxBatch = 48 * 1024 / (32 * 8);

struct Seq {  // one op sequence of the plan
    std::vector<Op> ops;
    gn_sum_t* slots = nullptr;  // its GroupNorms' accumulator slots [kMaxGnSlots][B][32][kGnVals], or null: none
    int gn_used = 0;            // slots in use (the sequence's first op clears them)
};

struct cdc_ctx {
    cdc_config cfg;
    int device = 0, num_sms = 148;
    std::string err;
    std::map<std::string, WeightT> w;
    std::map<std::string, ConvW> convs;
    Arena warena;  // weights
    bool finalized = false, has_ctx = false, has_codec = false;
    int C[4];

    PlanOpts opts;
    bool opts_dirty = false;  // an option changed since the plan was built: the next cdc_bind_io re-plans

    // schedule
    int K = 0;
    std::vector<int> idx;
    SamplerTab samp;         // c0, c1, e0, e1, sigma per step
    int pred_eps = 0;        // cdc_set_sampler: 0 = the network predicts x0, 1 = it predicts the noise
    float eta = 0.0f;
    unsigned long long seed = 0;
    float* film = nullptr;   // [K][film_total]
    float* sinus = nullptr;  // [K][64]
    int film_total = 0;
    std::vector<int> film_off;  // per RB

    // plan
    Arena arena;
    int B = 0, H = 0, W = 0;
    Seq step_seq, ctx_seq;
    // codec side (SURVEY.md section 8 row f2; oracle/codec.py Encoder / HyperEncoder / HyperDecoder), present when the
    // "codec.*" weights were loaded: analysis encoder, hyper-encoder, hyper-decoder -- three more op sequences
    Seq enc_seq, henc_seq, hdec_seq;
    Act img64, enc_y, henc_in, henc_z, hdec_in, hdec_out;
    Act cond[4], xpad, latent;
    float *xs = nullptr, *x0s = nullptr;
    // cdc_set_image_seeds: the seed block the final conv's epilogue and init_noise read ([1 + B], kernels.cuh), whether
    // per-image mode is on, and the end of the most recent launch that reads the block (it may be rewritten after it)
    unsigned long long* img_seeds = nullptr;
    bool seeded = false;
    cudaEvent_t seeds_done = nullptr;
    gn_sum_t* gn_slots = nullptr;  // [3][kMaxGnSlots][B][32][kGnVals] fixed-point GroupNorm accumulators (gn_sums.cuh)
    unsigned int* sat_dev = nullptr;  // saturation diagnostics counter (cdc_saturation_count)
    float *stage_f32 = nullptr;  // NCHW fp32 staging for host-buffer calls
    size_t stage_elems = 0;
    float *pin_in = nullptr, *pin_x = nullptr, *pin_out = nullptr;
    size_t pin_nl = 0, pin_nx = 0;  // elements the pinned staging buffers hold
    cudaStream_t copy_stream = nullptr;  // cdc_decode_host: x_T upload overlaps the context net
    cudaEvent_t ev_x = nullptr, ev_fork = nullptr;
    cudaGraphExec_t graph = nullptr;
    int graph_K = 0;
    int graph_skip = 0;  // tools build only (cdc_debug_graph_skip): class of ops left out of the captured graph
    cudaStream_t cap_stream = nullptr;
    // cdc_decode_trajectory: a second graph, the K-step loop plus trajectory store nodes and one event-record node per slot
    cudaGraphExec_t traj_graph = nullptr;
    int traj_K = 0, traj_every = 0;
    std::vector<cudaEvent_t> traj_ev;  // [slots]: slot j of the most recent launch is written
    int traj_issued = 0;               // slots of the most recent launch of traj_graph (0: none since it was built)
    TrajPtrs* traj_ptrs = nullptr;     // device block the store nodes read the caller's buffers from
    cudaEvent_t traj_done = nullptr;   // end of the most recent launch: traj_ptrs may be rewritten after it
    ByteCodec* byte_codec = nullptr;   // cdc_compress_rgb8 / cdc_decompress_rgb8 (bitstream.cu); null until first used

    int fail(int code, const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        err = buf;
        return code;
    }
};

#define CK(expr)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (expr);                                                              \
        if (e_ != cudaSuccess) return ctx->fail(CDC_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

static cudaStream_t S(cdc_stream s) { return reinterpret_cast<cudaStream_t>(s); }

// ------------------------------------------------------------------------------------------------ weights
static const WeightT* find_w(cdc_ctx* ctx, const std::string& name) {
    auto it = ctx->w.find(name);
    return it == ctx->w.end() ? nullptr : &it->second;
}

// Repack "<pfx>.weight"/".bias" (OIHW fp32) to the K-conv layout.  `split`/`split_pad`: input channels
// >= split start at slot split_pad (stem: 3 image channels padded to 64, then the 64 context channels).
static int make_conv_w(cdc_ctx* ctx, Arena& ar, const float* wsrc, const float* bsrc, int O, int I, int ks, int split,
                       int split_pad, bool is_final, ConvW* out, cudaStream_t s, bool up2 = false, bool convt = false) {
    const int taps = convt ? 36 : up2 ? 16 : ks * ks;
    const int c_pad = (split < I && split_pad > split) ? split_pad + ((I - split + 63) / 64) * 64 : ((I + 63) / 64) * 64;
    const int n_pad = is_final ? 16 : ((O + 63) / 64) * 64;
    ConvW cw;
    cw.n_true = O;
    cw.n_pad = n_pad;
    cw.taps = taps;
    cw.c_pad = c_pad;
    cw.c_true = I;
    CK(ar.alloc(reinterpret_cast<void**>(&cw.w), static_cast<size_t>(n_pad) * taps * c_pad * 2));
    CK(ar.alloc(reinterpret_cast<void**>(&cw.bias), static_cast<size_t>(n_pad) * 4));
    CK(cudaMemsetAsync(cw.bias, 0, static_cast<size_t>(n_pad) * 4, s));
    CK(cudaMemcpyAsync(cw.bias, bsrc, static_cast<size_t>(O) * 4, cudaMemcpyDeviceToDevice, s));
    const int sp = (split < I && split_pad > split) ? split : I;
    const int spp = (split < I && split_pad > split) ? split_pad : I;
    cw.up2 = up2;
    cw.convt = convt;
    if (convt)
        CK(launch_repack_weight_convt5(wsrc, cw.w, O, I, n_pad, c_pad, s));
    else if (up2)
        CK(launch_repack_weight_up2(wsrc, cw.w, O, I, n_pad, c_pad, s));
    else
        CK(launch_repack_weight(wsrc, cw.w, O, I, taps, n_pad, c_pad, sp, spp, s));
    *out = cw;
    return CDC_OK;
}

static int conv_from_store(cdc_ctx* ctx, const std::string& pfx, int O, int I, int ks, int split, int split_pad,
                           bool is_final, bool up2 = false, bool convt = false) {
    const WeightT* w = find_w(ctx, pfx + ".weight");
    const WeightT* b = find_w(ctx, pfx + ".bias");
    if (!w || !b) return ctx->fail(CDC_ERR_WEIGHT, "missing weight tensor %s.weight/.bias", pfx.c_str());
    // (ConvTranspose2d keeps its weight as [in, out, k, k])
    if (w->shape.size() != 4 || w->shape[0] != (convt ? I : O) || w->shape[1] != (convt ? O : I) || w->shape[2] != ks || w->shape[3] != ks ||
        b->numel != static_cast<size_t>(O))
        return ctx->fail(CDC_ERR_WEIGHT, "%s: expected %s weight [%d,%d,%d,%d]", pfx.c_str(), convt ? "transposed-conv" : "conv",
                         convt ? I : O, convt ? O : I, ks, ks);
    ConvW cw;
    int r = make_conv_w(ctx, ctx->warena, w->p, b->p, O, I, ks, split, split_pad, is_final, &cw, nullptr, up2, convt);
    if (r) return r;
    ctx->convs[pfx] = cw;
    return CDC_OK;
}

static int need_vec(cdc_ctx* ctx, const std::string& name, size_t n) {
    const WeightT* w = find_w(ctx, name);
    if (!w) return ctx->fail(CDC_ERR_WEIGHT, "missing weight tensor %s", name.c_str());
    if (w->numel != n) return ctx->fail(CDC_ERR_WEIGHT, "%s: expected %zu elements, got %zu", name.c_str(), n, w->numel);
    return CDC_OK;
}

static int rb_weights(cdc_ctx* ctx, const std::string& pfx, int cin, int cout, bool film) {
    int r;
    if ((r = conv_from_store(ctx, pfx + ".conv1", cout, cin, 3, cin, cin, false))) return r;
    if ((r = conv_from_store(ctx, pfx + ".conv2", cout, cout, 3, cout, cout, false))) return r;
    if (cin != cout && (r = conv_from_store(ctx, pfx + ".res", cout, cin, 1, cin, cin, false))) return r;
    for (const char* g : {".gn1", ".gn2"}) {
        if ((r = need_vec(ctx, pfx + g + ".weight", cout))) return r;
        if ((r = need_vec(ctx, pfx + g + ".bias", cout))) return r;
    }
    if (film) {
        if ((r = need_vec(ctx, pfx + ".film.weight", static_cast<size_t>(2) * cout * ctx->cfg.temb))) return r;
        if ((r = need_vec(ctx, pfx + ".film.bias", static_cast<size_t>(2) * cout))) return r;
    }
    return CDC_OK;
}

static std::vector<std::string> film_rb_names(cdc_ctx* ctx, std::vector<int>* couts) {
    std::vector<std::string> n;
    for (int i = 0; i < 4; ++i)
        for (const char* rb : {".rb1", ".rb2"}) {
            n.push_back("down." + std::to_string(i) + rb);
            couts->push_back(ctx->C[i]);
        }
    for (const char* rb : {"mid.rb1", "mid.rb2"}) {
        n.push_back(rb);
        couts->push_back(ctx->C[3]);
    }
    for (int i = 3; i >= 0; --i)
        for (const char* rb : {".rb1", ".rb2"}) {
            n.push_back("up." + std::to_string(i) + rb);
            couts->push_back(ctx->C[i]);
        }
    return n;
}

// ------------------------------------------------------------------------------------------------ plan
struct PlanB {
    cdc_ctx* ctx;
    Seq& seq;
    std::map<std::string, Act> tmp;  // per-shape temporaries shared by the ResBlocks of a level
    int rc = CDC_OK;

    // Every GroupNorm of a sequence gets its own accumulator slot; one memset, the first op of the sequence, clears the
    // slots in use (read when it runs: the sequence is complete by then).
    PlanB(cdc_ctx* c, Seq& s) : ctx(c), seq(s) {
        if (!seq.slots) return;
        Op z;
        z.name = "gn.clear";
        gn_sum_t* base = seq.slots;
        const int* used = &seq.gn_used;
        z.run = [c, base, used](cudaStream_t st, int, long long*) {
            return cudaMemsetAsync(base, 0, static_cast<size_t>(*used) * c->B * kGnImgStride * sizeof(gn_sum_t), st);
        };
        z.desc.kind = CDC_OPK_MEMSET;
        z.desc.film_off = -1;
        z.desc.gn_out_acc = base;  // (gn_slots: filled in when described)
        seq.ops.push_back(z);
    }
    Act act(int C, int H, int W) {
        Act a;
        a.C = C;
        a.H = H;
        a.W = W;
        if (cudaSuccess != ctx->arena.alloc(reinterpret_cast<void**>(&a.p), static_cast<size_t>(ctx->B) * H * W * C * 2)) {
            rc = ctx->fail(CDC_ERR_CUDA, "workspace allocation failed (%d x %d x %d x %d bf16)", ctx->B, H, W, C);
            a.p = nullptr;
        }
        return a;
    }
    Act shared(const std::string& tag, int C, int H, int W) {
        const std::string key = tag + ":" + std::to_string(C) + "x" + std::to_string(H) + "x" + std::to_string(W);
        auto it = tmp.find(key);
        if (it != tmp.end()) return it->second;
        Act a = act(C, H, W);
        tmp[key] = a;
        return a;
    }
    // the op of a conv, not yet in the sequence (op.desc says which offered fusions it took); on error rc is set
    Op conv_op(ConvBuild cb) {
        Op op;
        if (rc) return op;
        std::string e;
        cb.sat = ctx->sat_dev;
        int r = build_conv(cb, ctx->B, ctx->opts.plan_sms(ctx->num_sms), ctx->opts, &op, &e);
        if (r) {
            rc = ctx->fail(r, "%s", e.c_str());
            return op;
        }
        for (const auto& kv : ctx->convs) {  // parameter prefixes, for the op description
            if (&kv.second == cb.w) set_desc_name(op.desc.weight, kv.first);
            if (op.desc.res1 && &kv.second == cb.res_w) set_desc_name(op.desc.res_weight, kv.first);
        }
        return op;
    }
    void conv(const ConvBuild& cb) {
        Op op = conv_op(cb);
        if (!rc) seq.ops.push_back(op);
    }
    gn_sum_t* new_gn_slot() {
        if (seq.gn_used >= kMaxGnSlots) {
            rc = ctx->fail(CDC_ERR_SHAPE, "too many GroupNorms in one sequence");
            return seq.slots;
        }
        return seq.slots + static_cast<size_t>(seq.gn_used++) * ctx->B * kGnImgStride;
    }
    // GroupNorm (+FiLM of step k) apply: coefficients come from the accumulator slot inside the kernel
    void gn(const std::string& name, const std::string& gnp, int film_idx, const gn_sum_t* acc, Act x, const act_t* res, Act y,
            bool silu) {
        if (rc) return;
        cdc_ctx* c = ctx;
        const float* gamma = find_w(c, gnp + ".weight")->p;
        const float* beta = find_w(c, gnp + ".bias")->p;
        const int Cc = x.C, HW = x.H * x.W, B = c->B;
        const int foff = film_idx >= 0 ? c->film_off[film_idx] : -1;
        const int sms = c->opts.plan_sms(c->num_sms);
        Op a;
        a.name = name + (silu ? ".apply_silu" : ".apply") + (res ? "_res" : "");
        a.bytes = static_cast<double>(B) * HW * Cc * 2 * (res ? 3 : 2);
        const act_t *xp = x.p, *rp = res;
        act_t* yp = y.p;
        const int si = silu ? 1 : 0;
        a.run = [c, acc, gamma, beta, foff, xp, rp, yp, B, HW, Cc, si, sms](cudaStream_t s, int k, long long* stamp) {
            const float* film = foff >= 0 ? c->film + static_cast<size_t>(k) * c->film_total + foff : nullptr;
            return launch_gn_apply(xp, acc, gamma, beta, film, c->cfg.gn_eps, rp, yp, B, HW, Cc, si, sms, s, stamp, c->sat_dev);
        };
        cdc_step_op_desc& d = a.desc;
        d.kind = CDC_OPK_GN_APPLY;
        set_desc_name(d.weight, gnp);
        d.film_off = foff;
        d.silu = si;
        d.src[0] = tensor_desc(x);
        d.out = tensor_desc(y);
        if (res) {
            d.residual = d.out;
            d.residual.p = const_cast<act_t*>(res);
        }
        d.gn_in_acc = const_cast<gn_sum_t*>(acc);
        seq.ops.push_back(a);
    }
    // Time-conditioned ResBlock (oracle/unet.py RB).  film_idx < 0: RBn (context net).
    void rb(const std::string& name, const std::string& wp, std::vector<Act> in, int cout, int film_idx, Act out) {
        if (rc) return;
        const int H = in[0].H, W = in[0].W, cpg = cout / ctx->cfg.groups;
        int cin = 0;
        for (auto& a : in) cin += a.C;
        Act t1 = shared("t1", cout, H, W), t2 = shared("t2", cout, H, W);
        ConvBuild c1;
        c1.name = name + ".conv1";
        c1.srcs = in;
        c1.w = &ctx->convs[wp + ".conv1"];
        c1.out = t1;
        c1.epi = EPI_STATS;
        c1.cpg = cpg;
        c1.gn_acc = new_gn_slot();
        Act rbuf;
        if (cin != cout) {  // the 1x1 residual conv reads the same input: offered to ride along in the kh-fused kernel
            rbuf = shared("res", cout, H, W);
            c1.res_w = &ctx->convs[wp + ".res"];
            c1.res_out = rbuf;
        }
        const Op conv1 = conv_op(c1);
        if (rc) return;
        seq.ops.push_back(conv1);
        ConvBuild c2;
        c2.name = name + ".conv2";
        c2.srcs = {t1};
        c2.w = &ctx->convs[wp + ".conv2"];
        c2.out = t2;
        c2.epi = EPI_STATS;
        c2.cpg = cpg;
        c2.gn_acc = new_gn_slot();
        // GroupNorm 1 (+FiLM) + SiLU: applied by conv2 to its own input rows in shared memory when the kh-fused kernel has
        // that instantiation (saves a read + write of the tensor in HBM and a launch), else as a pass of its own
        c2.in_acc = c1.gn_acc;
        c2.in_gamma = find_w(ctx, wp + ".gn1.weight")->p;
        c2.in_beta = find_w(ctx, wp + ".gn1.bias")->p;
        c2.in_eps = ctx->cfg.gn_eps;
        c2.in_gn = wp + ".gn1";
        if (film_idx >= 0) {
            c2.in_film_off = ctx->film_off[film_idx];
            c2.film_base = &ctx->film;
            c2.film_total = &ctx->film_total;
        }
        const Op conv2 = conv_op(c2);
        if (rc) return;
        if (!conv2.desc.apply) gn(name + ".gn1", wp + ".gn1", film_idx, c1.gn_acc, t1, nullptr, t1, true);
        seq.ops.push_back(conv2);
        const act_t* resp = in[0].p;
        if (cin != cout) {
            if (!conv1.desc.res1) {
                ConvBuild cr;
                cr.name = name + ".res";
                cr.srcs = in;
                cr.w = &ctx->convs[wp + ".res"];
                cr.ksize = 1;
                cr.out = rbuf;
                conv(cr);
            }
            resp = rbuf.p;
        }
        gn(name + ".gn2", wp + ".gn2", -1, c2.gn_acc, t2, resp, out, true);
    }
};

static int build_plans(cdc_ctx* ctx) {
    const int B = ctx->B, H = ctx->H, W = ctx->W;
    const int* C = ctx->C;
    Arena& ar = ctx->arena;
    const size_t px = static_cast<size_t>(B) * H * W;
    CK(ar.alloc(reinterpret_cast<void**>(&ctx->xs), px * 3 * 4));
    CK(ar.alloc(reinterpret_cast<void**>(&ctx->x0s), px * 3 * 4));
    CK(ar.alloc(reinterpret_cast<void**>(&ctx->img_seeds), (static_cast<size_t>(B) + 1) * 8));
    CK(cudaMemset(ctx->img_seeds, 0, (static_cast<size_t>(B) + 1) * 8));  // per-image mode off
    ctx->seeded = false;
    CK(ar.alloc(reinterpret_cast<void**>(&ctx->gn_slots), 3 * static_cast<size_t>(kMaxGnSlots) * B * kGnImgStride * sizeof(gn_sum_t)));
    Seq* gn_seqs[3] = {&ctx->step_seq, &ctx->ctx_seq, &ctx->enc_seq};  // the sequences with GroupNorms
    for (int i = 0; i < 3; ++i) gn_seqs[i]->slots = ctx->gn_slots + static_cast<size_t>(i) * kMaxGnSlots * B * kGnImgStride;
    CK(ar.alloc(reinterpret_cast<void**>(&ctx->sat_dev), 256));
    CK(cudaMemset(ctx->sat_dev, 0, 256));

    ctx->stage_elems = px * 64;  // largest NCHW fp32 tensor crossing the boundary (c0)
    CK(ar.alloc(reinterpret_cast<void**>(&ctx->stage_f32), ctx->stage_elems * 4));

    PlanB pb(ctx, ctx->step_seq);
    ctx->xpad = pb.act(kXpadC, H, W);  // physically kXpadC channels per pixel ...
    if (pb.rc) return pb.rc;
    CK(cudaMemset(ctx->xpad.p, 0, px * kXpadC * 2));
    ctx->xpad.Cphys = kXpadC;          // ... logically one 64-channel chunk of the stem's input (kernels.cuh)
    ctx->xpad.C = 64;
    for (int i = 0; i < 4; ++i) ctx->cond[i] = pb.act(C[i], H >> i, W >> i);
    ctx->latent = pb.act(ctx->cfg.latent_ch, H >> 4, W >> 4);
    if (pb.rc) return pb.rc;

    // ---- one denoise step (oracle/unet.py UNet.forward + sampler.ddim_update) ----
    int film = 0;
    Act h = pb.act(C[0], H, W);
    {
        ConvBuild cb;
        cb.name = "stem";
        cb.x16 = true;
        cb.srcs = {ctx->xpad, ctx->cond[0]};
        cb.w = &ctx->convs["stem"];
        cb.out = h;
        pb.conv(cb);
    }
    Act skip[4];
    for (int i = 0; i < 4; ++i) {
        const int Hl = H >> i, Wl = W >> i;
        const std::string p = "down." + std::to_string(i);
        Act a = pb.act(C[i], Hl, Wl);
        std::vector<Act> in = {h};
        if (i > 0) in.push_back(ctx->cond[i]);
        pb.rb(p + ".rb1", p + ".rb1", in, C[i], film++, a);
        skip[i] = pb.act(C[i], Hl, Wl);
        pb.rb(p + ".rb2", p + ".rb2", {a}, C[i], film++, skip[i]);
        h = pb.act(C[i], Hl / 2, Wl / 2);
        ConvBuild cb;
        cb.name = p + ".down";
        cb.srcs = {skip[i]};
        cb.w = &ctx->convs[p + ".down"];
        cb.mode = MODE_S2;
        cb.out = h;
        pb.conv(cb);
    }
    {
        const int Hm = H >> 4, Wm = W >> 4, Cm = C[3], HW = Hm * Wm;
        Act m1 = pb.act(Cm, Hm, Wm), m2 = pb.act(Cm, Hm, Wm), m3 = pb.act(Cm, Hm, Wm);
        pb.rb("mid.rb1", "mid.rb1", {h}, Cm, film++, m1);
        // attention: GN -> qkv 1x1 -> flash attention -> proj 1x1 + residual
        Act n = pb.act(Cm, Hm, Wm), qkv = pb.act(3 * Cm, Hm, Wm), o = pb.act(Cm, Hm, Wm);
        if (pb.rc) return pb.rc;
        Op st;
        st.name = "mid.attn.gn.stats";
        st.bytes = static_cast<double>(B) * HW * Cm * 2;
        const act_t* m1p = m1.p;
        gn_sum_t* aslot = pb.new_gn_slot();
        st.run = [aslot, m1p, B, HW, Cm](cudaStream_t s, int, long long* stamp) { return launch_gn_stats(m1p, aslot, B, HW, Cm, s, stamp); };
        st.desc.kind = CDC_OPK_GN_STATS;
        set_desc_name(st.desc.weight, "mid.attn.gn");
        st.desc.film_off = -1;
        st.desc.src[0] = tensor_desc(m1);
        st.desc.gn_out_acc = aslot;
        pb.seq.ops.push_back(st);
        pb.gn("mid.attn.gn", "mid.attn.gn", -1, aslot, m1, nullptr, n, false);
        ConvBuild cq;
        cq.name = "mid.attn.qkv";
        cq.srcs = {n};
        cq.w = &ctx->convs["mid.attn.qkv"];
        cq.ksize = 1;
        cq.out = qkv;
        pb.conv(cq);
        Op at;
        at.name = "mid.attn.sdpa";
        at.flops = static_cast<double>(B) * ctx->cfg.heads * 4.0 * HW * HW * ctx->cfg.head_dim;
        at.bytes = static_cast<double>(B) * HW * Cm * 2 * 4;
        auto ap = std::shared_ptr<AttnTcParams>(new AttnTcParams());
        memset(ap.get(), 0, sizeof(AttnTcParams));
        if (encode_qkv_map(&ap->qkv_map, qkv.p, 3 * Cm, HW, B)) return ctx->fail(CDC_ERR_CUDA, "cuTensorMapEncodeTiled (qkv) failed");
        ap->out = o.p;
        ap->N = HW;
        ap->heads = ctx->cfg.heads;
        at.run = [ap, B](cudaStream_t s, int, long long* stamp) {
            AttnTcParams q = *ap;
            q.stamp = stamp;
            return launch_attention_tc(q, B, s);
        };
        at.desc.kind = CDC_OPK_ATTENTION;
        at.desc.film_off = -1;
        at.desc.src[0] = tensor_desc(qkv);
        at.desc.out = tensor_desc(o);
        pb.seq.ops.push_back(at);
        ConvBuild cpj;
        cpj.name = "mid.attn.proj";
        cpj.srcs = {o};
        cpj.w = &ctx->convs["mid.attn.proj"];
        cpj.ksize = 1;
        cpj.out = m2;
        cpj.residual = m1.p;
        pb.conv(cpj);
        pb.rb("mid.rb2", "mid.rb2", {m2}, Cm, film++, m3);
        h = m3;
    }
    for (int i = 3; i >= 0; --i) {
        const int Hl = H >> i, Wl = W >> i;
        const std::string p = "up." + std::to_string(i);
        Act u = pb.act(C[i], Hl, Wl);
        ConvBuild cb;
        cb.name = p + ".up";
        cb.srcs = {h};
        cb.w = &ctx->convs[p + ".up.up"];
        cb.mode = MODE_UP2;
        cb.out = u;
        pb.conv(cb);
        Act a = pb.act(C[i], Hl, Wl);
        pb.rb(p + ".rb1", p + ".rb1", {u, skip[i]}, C[i], film++, a);
        h = pb.act(C[i], Hl, Wl);
        pb.rb(p + ".rb2", p + ".rb2", {a}, C[i], film++, h);
    }
    {
        ConvBuild cb;
        cb.name = "final+ddim";
        cb.srcs = {h};
        cb.w = &ctx->convs["final"];
        cb.epi = EPI_DDIM;
        cb.x = ctx->xs;
        cb.xpad = ctx->xpad.p;
        cb.x0_out = ctx->x0s;
        cb.samp = &ctx->samp;
        cb.img_seeds = ctx->img_seeds;
        pb.conv(cb);
    }
    if (pb.rc) return pb.rc;

    // ---- context net (oracle/codec.py ContextNet): cond = context_net(y_hat), once per image ----
    if (ctx->has_ctx) {
        PlanB pc(ctx, ctx->ctx_seq);
        Act hh = ctx->latent;
        for (int i = 3; i >= 0; --i) {
            const int Hl = H >> i, Wl = W >> i;
            const std::string p = "context.ups." + std::to_string(i), r = "context.rbs." + std::to_string(i);
            Act u = pc.act(C[i], Hl, Wl);
            ConvBuild cb;
            cb.name = p;
            cb.srcs = {hh};
            cb.w = &ctx->convs[p + ".up"];
            cb.mode = MODE_UP2;
            cb.out = u;
            pc.conv(cb);
            pc.rb(r, r, {u}, C[i], -1, ctx->cond[i]);
            hh = ctx->cond[i];
        }
        if (pc.rc) return pc.rc;
    }

    // ---- codec side (oracle/codec.py Encoder, HyperEncoder, HyperDecoder): SURVEY.md section 8 row f2 ----
    if (ctx->has_codec) {
        const int Cl = ctx->cfg.latent_ch;
        PlanB pe(ctx, ctx->enc_seq);
        ctx->img64 = pe.act(64, H, W);  // 2 * img - 1 in channels 0..2, the rest stays zero
        if (pe.rc) return pe.rc;
        CK(cudaMemset(ctx->img64.p, 0, px * 64 * 2));
        Act eh = pe.act(C[0], H, W);
        {
            ConvBuild cb;
            cb.name = "enc.stem";
            cb.srcs = {ctx->img64};
            cb.w = &ctx->convs["codec.encoder.stem"];
            cb.out = eh;
            pe.conv(cb);
        }
        for (int i = 0; i < 4; ++i) {
            const int Hl = H >> i, Wl = W >> i;
            const std::string si = std::to_string(i);
            Act a = pe.act(C[i], Hl, Wl);
            pe.rb("enc.rb" + si, "codec.encoder.rbs." + si, {eh}, C[i], -1, a);
            eh = pe.act(C[i], Hl / 2, Wl / 2);
            ConvBuild cb;
            cb.name = "enc.down" + si;
            cb.srcs = {a};
            cb.w = &ctx->convs["codec.encoder.downs." + si];
            cb.mode = MODE_S2;
            cb.out = eh;
            pe.conv(cb);
        }
        if (pe.rc) return pe.rc;
        ctx->enc_y = eh;

        auto plain = [&](PlanB& pb, const char* name, const char* wname, Act src, Act dst, int ks, int mode, float slope) {
            ConvBuild cb;
            cb.name = name;
            cb.srcs = {src};
            cb.w = &ctx->convs[wname];
            cb.ksize = ks;
            cb.mode = mode;
            cb.out = dst;
            cb.act_slope = slope;
            cb.force_bn = -1;  // the general kernel: it has the LeakyReLU epilogue, the 5x5 taps and the transposed mode
            pb.conv(cb);
        };
        const int Hy = H >> 4, Wy = W >> 4;
        PlanB ph(ctx, ctx->henc_seq);
        ctx->henc_in = ph.act(Cl, Hy, Wy);
        Act h1 = ph.act(Cl, Hy, Wy), h2 = ph.act(Cl, Hy / 2, Wy / 2);
        ctx->henc_z = ph.act(Cl, Hy / 4, Wy / 4);
        if (ph.rc) return ph.rc;
        plain(ph, "henc.c1", "codec.hyper_enc.c1", ctx->henc_in, h1, 3, MODE_S1, 0.2f);
        plain(ph, "henc.c2", "codec.hyper_enc.c2", h1, h2, 5, MODE_S2, 0.2f);
        plain(ph, "henc.c3", "codec.hyper_enc.c3", h2, ctx->henc_z, 5, MODE_S2, 0.0f);
        if (ph.rc) return ph.rc;

        PlanB pd(ctx, ctx->hdec_seq);
        ctx->hdec_in = pd.act(Cl, Hy / 4, Wy / 4);
        Act d1 = pd.act(Cl, Hy / 2, Wy / 2), d2 = pd.act(Cl, Hy, Wy);
        ctx->hdec_out = pd.act(2 * Cl, Hy, Wy);
        if (pd.rc) return pd.rc;
        plain(pd, "hdec.t1", "codec.hyper_dec.t1", ctx->hdec_in, d1, 5, MODE_CONVT, 0.2f);
        plain(pd, "hdec.t2", "codec.hyper_dec.t2", d1, d2, 5, MODE_CONVT, 0.2f);
        plain(pd, "hdec.c3", "codec.hyper_dec.c3", d2, ctx->hdec_out, 3, MODE_S1, 0.0f);
        if (pd.rc) return pd.rc;
    }
    return CDC_OK;
}

static void drop_traj_graph(cdc_ctx* ctx) {
    if (ctx->traj_graph) cudaGraphExecDestroy(ctx->traj_graph);
    for (cudaEvent_t ev : ctx->traj_ev)
        if (ev) cudaEventDestroy(ev);
    ctx->traj_graph = nullptr;
    ctx->traj_ev.clear();
    ctx->traj_K = ctx->traj_every = ctx->traj_issued = 0;
}

static void drop_graph(cdc_ctx* ctx) {
    if (ctx->graph) cudaGraphExecDestroy(ctx->graph);
    ctx->graph = nullptr;
    ctx->graph_K = 0;
    drop_traj_graph(ctx);
}

// Captures the K-step loop into one graph.  stamps != null: the timing variant (cdc_profile_graph) -- every kernel gets
// its own (start, end) slot [k][op][2].  every > 0: the trajectory variant (cdc_decode_trajectory) -- slot j records step
// k = j * every.  The final conv's epilogue overwrites xs with x_{k+1}, so x_k is stored before step k's ops and x0_hat_k
// after them: one store node at the top of step k takes x_k and x0_hat_{k-1}, a trailing one x0_hat_{K-1}, and the event of
// slot j is recorded once both of its planes are stored.
static int capture_graph(cdc_ctx* ctx, cudaGraphExec_t* out, long long* stamps, int every = 0) {
    if (!ctx->cap_stream) CK(cudaStreamCreateWithFlags(&ctx->cap_stream, cudaStreamNonBlocking));
    cudaGraph_t g = nullptr;
    CK(cudaStreamBeginCapture(ctx->cap_stream, cudaStreamCaptureModeThreadLocal));
    cudaError_t e = cudaSuccess;
    std::string bad;
#ifdef CDC_TOOLS
    // tools build only: CDC_GRAPH_SKIP=substr[,substr...] leaves ops whose name contains a substring out of the graph, so
    // that the in-graph cost of a class of ops can be read off as a difference of replay times (results are then garbage
    // and cdc_get_x refuses to return them)
    std::vector<std::string> skip;
    if (const char* sk = getenv("CDC_GRAPH_SKIP")) {
        std::string t(sk);
        size_t pos = 0;
        while (pos <= t.size()) {
            const size_t c = t.find(',', pos);
            const std::string w = t.substr(pos, c == std::string::npos ? std::string::npos : c - pos);
            if (!w.empty()) skip.push_back(w);
            if (c == std::string::npos) break;
            pos = c + 1;
        }
    }
    if (!skip.empty() && ctx->graph_skip == 0) ctx->graph_skip = 4;
#endif
    const size_t nops = ctx->step_seq.ops.size();
    auto store = [&](int k) {  // trajectory variant, top of step k (k == K: after the last step)
        const int sx = k < ctx->K && k % every == 0 ? k / every : -1;
        const int sx0 = k > 0 && (k - 1) % every == 0 ? (k - 1) / every : -1;
        if (sx < 0 && sx0 < 0) return;
        e = launch_traj_store(ctx->xs, ctx->x0s, ctx->traj_ptrs, sx, sx0, ctx->B, ctx->H * ctx->W, ctx->cap_stream);
        if (e == cudaSuccess && sx0 >= 0) e = cudaEventRecordWithFlags(ctx->traj_ev[sx0], ctx->cap_stream, cudaEventRecordExternal);
        if (e != cudaSuccess) bad = "trajectory store";
    };
    for (int k = 0; k < ctx->K && e == cudaSuccess; ++k) {
        if (every > 0) {
            store(k);
            if (e != cudaSuccess) break;
        }
        for (size_t i = 0; i < nops; ++i) {
            Op& op = ctx->step_seq.ops[i];
#ifdef CDC_TOOLS
            const bool is_conv = op.flops > 0 && op.name.find("sdpa") == std::string::npos;
            const bool is_attn = op.name.find("sdpa") != std::string::npos;
            bool skipped = (ctx->graph_skip == 1 && is_conv) || (ctx->graph_skip == 2 && op.flops == 0 && op.name != "gn.clear") ||
                           (ctx->graph_skip == 3 && is_attn);
            for (const std::string& w : skip) skipped = skipped || op.name.find(w) != std::string::npos;
            if (skipped) continue;
#endif
            e = op.run(ctx->cap_stream, k, stamps ? stamps + (static_cast<size_t>(k) * nops + i) * 2 : nullptr);
            if (e != cudaSuccess) {
                bad = op.name;
                break;
            }
        }
    }
    if (every > 0 && e == cudaSuccess) store(ctx->K);
    cudaError_t e2 = cudaStreamEndCapture(ctx->cap_stream, &g);
    if (e != cudaSuccess) {
        if (g) cudaGraphDestroy(g);
        return ctx->fail(CDC_ERR_CUDA, "graph capture: %s failed: %s", bad.c_str(), cudaGetErrorString(e));
    }
    CK(e2);
    e = cudaGraphInstantiate(out, g, 0);
    cudaGraphDestroy(g);
    CK(e);
    return CDC_OK;
}

static int ensure_graph(cdc_ctx* ctx) {
    if (ctx->graph && ctx->graph_K == ctx->K) return CDC_OK;
    drop_graph(ctx);
    int r = capture_graph(ctx, &ctx->graph, nullptr);
    if (r) return r;
    ctx->graph_K = ctx->K;
    return CDC_OK;
}

static int ensure_traj_graph(cdc_ctx* ctx, int every) {
    if (ctx->traj_graph && ctx->traj_K == ctx->K && ctx->traj_every == every) return CDC_OK;
    if (ctx->traj_graph) CK(cudaEventSynchronize(ctx->traj_done));  // its last launch may still be running
    drop_traj_graph(ctx);
    ctx->traj_ev.assign((ctx->K + every - 1) / every, nullptr);
    for (cudaEvent_t& ev : ctx->traj_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    int r = capture_graph(ctx, &ctx->traj_graph, nullptr, every);
    if (r) {
        drop_traj_graph(ctx);
        return r;
    }
    ctx->traj_K = ctx->K;
    ctx->traj_every = every;
    return CDC_OK;
}

// After a launch that may read the seed block: marks where cdc_set_image_seeds may rewrite it (nothing to mark before the
// first cdc_set_image_seeds: the block has not been written since the bind zeroed it).
static int seeds_read(cdc_ctx* ctx, cudaStream_t s) {
    if (ctx->seeds_done) CK(cudaEventRecord(ctx->seeds_done, s));
    return CDC_OK;
}

// ------------------------------------------------------------------------------------------------ C ABI
#define GUARD() DevGuard dev_guard_(ctx->device)

extern "C" {

int cdc_abi_version(void) { return 2; }

int cdc_act_dtype(void) { return CDC_ACT_FP16 ? 1 : 0; }

const char* cdc_last_error(cdc_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int cdc_create(const cdc_config* cfg, int device, cdc_ctx** out) {
    if (!cfg || !out) {
        g_create_err = "null argument";
        return CDC_ERR_SHAPE;
    }
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        g_create_err = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
        return CDC_ERR_CUDA;
    }
    if (prop.major != 10) {
        g_create_err = "device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                       "; this library is sm_100a only and has no fallback";
        return CDC_ERR_ARCH;
    }
    bool mults_ok = true;
    for (int i = 0; i < 4; ++i) mults_ok = mults_ok && cfg->mults[i] >= 1 && cfg->mults[i] <= 4;
    if (!mults_ok || cfg->groups != 32 || cfg->head_dim != 64 || cfg->heads < 1 || cfg->heads * cfg->head_dim != cfg->base * cfg->mults[3] ||
        cfg->base != 64 || cfg->temb < 1 || cfg->temb > 256 || cfg->latent_ch < 64 || cfg->latent_ch % 64 || cfg->T < 1 ||
        !(cfg->gn_eps > 0.0f)) {
        g_create_err = "unsupported config (need base 64, mults in 1..4, 32 groups, head_dim 64, heads * 64 == base * mults[3], "
                       "1 <= temb <= 256, latent_ch a multiple of 64, T >= 1, gn_eps > 0)";
        return CDC_ERR_SHAPE;
    }
    DevGuard guard(device);
    if (!get_encode()) {
        g_create_err = "cuTensorMapEncodeTiled entry point not found";
        return CDC_ERR_CUDA;
    }
    if ((e = configure_attention_tc()) != cudaSuccess || (e = configure_conv_kernels()) != cudaSuccess ||
        (e = configure_kf_kernels()) != cudaSuccess) {
        g_create_err = std::string("cudaFuncSetAttribute(conv kernels): ") + cudaGetErrorString(e);
        return CDC_ERR_CUDA;
    }
    cdc_ctx* ctx = new cdc_ctx();
    ctx->cfg = *cfg;
    ctx->device = device;
    ctx->num_sms = prop.multiProcessorCount;
    for (int i = 0; i < 4; ++i) ctx->C[i] = cfg->base * cfg->mults[i];
    *out = ctx;
    return CDC_OK;
}

void cdc_destroy(cdc_ctx* ctx) {
    if (!ctx) return;
    {
        GUARD();
        cudaDeviceSynchronize();
        drop_graph(ctx);
        if (ctx->cap_stream) cudaStreamDestroy(ctx->cap_stream);
        ctx->arena.release();
        ctx->warena.release();
        if (ctx->film) cudaFree(ctx->film);
        if (ctx->sinus) cudaFree(ctx->sinus);
        if (ctx->pin_in) cudaFreeHost(ctx->pin_in);
        if (ctx->pin_x) cudaFreeHost(ctx->pin_x);
        if (ctx->pin_out) cudaFreeHost(ctx->pin_out);
        if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
        if (ctx->ev_x) cudaEventDestroy(ctx->ev_x);
        if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
        if (ctx->traj_ptrs) cudaFree(ctx->traj_ptrs);
        if (ctx->traj_done) cudaEventDestroy(ctx->traj_done);
        if (ctx->seeds_done) cudaEventDestroy(ctx->seeds_done);
        byte_codec_destroy(ctx->byte_codec);
    }
    delete ctx;
}

int cdc_load_weights(cdc_ctx* ctx, const char* name, const void* dev_ptr, const int64_t* shape, int ndim) {
    if (!ctx) return CDC_ERR_STATE;
    if (!name || !dev_ptr || !shape || ndim < 1 || ndim > 4) return ctx->fail(CDC_ERR_SHAPE, "cdc_load_weights: null argument or ndim outside 1..4");
    if (ctx->finalized) return ctx->fail(CDC_ERR_STATE, "weights already finalized");
    GUARD();
    WeightT t;
    t.numel = 1;
    for (int i = 0; i < ndim; ++i) {
        if (shape[i] < 1) return ctx->fail(CDC_ERR_SHAPE, "%s: non-positive dimension", name);
        t.shape.push_back(shape[i]);
        t.numel *= static_cast<size_t>(shape[i]);
    }
    CK(ctx->warena.alloc(reinterpret_cast<void**>(&t.p), t.numel * 4));
    CK(cudaMemcpy(t.p, dev_ptr, t.numel * 4, cudaMemcpyDeviceToDevice));
    ctx->w[name] = t;
    return CDC_OK;
}

int cdc_finalize_weights(cdc_ctx* ctx) {
    if (!ctx) return CDC_ERR_STATE;
    if (ctx->finalized) return CDC_OK;
    GUARD();
    const int* C = ctx->C;
    int r;
    // stem: cat[x_t (3), c0 (64)] -> image channels padded to 64, context follows at slot 64
    if ((r = conv_from_store(ctx, "stem", C[0], 3 + C[0], 3, 3, 64, false))) return r;
    for (int i = 0; i < 4; ++i) {
        const std::string p = "down." + std::to_string(i);
        const int cin = i == 0 ? C[0] : C[i - 1] + C[i];
        if ((r = rb_weights(ctx, p + ".rb1", cin, C[i], true))) return r;
        if ((r = rb_weights(ctx, p + ".rb2", C[i], C[i], true))) return r;
        if ((r = conv_from_store(ctx, p + ".down", C[i], C[i], 3, C[i], C[i], false))) return r;
    }
    if ((r = rb_weights(ctx, "mid.rb1", C[3], C[3], true))) return r;
    if ((r = rb_weights(ctx, "mid.rb2", C[3], C[3], true))) return r;
    if ((r = need_vec(ctx, "mid.attn.gn.weight", C[3])) || (r = need_vec(ctx, "mid.attn.gn.bias", C[3]))) return r;
    if ((r = conv_from_store(ctx, "mid.attn.qkv", 3 * C[3], C[3], 1, C[3], C[3], false))) return r;
    if ((r = conv_from_store(ctx, "mid.attn.proj", C[3], C[3], 1, C[3], C[3], false))) return r;
    int prev = C[3];
    for (int i = 3; i >= 0; --i) {
        const std::string p = "up." + std::to_string(i);
        if ((r = conv_from_store(ctx, p + ".up.up", C[i], prev, 3, prev, prev, false, true))) return r;
        if ((r = rb_weights(ctx, p + ".rb1", 2 * C[i], C[i], true))) return r;
        if ((r = rb_weights(ctx, p + ".rb2", C[i], C[i], true))) return r;
        prev = C[i];
    }
    if ((r = conv_from_store(ctx, "final", 3, C[0], 3, C[0], C[0], true))) return r;
    const int te = ctx->cfg.temb;
    if ((r = need_vec(ctx, "temb.lin1.weight", static_cast<size_t>(te) * 64)) || (r = need_vec(ctx, "temb.lin1.bias", te)) ||
        (r = need_vec(ctx, "temb.lin2.weight", static_cast<size_t>(te) * te)) || (r = need_vec(ctx, "temb.lin2.bias", te)))
        return r;
    // optional context net
    ctx->has_ctx = find_w(ctx, "context.ups.3.up.weight") != nullptr;
    if (ctx->has_ctx) {
        prev = ctx->cfg.latent_ch;
        for (int i = 3; i >= 0; --i) {
            const std::string s = std::to_string(i);
            if ((r = conv_from_store(ctx, "context.ups." + s + ".up", C[i], prev, 3, prev, prev, false, true))) return r;
            if ((r = rb_weights(ctx, "context.rbs." + s, C[i], C[i], false))) return r;
            prev = C[i];
        }
    }
    // optional codec side: analysis encoder + hyper-encoder / hyper-decoder ("codec." + oracle Codec.state_dict() names)
    ctx->has_codec = find_w(ctx, "codec.encoder.stem.weight") != nullptr;
    if (ctx->has_codec) {
        const int Cl = ctx->cfg.latent_ch;
        if (Cl != C[3]) return ctx->fail(CDC_ERR_WEIGHT, "codec weights need latent_ch == base * mults[3]");
        if ((r = conv_from_store(ctx, "codec.encoder.stem", C[0], 3, 3, 3, 3, false))) return r;
        prev = C[0];
        for (int i = 0; i < 4; ++i) {
            const std::string s = std::to_string(i);
            if ((r = rb_weights(ctx, "codec.encoder.rbs." + s, prev, C[i], false))) return r;
            if ((r = conv_from_store(ctx, "codec.encoder.downs." + s, C[i], C[i], 3, C[i], C[i], false))) return r;
            prev = C[i];
        }
        if ((r = conv_from_store(ctx, "codec.hyper_enc.c1", Cl, Cl, 3, Cl, Cl, false))) return r;
        if ((r = conv_from_store(ctx, "codec.hyper_enc.c2", Cl, Cl, 5, Cl, Cl, false))) return r;
        if ((r = conv_from_store(ctx, "codec.hyper_enc.c3", Cl, Cl, 5, Cl, Cl, false))) return r;
        if ((r = conv_from_store(ctx, "codec.hyper_dec.t1", Cl, Cl, 5, Cl, Cl, false, false, true))) return r;
        if ((r = conv_from_store(ctx, "codec.hyper_dec.t2", Cl, Cl, 5, Cl, Cl, false, false, true))) return r;
        if ((r = conv_from_store(ctx, "codec.hyper_dec.c3", 2 * Cl, Cl, 3, Cl, Cl, false))) return r;
    }
    // FiLM offsets
    std::vector<int> couts;
    film_rb_names(ctx, &couts);
    ctx->film_off.clear();
    int off = 0;
    for (int c : couts) {
        ctx->film_off.push_back(off);
        off += 2 * c;
    }
    ctx->film_total = off;
    CK(cudaDeviceSynchronize());
    ctx->finalized = true;
    return CDC_OK;
}

int cdc_has_context_net(cdc_ctx* ctx) { return ctx && ctx->has_ctx ? 1 : 0; }
int cdc_has_codec(cdc_ctx* ctx) { return ctx && ctx->has_codec ? 1 : 0; }

int cdc_set_sampler(cdc_ctx* ctx, int pred_eps, float eta, uint64_t seed) {
    if (!ctx) return CDC_ERR_STATE;
    if ((pred_eps != 0 && pred_eps != 1) || !(eta >= 0.0f) || eta > 10.0f) return ctx->fail(CDC_ERR_SHAPE, "pred_eps must be 0/1 and 0 <= eta <= 10");
    if (pred_eps != ctx->pred_eps || eta != ctx->eta || seed != ctx->seed) {
        ctx->pred_eps = pred_eps;
        ctx->eta = eta;
        ctx->seed = seed;
        if (ctx->K > 0) {  // coefficients are baked into the graph: recompute them now
            const int K = ctx->K;
            ctx->K = 0;
            return cdc_set_schedule(ctx, K);
        }
    }
    return CDC_OK;
}

int cdc_set_schedule(cdc_ctx* ctx, int K) {
    if (!ctx || !ctx->finalized) return ctx ? ctx->fail(CDC_ERR_STATE, "finalize weights first") : CDC_ERR_STATE;
    if (K < 1 || K > ctx->cfg.T) return ctx->fail(CDC_ERR_SHAPE, "steps must be in [1, T]");
    GUARD();
    const int T = ctx->cfg.T;
    // cosine schedule, float64 (oracle/sampler.py alphas_cumprod)
    std::vector<double> ab(T);
    auto f = [&](double u) {
        const double c = cos((u / T + 0.008) / 1.008 * M_PI / 2.0);
        return c * c;
    };
    double cum = 1.0;
    for (int t = 0; t < T; ++t) {
        double beta = 1.0 - f(t + 1.0) / f(static_cast<double>(t));
        beta = beta < 0.0 ? 0.0 : (beta > 0.999 ? 0.999 : beta);
        cum *= 1.0 - beta;
        ab[t] = cum;
    }
    std::vector<int> idx(K);
    SamplerTab st;
    st.c0.resize(K);
    st.c1.resize(K);
    st.e0.resize(K);
    st.e1.resize(K);
    st.sg.resize(K);
    st.seed = ctx->seed;
    for (int k = 0; k < K; ++k)
        idx[k] = K == 1 ? T - 1 : static_cast<int>((static_cast<long long>(K - 1 - k) * (T - 1) + (K - 1) / 2) / (K - 1));
    for (int k = 0; k < K; ++k) {  // oracle/sampler.py make_schedule, float64 -> fp32
        const double at = ab[idx[k]], ap = k + 1 < K ? ab[idx[k + 1]] : 1.0;
        const double sg = ctx->eta > 0.0f && ap < 1.0 ? static_cast<double>(ctx->eta) * sqrt((1.0 - ap) / (1.0 - at)) * sqrt(1.0 - at / ap) : 0.0;
        const double dir2 = 1.0 - ap - sg * sg;
        const double v1 = sqrt(dir2 > 0.0 ? dir2 : 0.0) / sqrt(1.0 - at);
        st.c1[k] = static_cast<float>(v1);
        st.c0[k] = static_cast<float>(sqrt(ap) - v1 * sqrt(at));
        st.sg[k] = static_cast<float>(sg);
        st.e0[k] = ctx->pred_eps ? static_cast<float>(1.0 / sqrt(at)) : 0.0f;
        st.e1[k] = ctx->pred_eps ? static_cast<float>(-sqrt(1.0 - at) / sqrt(at)) : 1.0f;
    }
    // the graph bakes per-step pointers/coefficients: any schedule change invalidates it
    drop_graph(ctx);
    ctx->K = K;
    ctx->idx = idx;
    ctx->samp = st;

    // sinusoidal embedding per step (host, float64 -> fp32), then MLP + FiLM on the device
    std::vector<float> sin_h(static_cast<size_t>(K) * 64);
    for (int k = 0; k < K; ++k)
        for (int j = 0; j < 32; ++j) {
            const float fj = static_cast<float>(exp(-log(10000.0) * j / 32.0));
            const float a = static_cast<float>(idx[k]) * fj;  // fp32 product like the oracle
            sin_h[static_cast<size_t>(k) * 64 + j] = static_cast<float>(sin(static_cast<double>(a)));
            sin_h[static_cast<size_t>(k) * 64 + 32 + j] = static_cast<float>(cos(static_cast<double>(a)));
        }
    if (ctx->film) cudaFree(ctx->film);
    if (ctx->sinus) cudaFree(ctx->sinus);
    ctx->film = nullptr;
    ctx->sinus = nullptr;
    CK(cudaMalloc(&ctx->film, static_cast<size_t>(K) * ctx->film_total * 4));
    CK(cudaMalloc(&ctx->sinus, sin_h.size() * 4));
    CK(cudaMemcpy(ctx->sinus, sin_h.data(), sin_h.size() * 4, cudaMemcpyHostToDevice));
    FilmParams fp;
    memset(&fp, 0, sizeof fp);
    fp.sinus = ctx->sinus;
    fp.w1 = find_w(ctx, "temb.lin1.weight")->p;
    fp.b1 = find_w(ctx, "temb.lin1.bias")->p;
    fp.w2 = find_w(ctx, "temb.lin2.weight")->p;
    fp.b2 = find_w(ctx, "temb.lin2.bias")->p;
    std::vector<int> couts;
    std::vector<std::string> names = film_rb_names(ctx, &couts);
    fp.nlayers = static_cast<int>(names.size());
    for (int i = 0; i < fp.nlayers; ++i) {
        fp.layer[i].w = find_w(ctx, names[i] + ".film.weight")->p;
        fp.layer[i].b = find_w(ctx, names[i] + ".film.bias")->p;
        fp.layer[i].c2 = 2 * couts[i];
        fp.layer[i].offset = ctx->film_off[i];
    }
    fp.temb = ctx->cfg.temb;
    fp.total = ctx->film_total;
    fp.out = ctx->film;
    CK(launch_temb_film(fp, K, nullptr));
    CK(cudaDeviceSynchronize());
    return CDC_OK;
}

int cdc_schedule_index(cdc_ctx* ctx, int k) { return (ctx && k >= 0 && k < ctx->K) ? ctx->idx[k] : -1; }

int cdc_schedule_coeffs(cdc_ctx* ctx, int k, float* c0, float* c1) {
    if (!ctx || k < 0 || k >= ctx->K || !c0 || !c1) return CDC_ERR_SHAPE;
    *c0 = ctx->samp.c0[k];
    *c1 = ctx->samp.c1[k];
    return CDC_OK;
}

int cdc_schedule_coeffs5(cdc_ctx* ctx, int k, float* c0, float* c1, float* e0, float* e1, float* sigma) {
    if (!ctx || k < 0 || k >= ctx->K || !c0 || !c1 || !e0 || !e1 || !sigma) return CDC_ERR_SHAPE;
    *c0 = ctx->samp.c0[k];
    *c1 = ctx->samp.c1[k];
    *e0 = ctx->samp.e0[k];
    *e1 = ctx->samp.e1[k];
    *sigma = ctx->samp.sg[k];
    return CDC_OK;
}

int cdc_film_size(cdc_ctx* ctx) { return ctx && ctx->finalized ? ctx->film_total : 0; }

int cdc_get_film(cdc_ctx* ctx, float* film_dev, cdc_stream s) {
    if (!ctx || !ctx->film || ctx->K < 1) return ctx ? ctx->fail(CDC_ERR_STATE, "call cdc_set_schedule first") : CDC_ERR_STATE;
    if (!film_dev) return ctx->fail(CDC_ERR_SHAPE, "null output");
    GUARD();
    CK(cudaMemcpyAsync(film_dev, ctx->film, static_cast<size_t>(ctx->K) * ctx->film_total * 4, cudaMemcpyDeviceToDevice, S(s)));
    return CDC_OK;
}

static void release_plan(cdc_ctx* ctx) {  // every op sequence and the workspace they run on
    for (Seq* q : {&ctx->step_seq, &ctx->ctx_seq, &ctx->enc_seq, &ctx->henc_seq, &ctx->hdec_seq}) *q = Seq();
    byte_codec_release_buffers(ctx->byte_codec);
    ctx->arena.release();
}

int cdc_bind_io(cdc_ctx* ctx, int B, int H, int W) {
    if (!ctx || !ctx->finalized) return ctx ? ctx->fail(CDC_ERR_STATE, "finalize weights first") : CDC_ERR_STATE;
    if (B < 1 || H < 64 || W < 64 || (H % 64) || (W % 64)) return ctx->fail(CDC_ERR_SHAPE, "H and W must be multiples of 64, batch >= 1");
    if (B > kMaxBatch)
        return ctx->fail(CDC_ERR_SHAPE, "batch %d > %d: the GroupNorm apply kernel holds every image's statistics table in 48 KB of shared memory", B, kMaxBatch);
    if (B == ctx->B && H == ctx->H && W == ctx->W && !ctx->step_seq.ops.empty() && !ctx->opts_dirty) return CDC_OK;
    GUARD();
    CK(cudaDeviceSynchronize());
    drop_graph(ctx);
    release_plan(ctx);
    ctx->B = B;
    ctx->H = H;
    ctx->W = W;
    ctx->opts_dirty = false;
    int r = build_plans(ctx);
    if (r) {
        release_plan(ctx);
        ctx->B = ctx->H = ctx->W = 0;
        return r;
    }
    CK(cudaDeviceSynchronize());
    return CDC_OK;
}

int cdc_set_batch_invariant(cdc_ctx* ctx, int on) {
    if (!ctx) return CDC_ERR_STATE;
    if (on != 0 && on != 1) return ctx->fail(CDC_ERR_SHAPE, "cdc_set_batch_invariant: %d is neither 0 nor 1", on);
    if (ctx->opts.batch_invariant != (on == 1)) {
        ctx->opts.batch_invariant = on == 1;
        ctx->opts_dirty = true;  // the next cdc_bind_io re-plans, also for the bound shape
    }
    return CDC_OK;
}

#define NEED_PLAN()                                                                     \
    if (!ctx || ctx->step_seq.ops.empty()) return ctx ? ctx->fail(CDC_ERR_STATE, "call cdc_bind_io first") : CDC_ERR_STATE; \
    GUARD()

int cdc_set_cond(cdc_ctx* ctx, const float* c0, const float* c1, const float* c2, const float* c3, cdc_stream s) {
    NEED_PLAN();
    const float* src[4] = {c0, c1, c2, c3};
    for (int i = 0; i < 4; ++i) {
        if (!src[i]) return ctx->fail(CDC_ERR_SHAPE, "cdc_set_cond: null context map %d", i);
        const Act& a = ctx->cond[i];
        CK(launch_nchw_f32_to_nhwc_act(src[i], a.p, ctx->B, a.C, a.H * a.W, a.C, S(s)));
    }
    return CDC_OK;
}

int cdc_get_cond(cdc_ctx* ctx, float* c0, float* c1, float* c2, float* c3, cdc_stream s) {
    NEED_PLAN();
    float* dst[4] = {c0, c1, c2, c3};
    for (int i = 0; i < 4; ++i) {
        if (!dst[i]) continue;
        const Act& a = ctx->cond[i];
        CK(launch_nhwc_act_to_nchw_f32(a.p, dst[i], ctx->B, a.C, a.H * a.W, S(s)));
    }
    return CDC_OK;
}

static int run_ops(cdc_ctx* ctx, Seq& seq, cudaStream_t s, int k = 0) {
    for (Op& op : seq.ops) {
        cudaError_t e = op.run(s, k, nullptr);
        if (e != cudaSuccess) return ctx->fail(CDC_ERR_CUDA, "%s: %s", op.name.c_str(), cudaGetErrorString(e));
    }
    return CDC_OK;
}

int cdc_set_latent(cdc_ctx* ctx, const float* y_hat, cdc_stream s) {
    NEED_PLAN();
    if (!ctx->has_ctx) return ctx->fail(CDC_ERR_WEIGHT, "context-net weights (context.*) were not loaded");
    if (!y_hat) return ctx->fail(CDC_ERR_SHAPE, "null latent");
    const Act& a = ctx->latent;
    CK(launch_nchw_f32_to_nhwc_act(y_hat, a.p, ctx->B, a.C, a.H * a.W, a.C, S(s)));
    return run_ops(ctx, ctx->ctx_seq, S(s));
}

// ---- codec side (row f2) ----
#define NEED_CODEC() \
    if (!ctx->has_codec) return ctx->fail(CDC_ERR_WEIGHT, "codec weights (codec.encoder.* / codec.hyper_enc.* / codec.hyper_dec.*) were not loaded")

int cdc_encode_analysis(cdc_ctx* ctx, const float* img01, float* y, cdc_stream s) {
    NEED_PLAN();
    NEED_CODEC();
    if (!img01 || !y) return ctx->fail(CDC_ERR_SHAPE, "null buffer");
    CK(launch_img_in(img01, ctx->img64.p, ctx->B, ctx->H * ctx->W, S(s)));
    int r = run_ops(ctx, ctx->enc_seq, S(s));
    if (r) return r;
    const Act& a = ctx->enc_y;
    CK(launch_nhwc_act_to_nchw_f32(a.p, y, ctx->B, a.C, a.H * a.W, S(s)));
    return CDC_OK;
}

int cdc_hyper_encode(cdc_ctx* ctx, const float* y, float* z, cdc_stream s) {
    NEED_PLAN();
    NEED_CODEC();
    if (!y || !z) return ctx->fail(CDC_ERR_SHAPE, "null buffer");
    const Act& a = ctx->henc_in;
    CK(launch_nchw_f32_to_nhwc_act(y, a.p, ctx->B, a.C, a.H * a.W, a.C, S(s)));
    int r = run_ops(ctx, ctx->henc_seq, S(s));
    if (r) return r;
    const Act& zz = ctx->henc_z;
    CK(launch_nhwc_act_to_nchw_f32(zz.p, z, ctx->B, zz.C, zz.H * zz.W, S(s)));
    return CDC_OK;
}

int cdc_hyper_decode(cdc_ctx* ctx, const float* z_hat, float* mu, float* sigma, cdc_stream s) {
    NEED_PLAN();
    NEED_CODEC();
    if (!z_hat || !mu || !sigma) return ctx->fail(CDC_ERR_SHAPE, "null buffer");
    const Act& a = ctx->hdec_in;
    CK(launch_nchw_f32_to_nhwc_act(z_hat, a.p, ctx->B, a.C, a.H * a.W, a.C, S(s)));
    int r = run_ops(ctx, ctx->hdec_seq, S(s));
    if (r) return r;
    const Act& o = ctx->hdec_out;
    const int Cl = o.C / 2, HW = o.H * o.W;
    CK(launch_nhwc_slice_to_nchw_f32(o.p, mu, ctx->B, Cl, HW, o.C, 0, 0.0f, 0, S(s)));
    CK(launch_nhwc_slice_to_nchw_f32(o.p, sigma, ctx->B, Cl, HW, o.C, Cl, kMinSigma, 1, S(s)));  // sigma = max(sigma_raw, 0.11)
    return CDC_OK;
}

int cdc_set_x(cdc_ctx* ctx, const float* x, cdc_stream s) {
    NEED_PLAN();
    if (!x) return ctx->fail(CDC_ERR_SHAPE, "null x");
    CK(launch_x_in(x, ctx->xs, ctx->xpad.p, ctx->B, ctx->H * ctx->W, S(s)));
    return CDC_OK;
}

int cdc_get_x(cdc_ctx* ctx, float* x, int to_image, cdc_stream s) {
    NEED_PLAN();
    if (!x) return ctx->fail(CDC_ERR_SHAPE, "null output");
    if (ctx->graph_skip) return ctx->fail(CDC_ERR_STATE, "ops are being left out of the graph (tools build, graph skip): x is garbage");
    CK(launch_x_out(ctx->xs, x, ctx->B, ctx->H * ctx->W, to_image, S(s)));
    return CDC_OK;
}

int cdc_get_x0(cdc_ctx* ctx, float* x0, cdc_stream s) {
    NEED_PLAN();
    if (!x0) return ctx->fail(CDC_ERR_SHAPE, "null output");
    CK(launch_x_out(ctx->x0s, x0, ctx->B, ctx->H * ctx->W, 0, S(s)));
    return CDC_OK;
}

int cdc_set_image_seeds(cdc_ctx* ctx, const uint64_t* seeds_host, int n, cdc_stream s) {
    NEED_PLAN();
    if (n != 0 && n != ctx->B) return ctx->fail(CDC_ERR_SHAPE, "cdc_set_image_seeds: %d seeds for a batch of %d (give B, or 0 to turn per-image mode off)", n, ctx->B);
    if (n != 0 && !seeds_host) return ctx->fail(CDC_ERR_SHAPE, "cdc_set_image_seeds: null seeds");
    if (n == 0 && !ctx->seeded) return CDC_OK;
    if (!ctx->seeds_done) CK(cudaEventCreateWithFlags(&ctx->seeds_done, cudaEventDisableTiming));
    // the previous launch that reads the block (possibly on another stream) must be past it
    CK(cudaStreamWaitEvent(S(s), ctx->seeds_done, 0));
    if (n == 0) {
        CK(cudaMemsetAsync(ctx->img_seeds, 0, 8, S(s)));
    } else {
        std::vector<unsigned long long> blk(static_cast<size_t>(n) + 1);
        blk[0] = 1;
        for (int b = 0; b < n; ++b) blk[b + 1] = seeds_host[b];
        // (pageable source: staged by the driver before the call returns, so blk may go out of scope)
        CK(cudaMemcpyAsync(ctx->img_seeds, blk.data(), blk.size() * 8, cudaMemcpyHostToDevice, S(s)));
    }
    ctx->seeded = n != 0;
    return CDC_OK;
}

int cdc_init_noise(cdc_ctx* ctx, float gamma, cdc_stream s) {
    NEED_PLAN();
    if (!ctx->seeded) return ctx->fail(CDC_ERR_STATE, "cdc_init_noise: no per-image seeds bound (cdc_set_image_seeds)");
    CK(launch_init_noise(ctx->img_seeds, ctx->xs, ctx->xpad.p, gamma, ctx->B, ctx->H * ctx->W, S(s)));
    return seeds_read(ctx, S(s));
}

int cdc_denoise_step(cdc_ctx* ctx, int k, cdc_stream s) {
    NEED_PLAN();
    if (k < 0 || k >= ctx->K) return ctx->fail(CDC_ERR_SHAPE, "step %d outside the %d-step schedule", k, ctx->K);
    int r = run_ops(ctx, ctx->step_seq, S(s), k);
    return r ? r : seeds_read(ctx, S(s));
}

int cdc_decode(cdc_ctx* ctx, cdc_stream s) {
    NEED_PLAN();
    if (ctx->K < 1) return ctx->fail(CDC_ERR_STATE, "call cdc_set_schedule first");
    int r = ensure_graph(ctx);
    if (r) return r;
    CK(cudaGraphLaunch(ctx->graph, S(s)));
    return seeds_read(ctx, S(s));
}

int cdc_decode_trajectory(cdc_ctx* ctx, float* x_traj, float* x0_traj, int every, cdc_stream s) {
    NEED_PLAN();
    if (ctx->K < 1) return ctx->fail(CDC_ERR_STATE, "call cdc_set_schedule first");
    if (every < 1) return ctx->fail(CDC_ERR_SHAPE, "cdc_decode_trajectory: every must be >= 1, got %d", every);
    if (!x_traj && !x0_traj) return ctx->fail(CDC_ERR_SHAPE, "cdc_decode_trajectory: both trajectory buffers are null");
    if (ctx->graph_skip) return ctx->fail(CDC_ERR_STATE, "ops are being left out of the graph (tools build, graph skip): x is garbage");
    if (!ctx->traj_ptrs) {  // both or neither
        TrajPtrs* p = nullptr;
        cudaEvent_t ev = nullptr;
        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        const cudaError_t e = cudaMalloc(&p, sizeof(TrajPtrs));
        if (e != cudaSuccess) {
            cudaEventDestroy(ev);
            return ctx->fail(CDC_ERR_CUDA, "cudaMalloc(trajectory pointer block): %s", cudaGetErrorString(e));
        }
        ctx->traj_ptrs = p;
        ctx->traj_done = ev;
    }
    int r = ensure_traj_graph(ctx, every);
    if (r) return r;
    // the previous launch (possibly on another stream) reads traj_ptrs until its last store node
    CK(cudaStreamWaitEvent(S(s), ctx->traj_done, 0));
    CK(launch_traj_set_ptrs(ctx->traj_ptrs, x_traj, x0_traj, S(s)));
    CK(cudaGraphLaunch(ctx->traj_graph, S(s)));
    CK(cudaEventRecord(ctx->traj_done, S(s)));
    ctx->traj_issued = static_cast<int>(ctx->traj_ev.size());
    return seeds_read(ctx, S(s));
}

int cdc_trajectory_wait(cdc_ctx* ctx, int j) {
    if (!ctx) return CDC_ERR_STATE;
    if (!ctx->traj_issued) return ctx->fail(CDC_ERR_STATE, "cdc_trajectory_wait: no cdc_decode_trajectory since the last bind / schedule change");
    if (j < 0 || j >= ctx->traj_issued)
        return ctx->fail(CDC_ERR_SHAPE, "cdc_trajectory_wait: slot %d outside the %d slots of the last trajectory decode", j, ctx->traj_issued);
    GUARD();
    CK(cudaEventSynchronize(ctx->traj_ev[j]));
    return CDC_OK;
}

static bool host_ptr_is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();  // (unregistered host memory reports an error on old drivers)
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

// cdc_decode_host (xT_host given) and cdc_decode_host_seeded (xT_host null: x_T drawn on the device from the bound seeds)
static int decode_host(cdc_ctx* ctx, const float* latent_host, const float* xT_host, float gamma, float* image_host, cdc_stream s) {
    if (!latent_host || !image_host) return ctx->fail(CDC_ERR_SHAPE, "null host buffer");
    const size_t nl = static_cast<size_t>(ctx->B) * ctx->cfg.latent_ch * (ctx->H / 16) * (ctx->W / 16);
    const size_t nx = static_cast<size_t>(ctx->B) * 3 * ctx->H * ctx->W;
    if (nl > ctx->pin_nl || nx > ctx->pin_nx) {  // (re)size the pinned staging buffers for this shape
        CK(cudaStreamSynchronize(S(s)));
        if (ctx->pin_in) cudaFreeHost(ctx->pin_in);
        if (ctx->pin_x) cudaFreeHost(ctx->pin_x);
        if (ctx->pin_out) cudaFreeHost(ctx->pin_out);
        ctx->pin_in = ctx->pin_x = ctx->pin_out = nullptr;
        ctx->pin_nl = ctx->pin_nx = 0;
        CK(cudaMallocHost(&ctx->pin_in, nl * 4));
        CK(cudaMallocHost(&ctx->pin_x, nx * 4));
        CK(cudaMallocHost(&ctx->pin_out, nx * 4));
        ctx->pin_nl = nl;
        ctx->pin_nx = nx;
    }
    if (!ctx->copy_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->ev_x, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    }
    // page-locked caller buffers are copied from / to directly; pageable ones go through the pinned staging buffers
    const float* lat_src = latent_host;
    const float* x_src = xT_host;
    if (!host_ptr_is_pinned(latent_host)) {
        memcpy(ctx->pin_in, latent_host, nl * 4);
        lat_src = ctx->pin_in;
    }
    if (xT_host && !host_ptr_is_pinned(xT_host)) {
        memcpy(ctx->pin_x, xT_host, nx * 4);
        x_src = ctx->pin_x;
    }
    float* d_lat = ctx->stage_f32;
    float* d_x = ctx->stage_f32 + nl;
    if (nl + nx > ctx->stage_elems) return ctx->fail(CDC_ERR_SHAPE, "staging buffer too small");
    if (xT_host) {  // x_T (4.7 MB at 768x512) rides a second stream while the context net runs on the latent
        CK(cudaEventRecord(ctx->ev_fork, S(s)));
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_fork, 0));
        CK(cudaMemcpyAsync(d_x, x_src, nx * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(ctx->ev_x, ctx->copy_stream));
    }
    CK(cudaMemcpyAsync(d_lat, lat_src, nl * 4, cudaMemcpyHostToDevice, S(s)));
    int r;
    if ((r = cdc_set_latent(ctx, d_lat, s))) return r;
    if (xT_host) {
        CK(cudaStreamWaitEvent(S(s), ctx->ev_x, 0));
        if ((r = cdc_set_x(ctx, d_x, s))) return r;
    } else if ((r = cdc_init_noise(ctx, gamma, s))) {
        return r;
    }
    if ((r = cdc_decode(ctx, s))) return r;
    if ((r = cdc_get_x(ctx, d_x, 1, s))) return r;
    const bool out_pinned = host_ptr_is_pinned(image_host);
    CK(cudaMemcpyAsync(out_pinned ? image_host : ctx->pin_out, d_x, nx * 4, cudaMemcpyDeviceToHost, S(s)));
    CK(cudaStreamSynchronize(S(s)));
    if (!out_pinned) memcpy(image_host, ctx->pin_out, nx * 4);
    return CDC_OK;
}

int cdc_decode_host(cdc_ctx* ctx, const float* latent_host, const float* xT_host, float* image_host, cdc_stream s) {
    NEED_PLAN();
    if (!xT_host) return ctx->fail(CDC_ERR_SHAPE, "null host buffer");
    return decode_host(ctx, latent_host, xT_host, 0.0f, image_host, s);
}

int cdc_decode_host_seeded(cdc_ctx* ctx, const float* latent_host, float gamma, float* image_host, cdc_stream s) {
    NEED_PLAN();
    if (!ctx->seeded) return ctx->fail(CDC_ERR_STATE, "cdc_decode_host_seeded: no per-image seeds bound (cdc_set_image_seeds)");
    return decode_host(ctx, latent_host, nullptr, gamma, image_host, s);
}

}  // extern "C"

// ---- what bitstream.cu (cdc_compress_rgb8 / cdc_decompress_rgb8) sees of a context (codec_io.cuh) ----
namespace cdc {
int bound_codec(cdc_ctx* ctx, BoundCodec* out) {
    NEED_PLAN();
    NEED_CODEC();
    BoundCodec v;
    v.B = ctx->B;
    v.H = ctx->H;
    v.W = ctx->W;
    v.latent_ch = ctx->cfg.latent_ch;
    v.num_sms = ctx->num_sms;
    v.device = ctx->device;
    v.K = ctx->K;
    v.has_ctx = ctx->has_ctx;
    v.seeded = ctx->seeded;
    v.graph_skip = ctx->graph_skip != 0;
    v.img64 = ctx->img64.p;
    v.enc_y = ctx->enc_y.p;
    v.hdec_in = ctx->hdec_in.p;
    v.hdec_out = ctx->hdec_out.p;
    v.latent = ctx->latent.p;
    v.xs = ctx->xs;
    v.state = &ctx->byte_codec;
    *out = v;
    return CDC_OK;
}
ByteCodec** byte_codec_slot(cdc_ctx* ctx) { return &ctx->byte_codec; }
int ctx_device(cdc_ctx* ctx) { return ctx->device; }
int ctx_latent_ch(cdc_ctx* ctx) { return ctx->cfg.latent_ch; }
int run_codec_seq(cdc_ctx* ctx, CodecSeq q, cudaStream_t s) {
    return run_ops(ctx, q == CODEC_SEQ_ENCODER ? ctx->enc_seq : q == CODEC_SEQ_HYPER_DEC ? ctx->hdec_seq : ctx->ctx_seq, s);
}
int ctx_fail(cdc_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    ctx->err = buf;
    return code;
}
}  // namespace cdc

extern "C" {

static int count_kernels(const std::vector<Op>& ops) {  // the GroupNorm-slot memset node is not a kernel of ours
    int n = 0;
    for (const Op& op : ops) n += op.name != "gn.clear";
    return n;
}
int cdc_launches_per_step(cdc_ctx* ctx) { return ctx ? count_kernels(ctx->step_seq.ops) : 0; }
int cdc_launches_context(cdc_ctx* ctx) { return ctx ? count_kernels(ctx->ctx_seq.ops) + 1 : 0; }

double cdc_flops_per_step(cdc_ctx* ctx) {
    if (!ctx) return 0;
    double f = 0;
    for (Op& op : ctx->step_seq.ops) f += op.flops;
    // time-embedding MLP + FiLM linears (precomputed per schedule; counted for parity with SURVEY 8d)
    f += 2.0 * ctx->B * (64.0 * ctx->cfg.temb + static_cast<double>(ctx->cfg.temb) * ctx->cfg.temb);
    f += 2.0 * ctx->B * ctx->cfg.temb * static_cast<double>(ctx->film_total);
    return f;
}

int cdc_saturation_count(cdc_ctx* ctx, uint64_t* count, int reset, cdc_stream s) {
    NEED_PLAN();
    if (!count) return ctx->fail(CDC_ERR_SHAPE, "null output");
    unsigned int v = 0;
    CK(cudaMemcpyAsync(&v, ctx->sat_dev, 4, cudaMemcpyDeviceToHost, S(s)));
    if (reset) CK(cudaMemsetAsync(ctx->sat_dev, 0, 4, S(s)));
    CK(cudaStreamSynchronize(S(s)));
    *count = v;
    return CDC_OK;
}

// ---------------------------------------------------------------------------------------------- tools header
int cdc_set_plan_option(cdc_ctx* ctx, int option, int value) {
    if (!ctx) return CDC_ERR_STATE;
    if (option < 0 || option >= CDC_OPT_COUNT || value < 0) return ctx->fail(CDC_ERR_SHAPE, "unknown plan option %d / negative value", option);
    if (ctx->opts.v[option] != value) {
        ctx->opts.v[option] = value;
        ctx->opts_dirty = true;
    }
    return CDC_OK;
}

// The op sequence `seq` (cdc_seq) of the plan, or null with the error in ctx->err and its code in *rc.
static Seq* find_seq(cdc_ctx* ctx, int seq, int* rc) {
    switch (seq) {
        case CDC_SEQ_STEP: return &ctx->step_seq;
        case CDC_SEQ_CONTEXT:
            if (ctx->has_ctx) return &ctx->ctx_seq;
            *rc = ctx->fail(CDC_ERR_WEIGHT, "op sequence %d: context-net weights (context.*) were not loaded", seq);
            return nullptr;
        case CDC_SEQ_ENCODER:
        case CDC_SEQ_HYPER_ENC:
        case CDC_SEQ_HYPER_DEC:
            if (ctx->has_codec) return seq == CDC_SEQ_ENCODER ? &ctx->enc_seq : seq == CDC_SEQ_HYPER_ENC ? &ctx->henc_seq : &ctx->hdec_seq;
            *rc = ctx->fail(CDC_ERR_WEIGHT, "op sequence %d: codec weights (codec.*) were not loaded", seq);
            return nullptr;
        default:
            *rc = ctx->fail(CDC_ERR_SHAPE, "unknown op sequence %d", seq);
            return nullptr;
    }
}
// op i of sequence seq, or null (error in ctx->err)
static const Op* find_op(cdc_ctx* ctx, int seq, int i) {
    int rc = CDC_OK;
    const Seq* q = ctx ? find_seq(ctx, seq, &rc) : nullptr;
    if (!q) return nullptr;
    if (i < 0 || i >= static_cast<int>(q->ops.size())) {
        ctx->fail(CDC_ERR_SHAPE, "op %d outside the %zu ops of sequence %d", i, q->ops.size(), seq);
        return nullptr;
    }
    return &q->ops[i];
}

int cdc_seq_num_ops(cdc_ctx* ctx, int seq) {
    if (!ctx) return 0;
    int rc = CDC_OK;
    const Seq* q = find_seq(ctx, seq, &rc);
    return q ? static_cast<int>(q->ops.size()) : rc;
}
const char* cdc_seq_op_name(cdc_ctx* ctx, int seq, int i) {
    const Op* op = find_op(ctx, seq, i);
    return op ? op->name.c_str() : "";
}
double cdc_seq_op_flops(cdc_ctx* ctx, int seq, int i) {
    const Op* op = find_op(ctx, seq, i);
    return op ? op->flops : 0;
}
double cdc_seq_op_bytes(cdc_ctx* ctx, int seq, int i) {
    const Op* op = find_op(ctx, seq, i);
    return op ? op->bytes : 0;
}
int cdc_seq_op_describe(cdc_ctx* ctx, int seq, int i, cdc_step_op_desc* out) {
    if (!ctx) return CDC_ERR_STATE;
    if (!out) return ctx->fail(CDC_ERR_SHAPE, "null output");
    int rc = CDC_OK;
    const Seq* q = find_seq(ctx, seq, &rc);
    if (!q) return rc;
    const Op* op = find_op(ctx, seq, i);
    if (!op) return CDC_ERR_SHAPE;
    *out = op->desc;
    if (out->kind == CDC_OPK_MEMSET) out->gn_slots = q->gn_used;
    return CDC_OK;
}
int cdc_run_seq_op(cdc_ctx* ctx, int seq, int i, int k, cdc_stream s) {
    NEED_PLAN();
    int rc = CDC_OK;
    if (!find_seq(ctx, seq, &rc)) return rc;
    const Op* op = find_op(ctx, seq, i);
    if (!op) return CDC_ERR_SHAPE;
    if (seq == CDC_SEQ_STEP && (k < 0 || k >= ctx->K)) return ctx->fail(CDC_ERR_SHAPE, "step %d outside the %d-step schedule", k, ctx->K);
    CK(op->run(S(s), seq == CDC_SEQ_STEP ? k : 0, nullptr));  // (the codec sequences run as run_ops runs them: k = 0)
    return CDC_OK;
}

int cdc_num_step_ops(cdc_ctx* ctx) { return cdc_seq_num_ops(ctx, CDC_SEQ_STEP); }
const char* cdc_step_op_name(cdc_ctx* ctx, int i) { return cdc_seq_op_name(ctx, CDC_SEQ_STEP, i); }
double cdc_step_op_flops(cdc_ctx* ctx, int i) { return cdc_seq_op_flops(ctx, CDC_SEQ_STEP, i); }
double cdc_step_op_bytes(cdc_ctx* ctx, int i) { return cdc_seq_op_bytes(ctx, CDC_SEQ_STEP, i); }
int cdc_step_op_describe(cdc_ctx* ctx, int i, cdc_step_op_desc* out) { return cdc_seq_op_describe(ctx, CDC_SEQ_STEP, i, out); }
int cdc_run_step_op(cdc_ctx* ctx, int i, int k, cdc_stream s) { return cdc_run_seq_op(ctx, CDC_SEQ_STEP, i, k, s); }

#ifdef CDC_TOOLS
// Tools build only: leave a class of ops out of the captured graph (0 = none, 1 = the tcgen05 convs, 2 = the
// elementwise / GroupNorm kernels, 3 = attention), so that a class's in-graph cost is the difference of two replay
// times.  The decoded image is garbage while a class is skipped: cdc_get_x / cdc_decode_host refuse to return it.
int cdc_debug_graph_skip(cdc_ctx* ctx, int op_class) {
    if (!ctx || op_class < 0 || op_class > 3) return CDC_ERR_SHAPE;
    if (op_class != ctx->graph_skip) drop_graph(ctx);
    ctx->graph_skip = op_class;
    return CDC_OK;
}
#endif

// Per-op device time of one denoise step, measured in stream order: all ops are enqueued back to back with an event
// between consecutive launches (the host stays ahead of the GPU, so the differences are the ops' in-stream durations
// including the inter-kernel gap), after `warm` untimed steps.
int cdc_profile_step(cdc_ctx* ctx, int k, int warm, float* us_out, cdc_stream s) {
    NEED_PLAN();
    if (k < 0 || k >= ctx->K || !us_out) return ctx->fail(CDC_ERR_SHAPE, "bad step index / output");
    const size_t n = ctx->step_seq.ops.size();
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) CK(cudaEventCreate(&e));
    for (int w = 0; w < warm; ++w)
        for (Op& op : ctx->step_seq.ops) CK(op.run(S(s), k, nullptr));
    CK(cudaEventRecord(ev[0], S(s)));
    for (size_t i = 0; i < n; ++i) {
        CK(ctx->step_seq.ops[i].run(S(s), k, nullptr));
        CK(cudaEventRecord(ev[i + 1], S(s)));
    }
    CK(cudaStreamSynchronize(S(s)));
    for (size_t i = 0; i < n; ++i) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
        us_out[i] = ms * 1e3f;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return CDC_OK;
}

// In-graph timing (include/cdc_b200_tools.h): the same captured K-step loop, every kernel stamping
// (earliest CTA start, latest CTA end) in globaltimer ns into its own slot.
int cdc_profile_graph(cdc_ctx* ctx, int reps, float* start_us, float* dur_us, cdc_stream s) {
    NEED_PLAN();
    if (ctx->K < 1) return ctx->fail(CDC_ERR_STATE, "call cdc_set_schedule first");
    if (reps < 1 || reps > 64 || !start_us || !dur_us) return ctx->fail(CDC_ERR_SHAPE, "reps must be in 1..64, outputs non-null");
    const size_t nops = ctx->step_seq.ops.size(), n = static_cast<size_t>(ctx->K) * nops;
    long long* dev = nullptr;
    CK(cudaMalloc(&dev, n * 2 * sizeof(long long)));
    std::vector<long long> init(n * 2), got(n * 2);
    for (size_t i = 0; i < n; ++i) {
        init[2 * i] = -1;  // = ~0 as unsigned: atomicMin target
        init[2 * i + 1] = 0;
    }
    cudaGraphExec_t gx = nullptr;
    int r = capture_graph(ctx, &gx, dev);
    if (r) {
        cudaFree(dev);
        return r;
    }
    std::vector<std::vector<float>> st(n), du(n);
    cudaError_t e = cudaSuccess;
    for (int it = 0; it <= reps && e == cudaSuccess; ++it) {  // replay 0 is the warm-up
        e = cudaMemcpyAsync(dev, init.data(), n * 16, cudaMemcpyHostToDevice, S(s));
        if (e == cudaSuccess) e = cudaGraphLaunch(gx, S(s));
        if (e == cudaSuccess) e = cudaMemcpyAsync(got.data(), dev, n * 16, cudaMemcpyDeviceToHost, S(s));
        if (e == cudaSuccess) e = cudaStreamSynchronize(S(s));
        if (e != cudaSuccess || it == 0) continue;
        unsigned long long t0 = ~0ull;
        for (size_t i = 0; i < n; ++i)
            if (got[2 * i + 1] != 0 && static_cast<unsigned long long>(got[2 * i]) < t0) t0 = static_cast<unsigned long long>(got[2 * i]);
        for (size_t i = 0; i < n; ++i) {
            const bool ran = got[2 * i + 1] != 0;
            st[i].push_back(ran ? static_cast<float>(static_cast<double>(static_cast<unsigned long long>(got[2 * i]) - t0) * 1e-3) : 0.0f);
            du[i].push_back(ran ? static_cast<float>(static_cast<double>(got[2 * i + 1] - got[2 * i]) * 1e-3) : 0.0f);
        }
    }
    cudaGraphExecDestroy(gx);
    cudaFree(dev);
    if (e != cudaSuccess) return ctx->fail(CDC_ERR_CUDA, "cdc_profile_graph: %s", cudaGetErrorString(e));
    auto median = [](std::vector<float>& v) {
        std::sort(v.begin(), v.end());
        return v.empty() ? 0.0f : v[v.size() / 2];
    };
    for (size_t i = 0; i < n; ++i) {
        start_us[i] = median(st[i]);
        dur_us[i] = median(du[i]);
    }
    return CDC_OK;
}

// ---- stateless integer path (runs on the CURRENT device: the pointers' device) ----
static int dev_sms() {
    int dev = 0, n = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
}

int cdc_quantize(const float* y, const float* mu, int32_t* q, float* y_hat, int64_t n, int64_t mu_inner, int64_t mu_mod,
                 cdc_stream s) {
    if (n < 0 || (n > 0 && (!y || !mu || !q))) return CDC_ERR_SHAPE;
    if (mu_mod && mu_inner < 1) return CDC_ERR_SHAPE;
    return launch_quantize(y, mu, q, y_hat, n, mu_inner, mu_mod, dev_sms(), S(s)) == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}

int cdc_cdf_lookup(const int32_t* q, const float* sigma, const int32_t* cdf, const int32_t* row_start,
                   const int32_t* cdf_length, const int32_t* offset, const float* scale_table, int rows, int64_t inner,
                   int32_t* idx, int32_t* v, int32_t* lo, int32_t* hi, int32_t* raw, int64_t n, cdc_stream s) {
    if (n < 0 || rows < 1 || rows > 256 || (!sigma && inner < 1)) return CDC_ERR_SHAPE;
    if (n > 0 && (!q || !cdf || !row_start || !cdf_length || !offset || !idx || !v || !lo || !hi || !raw)) return CDC_ERR_SHAPE;
    CdfTables t{cdf, row_start, cdf_length, offset, scale_table, rows};
    return launch_cdf_lookup(q, sigma, t, inner, idx, v, lo, hi, raw, n, dev_sms(), S(s)) == cudaSuccess ? CDC_OK
                                                                                                        : CDC_ERR_CUDA;
}

// ---- rANS bitstream (stateless; runs on the CURRENT device) ----
int cdc_rans_streams_per_channel(int64_t hw) {
    int s = 1;
    const int64_t lim = hw / 64 > 1 ? hw / 64 : 1;
    while (2 * s <= lim && s < 32) s *= 2;
    return s;
}
int64_t cdc_rans_scratch_bytes(int64_t n_chan, int64_t hw, int spc) {
    return (n_chan < 1 || hw < 1 || spc < 1) ? -1 : rans_scratch_bytes(n_chan, hw, spc);
}
int64_t cdc_rans_max_bytes(int64_t n_chan, int64_t hw, int spc) {
    return (n_chan < 1 || hw < 1 || spc < 1) ? -1 : rans_max_bytes(n_chan, hw, spc);
}
int cdc_rans_encode(const int32_t* idx, const int32_t* v, const int32_t* lo, const int32_t* hi, const int32_t* raw,
                    const int32_t* cdf_length, int64_t n_chan, int64_t hw, int spc, void* scratch, uint8_t* out, int64_t out_capacity,
                    uint64_t* out_bytes_dev, cdc_stream s) {
    if (!idx || !v || !lo || !hi || !raw || !cdf_length || !scratch || !out || !out_bytes_dev) return CDC_ERR_SHAPE;
    if (n_chan < 1 || hw < 1 || spc < 1 || spc > 32 || n_chan * spc > (1LL << 30) || hw > (1LL << 31) - 1) return CDC_ERR_SHAPE;
    if (out_capacity < rans_max_bytes(n_chan, hw, spc)) return CDC_ERR_SHAPE;
    return launch_rans_encode(idx, v, lo, hi, raw, cdf_length, n_chan, hw, spc, scratch, out,
                              reinterpret_cast<unsigned long long*>(out_bytes_dev), S(s)) == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}
int cdc_rans_decode(const uint8_t* data, int64_t data_bytes, const int32_t* idx, const int32_t* cdf, const int32_t* row_start,
                    const int32_t* cdf_length, const int32_t* offset, int rows, int64_t n_chan, int64_t hw, int spc, void* scratch,
                    int32_t* q, int32_t* status_dev, cdc_stream s) {
    if (!data || !idx || !cdf || !row_start || !cdf_length || !offset || !scratch || !q || !status_dev) return CDC_ERR_SHAPE;
    if (rows < 1 || n_chan < 1 || hw < 1 || spc < 1 || spc > 32 || data_bytes < 24 + 4 * n_chan * spc) return CDC_ERR_SHAPE;
    CdfTables t{cdf, row_start, cdf_length, offset, nullptr, rows};
    return launch_rans_decode(data, data_bytes, idx, t, n_chan, hw, spc, scratch, q, status_dev, S(s)) == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}

// ---- single-op entry points for kernel-level parity tests ----
int cdc_test_conv(int device, const void* src0, int c0, const void* src1, int c1, int B, int H, int W,
                  const float* w_oihw, const float* bias, int cout, int ksize, int mode, int force_bn,
                  const void* residual, void* out, int64_t* gn_sums, cdc_stream s) {
    cdc_ctx tmp;
    cdc_ctx* ctx = &tmp;
    DevGuard guard(device);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        g_create_err = "not an sm_100 device";
        return CDC_ERR_ARCH;
    }
    if (configure_conv_kernels() != cudaSuccess || configure_kf_kernels() != cudaSuccess) {
        g_create_err = "cudaFuncSetAttribute(conv kernels) failed";
        return CDC_ERR_CUDA;
    }
    Arena ar;
    ConvW cw;
    const int cin = c0 + c1;
    // (the nearest-x2 parity weights are pre-summed from 3x3 weights: build_conv refuses a nearest-x2 conv of another size)
    int r = make_conv_w(ctx, ar, w_oihw, bias, cout, cin, ksize, cin, cin, false, &cw, S(s), mode == MODE_UP2 && ksize == 3);
    if (r) {
        g_create_err = tmp.err;
        ar.release();
        return r;
    }
    ConvBuild cb;
    cb.name = "test_conv";
    Act a0;
    a0.p = static_cast<act_t*>(const_cast<void*>(src0));
    a0.C = c0;
    a0.H = H;
    a0.W = W;
    cb.srcs.push_back(a0);
    if (src1) {
        Act a1 = a0;
        a1.p = static_cast<act_t*>(const_cast<void*>(src1));
        a1.C = c1;
        cb.srcs.push_back(a1);
    }
    cb.w = &cw;
    cb.mode = mode;
    cb.ksize = ksize;
    cb.out.p = static_cast<act_t*>(out);
    cb.out.C = cw.n_pad;
    cb.out.H = mode == MODE_S2 ? H / 2 : (mode == MODE_UP2 ? 2 * H : H);
    cb.out.W = mode == MODE_S2 ? W / 2 : (mode == MODE_UP2 ? 2 * W : W);
    cb.residual = static_cast<const act_t*>(residual);
    cb.force_bn = force_bn;
    if (gn_sums) {
        cb.epi = EPI_STATS;
        cb.cpg = cout / 32;
        cb.gn_acc = reinterpret_cast<gn_sum_t*>(gn_sums);
    }
    Op op;
    std::string e;
    r = build_conv(cb, B, prop.multiProcessorCount, tmp.opts, &op, &e);
    if (r) {
        g_create_err = e;
        ar.release();
        return r;
    }
    cudaError_t ce = op.run(S(s), 0, nullptr);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(S(s));
#ifdef CDC_TOOLS
    if (ce == cudaSuccess && getenv("CDC_TEST_CONV_REPS")) {  // tools/conv_bench.py: device time of the conv launch alone
        const int reps = atoi(getenv("CDC_TEST_CONV_REPS"));
        void* flush = nullptr;
        const size_t fb = 256u << 20;  // > L2
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        float tot = 0.f, tmin = 1e30f;
        if (cudaMalloc(&flush, fb) == cudaSuccess) {
            for (int i = 0; i < reps && ce == cudaSuccess; ++i) {
                cudaMemsetAsync(flush, i, fb, S(s));
                cudaEventRecord(e0, S(s));
                ce = op.run(S(s), 0, nullptr);
                cudaEventRecord(e1, S(s));
                cudaStreamSynchronize(S(s));
                float ms = 0.f;
                cudaEventElapsedTime(&ms, e0, e1);
                tot += ms;
                tmin = ms < tmin ? ms : tmin;
            }
            cudaFree(flush);
            printf("conv_bench: %s mean %.2f us min %.2f us over %d flushed runs, %.1f TFLOP/s (mean)\n", op.name.c_str(), 1e3 * tot / reps,
                   1e3 * tmin, reps, op.flops / (tot / reps * 1e-3) / 1e12);
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    }
#endif
    ar.release();
    if (ce != cudaSuccess) {
        g_create_err = std::string("test_conv: ") + cudaGetErrorString(ce);
        return CDC_ERR_CUDA;
    }
    return CDC_OK;
}

int cdc_test_attention(const void* qkv, void* out, int B, int N, int heads, cdc_stream s) {
    if (!qkv || !out || B < 1 || N < 1 || heads < 1) return CDC_ERR_SHAPE;
    if (configure_attention_tc() != cudaSuccess) return CDC_ERR_CUDA;
    AttnTcParams ap;
    memset(&ap, 0, sizeof ap);
    if (encode_qkv_map(&ap.qkv_map, static_cast<const act_t*>(qkv), 3 * heads * 64, N, B)) return CDC_ERR_CUDA;
    ap.out = static_cast<act_t*>(out);
    ap.N = N;
    ap.heads = heads;
    return launch_attention_tc(ap, B, S(s)) == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}

int cdc_test_gn(const void* x, const void* r, void* y, const float* gamma, const float* beta, const float* film, int B,
                int HW, int C, int silu, float eps, cdc_stream s) {
    gn_sum_t* acc = nullptr;
    if (cudaMalloc(&acc, static_cast<size_t>(B) * kGnImgStride * sizeof(gn_sum_t)) != cudaSuccess) return CDC_ERR_CUDA;
    cudaError_t e = cudaMemsetAsync(acc, 0, static_cast<size_t>(B) * kGnImgStride * sizeof(gn_sum_t), S(s));
    if (e == cudaSuccess) e = launch_gn_stats(static_cast<const act_t*>(x), acc, B, HW, C, S(s));
    if (e == cudaSuccess)
        e = launch_gn_apply(static_cast<const act_t*>(x), acc, gamma, beta, film, eps, static_cast<const act_t*>(r),
                            static_cast<act_t*>(y), B, HW, C, silu, dev_sms(), S(s));
    if (e == cudaSuccess) e = cudaStreamSynchronize(S(s));
    cudaFree(acc);
    return e == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}

// ---- the byte-boundary kernels of cdc_compress_rgb8 / cdc_decompress_rgb8, alone ----
int cdc_test_scale_rows(const void* sigma_act, int ldc, int c_off, float min_sigma, const float* scale_table, int32_t* idx, int B,
                        int C, int HW, cdc_stream s) {
    if (!sigma_act || !scale_table || !idx || B < 1 || C < 1 || HW < 1 || c_off < 0 || ldc < c_off + C) return CDC_ERR_SHAPE;
    return launch_scale_rows(static_cast<const act_t*>(sigma_act), ldc, c_off, min_sigma, scale_table, idx, B, C, HW, S(s)) == cudaSuccess
               ? CDC_OK
               : CDC_ERR_CUDA;
}

int cdc_test_dequant(const int32_t* q, const float* mu_vec, const void* mu_act, int mu_ldc, void* dst, int B, int C, int HW,
                     cdc_stream s) {
    if (!q || !dst || !mu_vec == !mu_act || B < 1 || C < 1 || HW < 1 || (mu_act && mu_ldc < C)) return CDC_ERR_SHAPE;
    return launch_dequant_to_act(q, mu_vec, static_cast<const act_t*>(mu_act), mu_ldc, static_cast<act_t*>(dst), B, C, HW, S(s)) ==
                   cudaSuccess
               ? CDC_OK
               : CDC_ERR_CUDA;
}

int cdc_test_rgb8_in(const uint8_t* rgb, void* dst64, int64_t npix, cdc_stream s) {
    if (!rgb || !dst64 || npix < 16 || npix % 16 || (reinterpret_cast<uintptr_t>(rgb) & 15u)) return CDC_ERR_SHAPE;
    return launch_rgb8_in(rgb, static_cast<act_t*>(dst64), npix, S(s)) == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}

int cdc_test_rgb8_out(const float* xs, uint8_t* rgb, int64_t npix, cdc_stream s) {
    if (!xs || !rgb || npix < 16 || npix % 16 || ((reinterpret_cast<uintptr_t>(xs) | reinterpret_cast<uintptr_t>(rgb)) & 15u))
        return CDC_ERR_SHAPE;
    return launch_rgb8_out(xs, rgb, npix, S(s)) == cudaSuccess ? CDC_OK : CDC_ERR_CUDA;
}

}  // extern "C"
