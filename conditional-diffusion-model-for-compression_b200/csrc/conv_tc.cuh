// Parameter block of the tcgen05 implicit-GEMM convolution (K-conv, SURVEY.md 2.2 C3/C4/C9).
// One kernel covers conv3x3 / conv1x1, stride 1 / stride 2 / nearest-x2-input, single or
// dual (virtually concatenated) source, through a host-built table of K-blocks: each entry
// names an activation tensor map, a pixel shift and a channel offset, plus the K offset of the
// matching 64-wide slice of the [C_out][K] weight matrix.
#pragma once
#include <cuda.h>
#include "act.cuh"
#include <cuda_runtime.h>
#include <stdint.h>

#include "gn_sums.cuh"

namespace cdc {

constexpr int kMaxMaps = 8;      // activation tensor maps per launch (2 sources x 4 stride-2 phases)
constexpr int kMaxKBlocks = 144; // 4 output phases x 36 (nearest-x2 conv, C_in 256) or 1 x 72

struct KBlock {
    int8_t map;    // index into ConvParams::amap
    int8_t dw;     // pixel shift along W applied to the tile origin
    int8_t dh;     // pixel shift along H
    int8_t pad;
    uint16_t c0;   // first channel of the 64-channel slice inside that source
    uint16_t wk;   // K offset into the weight matrix row
};

enum ConvEpilogue : int {
    EPI_STORE = 0,  // +bias (+bf16 residual) -> act_t NHWC
    EPI_STATS = 1,  // EPI_STORE and per-(image, group) sum / sum-of-squares for GroupNorm (integer atomics)
    EPI_DDIM = 2,   // final conv: x0 = acc+bias; x_prev = c0*clamp(x0) + c1*x_t (fp32), act_t copy for the stem
};

struct alignas(64) ConvParams {
    CUtensorMap amap[kMaxMaps];
    CUtensorMap wmap;
    KBlock kb[kMaxKBlocks];
    int nkb;        // K-blocks per output tile
    int nphase;     // 1, or 4 for nearest-x2-input convs (output parity classes)
    int tiles_w, tiles_h, batch;
    int bw_log2;    // tile = (128 >> bw_log2) rows x (1 << bw_log2) columns of the tile grid
    int gw, gh;     // tile-grid extent (pixels) per phase, for masking
    int OH, OW;     // output tensor spatial size
    int os;         // output pixel = grid pixel * os + phase offset (1, or 2 with nphase 4)
    int ldc;        // channels of the output tensor (row pitch in elements)
    int n_total;    // true C_out rounded up to the N tile
    int n_tiles;    // n_total / BN
    act_t* out;
    const float* bias;                 // [n_total]
    const act_t* residual;     // optional, same layout as out
    gn_sum_t* gn_acc;                  // EPI_STATS: [batch][32][kGnVals] fixed-point accumulators (gn_sums.cuh), zero on entry
    // EPI_DDIM
    float* x;                          // [B*H*W][3] fp32, updated in place
    act_t* xpad;               // [B*H*W][64] bf16, channels 0..2 rewritten
    float* x0_out;                     // optional [B*H*W][3] raw x0_hat
    float c0, c1;
    // generalised sampler update (oracle/sampler.py ddim_update): x0 = e0*x_t + e1*out; x_prev = c0*clamp(x0) + c1*x_t + sg*z
    // (X-parameterised deterministic DDIM: e0 = 0, e1 = 1, sg = 0); z = Philox noise of (seed, step, pixel) -- sampler.cuh
    float e0, e1, sg;
    unsigned long long seed;
    int step;
    const unsigned long long* img_seeds;  // per-image seed block (kernels.cuh ImageSeeds), or null: read only when sg != 0
    // diagnostics (either may be null): [0] = earliest CTA start, [1] = latest CTA end (globaltimer ns, atomic min / max);
    // number of (thread, tile) epilogue passes that met a value beyond the fp16 range (stored saturated)
    long long* stamp;
    unsigned int* sat;
    float act_slope;  // EPI_STORE / EPI_STATS: 0 = none; s in (0, 1): LeakyReLU(s) after the bias (hyper-codec convs, oracle/codec.py)
};

// Launches the instantiation for (bn, cpg, epi).  Returns cudaErrorInvalidValue when that
// combination is not compiled.
cudaError_t launch_conv(const ConvParams& p, int bn, int cpg, int epi, int num_sms, cudaStream_t stream);

// Sets the dynamic shared-memory limit of every instantiation (call once, outside graph capture).
cudaError_t configure_conv_kernels();

}  // namespace cdc
