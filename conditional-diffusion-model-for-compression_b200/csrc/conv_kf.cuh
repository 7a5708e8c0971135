// Parameter block of the kh-fused strip conv (conv_kf.cu): 3x3 / stride 1, resident weights.
#pragma once
#include "conv_tc.cuh"

namespace cdc {

struct alignas(64) KfParams {
    CUtensorMap amap[4];  // activation sources, box {64 ch, 130 px, 1 row, 1 image}; mode 2: (even, odd)-pixel views per source
    CUtensorMap wmap;     // weights [n_pad][9 * CH * 64] K-major, box {64, BN}
    CUtensorMap omap;     // output, box {BN ch, 128 px, 1 row, 1 image} (staged TMA store only)
    CUtensorMap rmap;     // fused 1x1 residual conv: its weights [n_pad][CH * 64] K-major, box {64, BN}
    int chunks0;          // 64-channel chunks that come from source 0 (the rest from source 1)
    int tr;               // 1: transposed walk -- kernel rows = image columns, kernel pixels = image rows (H, W below are
                          // the kernel-space extents); tensor maps, weight taps and output addressing are swapped to match
    int H, W, batch;      // INPUT grid (mode 1: the low-resolution tensor; the output is 2H x 2W)
    int nseg;             // ceil(W / 128) column segments
    int S;                // strips per column (rows are spread evenly over them)
    int slot0;            // 1: every strip starts at logical accumulator slot 0, however many strips its CTA ran before
                          // (the aliased rings' sums then do not depend on the grid: batch-invariant plans)
    int NS;               // input-row ring slots
    int n_tiles;          // N tiles (mode 1: channel tiles x 4 parities); every CTA keeps ONE tile's weights resident
    int G1;               // CTAs per N tile (grid = n_tiles * G1)
    int ldc;              // channels of the output tensor
    act_t* out;
    const float* bias;    // [n_tiles * BN]
    act_t* res_out;       // fused 1x1 residual conv (same input, centre tap only): output tensor, channels, bias
    int res_ldc;
    const float* res_bias;
    gn_sum_t* gn_acc;     // EPI_STATS: [batch][32][kGnVals] fixed-point accumulators (gn_sums.cuh), zero on entry
    // APPLY: the input is the raw output of the preceding conv; GroupNorm (+ FiLM) + SiLU of THAT conv's statistics is
    // applied to every input row in shared memory before the MMAs read it (replaces a gn_apply_kernel pass over HBM)
    const gn_sum_t* in_acc;   // [batch][32][kGnVals] totals of the input tensor (complete: written by the preceding kernel)
    const float* in_gamma;    // [C_in]
    const float* in_beta;
    const float* in_film;     // [2 * C_in] (scale | shift) of this step, or null
    float in_eps;
    float* x;             // EPI_DDIM (see ConvParams)
    act_t* xpad;
    float* x0_out;
    float c0, c1;
    float e0, e1, sg;     // generalised sampler update (see ConvParams)
    unsigned long long seed;
    int step;
    const unsigned long long* img_seeds;  // (see ConvParams)
    long long* stamp;     // diagnostics, may be null (see ConvParams)
    unsigned int* sat;
};

// mode 0: 3x3 conv; mode 1: nearest-x2 upsample + 3x3 conv (four parity 2x2 convs on the low-resolution input);
// mode 2: 3x3 conv with stride 2 (H, W of KfParams are the OUTPUT grid)
// res: the ResBlock's 1x1 residual conv rides along (its weights are resident too, its accumulators share TMEM)
// apply: GroupNorm + SiLU of the input applied in shared memory (see in_acc)
bool kf_inst_ok(int bn, int cpg, int epi, int CH, int mode, bool res, bool apply = false);
bool kf_plan(int bn, int CH, int mode, bool res, int* NS, bool* staged);  // shared-memory plan; false if the weights do not fit
int kf_smem_bytes(int bn, int CH, int NS, bool staged, int mode, bool res);
cudaError_t configure_kf_kernels();
cudaError_t launch_conv_kf(const KfParams& p, int bn, int cpg, int epi, int CH, bool xk16, int mode, bool res, bool apply,
                           bool staged, cudaStream_t stream);  // xk16: chunk 0 has 16 real channels (stem)

}  // namespace cdc
