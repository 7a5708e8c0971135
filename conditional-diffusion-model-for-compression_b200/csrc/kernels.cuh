// Launchers of the non-GEMM kernels of the decode hot path (all HBM- or latency-bound).
#pragma once
#include "act.cuh"
#include "gn_sums.cuh"
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cdc {

// ---- GroupNorm (SURVEY.md 2.2 C5/C6; oracle/unet.py RB / Attn) -------------------------------
// Statistics are fixed-point integer accumulators [B][32 groups][2] (gn_sums.cuh), zero on entry, filled by the conv
// epilogues or by gn_stats (where the producer is not a conv: attention input).
cudaError_t launch_gn_stats(const act_t* x, gn_sum_t* acc, int B, int HW, int C, cudaStream_t s, long long* stamp = nullptr);
// y = act(GN(x) * (1 + film_scale) + film_shift) (+ r); act = SiLU if silu != 0; film may be null.  In place allowed.
// The normalisation coefficients are derived from `acc` inside the kernel (no finalize pass).
cudaError_t launch_gn_apply(const act_t* x, const gn_sum_t* acc, const float* gamma, const float* beta, const float* film,
                            float eps, const act_t* r, act_t* y, int B, int HW, int C, int silu, int num_sms, cudaStream_t s,
                            long long* stamp = nullptr, unsigned int* sat = nullptr);

// ---- time embedding + FiLM (C8; oracle/unet.py TimeEmbed, RB.film) ----------------------------
struct FilmLayer {
    const float* w;  // [2C][temb]
    const float* b;  // [2C]
    int c2;          // 2C
    int offset;      // offset of this layer's 2C outputs inside one step's FiLM vector
};
constexpr int kMaxFilm = 24;
struct FilmParams {
    const float* sinus;  // [K][64] sinusoidal embedding per step (host-computed)
    const float *w1, *b1, *w2, *b2;
    FilmLayer layer[kMaxFilm];
    int nlayers, temb, total;  // total floats per step
    float* out;                // [K][total]
};
cudaError_t launch_temb_film(const FilmParams& p, int K, cudaStream_t s);

// ---- layout conversion at the API boundary -----------------------------------------------------
cudaError_t launch_nchw_f32_to_nhwc_act(const float* src, act_t* dst, int B, int C, int HW, int ldc,
                                         cudaStream_t s);
cudaError_t launch_nhwc_act_to_nchw_f32(const act_t* src, float* dst, int B, int C, int HW, cudaStream_t s);
// The stem's first source: the 3-channel sampler state as a 16-bit tensor the conv kernels can TMA.  LOGICALLY 64
// channels (one 64-channel chunk of the stem's K dimension, channels 3..63 zero), PHYSICALLY kXpadC = 16 per pixel
// (32 B = one DRAM sector): its tensor maps declare a channel extent of 16 with the usual 64-channel box, so TMA
// zero-fills channels 16..63 in shared memory without reading them -- 37 MB per step less at 768x512 than the 64-channel
// copy of round 1, and the final conv's epilogue writes whole sectors instead of 8 bytes of each 128-byte pixel.
constexpr int kXpadC = 16;
// x NCHW fp32 [B,3,H,W] -> xs NHWC fp32 [B*HW][3] and xpad act_t [B*HW][kXpadC] (channels 0..2; rest untouched)
cudaError_t launch_x_in(const float* x_nchw, float* xs, act_t* xpad, int B, int HW, cudaStream_t s);
// Per-image seed block of the sampler state (cdc_set_image_seeds): unsigned long long [1 + B], word 0 = 1 while per-image
// mode is on, words 1 .. B = the seed of image b.  The conv epilogue reads it only when the step adds noise (sg != 0).
// init_noise: x_T = gamma * z from the seeds (sampler.cuh, x_T plane) -> xs and xpad, as launch_x_in stores them
cudaError_t launch_init_noise(const unsigned long long* seeds, float* xs, act_t* xpad, float gamma, int B, int HW, cudaStream_t s);
// xs NHWC fp32 -> NCHW fp32, optionally mapped to [0,1]: (clamp(x,-1,1)+1)/2
cudaError_t launch_x_out(const float* xs, float* x_nchw, int B, int HW, int to_image, cudaStream_t s);
// Trajectory recording (cdc_decode_trajectory): base pointers of the caller's NCHW fp32 [slots][B][3][H][W] buffers,
// either may be null.  They live in device memory so that one captured graph serves every call's buffers.
struct TrajPtrs {
    float* x;
    float* x0;
};
// xs -> slot slot_x of dst->x and x0s -> slot slot_x0 of dst->x0 (as launch_x_out, to_image = 0); a negative slot skips
cudaError_t launch_traj_store(const float* xs, const float* x0s, const TrajPtrs* dst, int slot_x, int slot_x0, int B, int HW,
                              cudaStream_t s);
// *dst = {x, x0} in stream order
cudaError_t launch_traj_set_ptrs(TrajPtrs* dst, float* x, float* x0, cudaStream_t s);
// conv weight repack: OIHW fp32 -> [O_pad][taps][I_pad] act_t with input channels >= split moved to split_pad
cudaError_t launch_repack_weight(const float* src, act_t* dst, int O, int I, int taps, int O_pad, int I_pad,
                                 int split, int split_pad, cudaStream_t s);

// ConvTranspose2d(k = 5, stride 2, padding 2, output_padding 1) as four output-parity convs of up to 3x3 taps on the
// input grid: src [I][O][5][5] fp32 (PyTorch layout) -> dst [O_pad][36 = (parity, a, b)][I_pad], missing taps zero
cudaError_t launch_repack_weight_convt5(const float* src, act_t* dst, int O, int I, int O_pad, int I_pad, cudaStream_t s);
// image NCHW fp32 in [0, 1] -> NHWC act_t, 64-channel pixels, channels 0..2 = 2 * img - 1 (channels 3..63 untouched: zero)
cudaError_t launch_img_in(const float* img_nchw, act_t* dst64, int B, int HW, cudaStream_t s);
// 8-bit interleaved RGB [npix][3] (16-byte aligned, npix a multiple of 16) -> img64 channels 0..2 = 2 * (v / 255) - 1,
// the values launch_img_in stores for the fp32 image v / 255
cudaError_t launch_rgb8_in(const uint8_t* rgb, act_t* dst64, long long npix, cudaStream_t s);
// xs NHWC fp32 [npix][3] -> 8-bit RGB [npix][3] = round_half_even(255 * (clamp(x,-1,1)+1)/2) (launch_x_out's to_image value)
cudaError_t launch_rgb8_out(const float* xs, uint8_t* rgb, long long npix, cudaStream_t s);
// q NCHW int32 [B][C][HW] -> NHWC act_t [B][HW][C] = q + mu in fp32, mu = mu_vec[c] (per channel) or channel c of the NHWC
// act_t tensor mu_act with mu_ldc channels per pixel (exactly one of the two)
cudaError_t launch_dequant_to_act(const int32_t* q, const float* mu_vec, const act_t* mu_act, int mu_ldc, act_t* dst, int B, int C,
                                  int HW, cudaStream_t s);
// channels [c_off, c_off + C) of an NHWC act_t tensor with ldc channels -> NCHW fp32, optionally clamped from below
cudaError_t launch_nhwc_slice_to_nchw_f32(const act_t* src, float* dst, int B, int C, int HW, int ldc, int c_off, float min_clamp,
                                          int use_clamp, cudaStream_t s);

// nearest-x2 + conv3x3 folded into 4 parity-specific 2x2 convs: dst [O_pad][16][I_pad] (see elementwise.cu)
cudaError_t launch_repack_weight_up2(const float* src, act_t* dst, int O, int I, int O_pad, int I_pad, cudaStream_t s);

// ---- attention (C7; oracle/unet.py Attn) --------------------------------------------------------
// qkv [B*N][768] act_t (q | k | v, head h = channels 64h..64h+63) -> o [B*N][256] bf16
// (attention.cu, tcgen05): qkv_map = 3-D tensor map {768 cols, N rows, B} of the qkv tensor, box {64, 128, 1},
// 128-byte swizzle (built by the host runtime)
struct alignas(64) AttnTcParams {
    CUtensorMap qkv_map;
    act_t* out;  // [B*N][heads * 64]
    int N, heads;
    long long* stamp;  // diagnostics, may be null (ptx.cuh stamp_begin / stamp_end)
};
cudaError_t configure_attention_tc();
cudaError_t launch_attention_tc(const AttnTcParams& p, int B, cudaStream_t s);

// ---- integer path (C10; oracle/entropy.py) ------------------------------------------------------
cudaError_t launch_quantize(const float* y, const float* mu, int32_t* q, float* yhat, int64_t n, int64_t mu_inner,
                            int64_t mu_mod, int num_sms, cudaStream_t s);
struct CdfTables {
    const int32_t* cdf;
    const int32_t* row_start;
    const int32_t* cdf_length;
    const int32_t* offset;
    const float* scale_table;  // [64] or null when idx comes from the channel
    int rows;
};
cudaError_t launch_cdf_lookup(const int32_t* q, const float* sigma, CdfTables t, int64_t inner, int32_t* idx,
                              int32_t* v, int32_t* lo, int32_t* hi, int32_t* raw, int64_t n, int num_sms,
                              cudaStream_t s);

// idx NCHW [B][C][HW] = the Gaussian CDF row (cdf_lookup's scale-table search) of max(sigma, min_sigma), sigma = channels
// [c_off, c_off + C) of an NHWC act_t tensor with ldc channels per pixel
cudaError_t launch_scale_rows(const act_t* src, int ldc, int c_off, float min_sigma, const float* scale_table, int32_t* idx, int B,
                              int C, int HW, cudaStream_t s);

// ---- rANS bitstream (rans.cu; oracle/rans.py pins the format) -------------------------------------------------
long long rans_scratch_bytes(long long n_chan, long long hw, int spc);
long long rans_max_bytes(long long n_chan, long long hw, int spc);
// symbols (channel-row major, n_chan * hw each) -> container bytes in `out` (device), total size in *out_bytes (device)
cudaError_t launch_rans_encode(const int32_t* idx, const int32_t* v, const int32_t* lo, const int32_t* hi, const int32_t* raw,
                               const int32_t* cdf_length, long long n_chan, long long hw, int spc, void* scratch, uint8_t* out,
                               unsigned long long* out_bytes, cudaStream_t s);
// container bytes (device) + the CDF row of every element -> q; *status (device) = 1 if the container is corrupt / truncated;
// scratch: 8 bytes per stream
cudaError_t launch_rans_decode(const uint8_t* data, long long data_bytes, const int32_t* idx, CdfTables t, long long n_chan, long long hw,
                               int spc, void* scratch, int32_t* q, int32_t* status, cudaStream_t s);

}  // namespace cdc
