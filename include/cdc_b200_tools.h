/* cdc_b200_tools -- test, profiling and A/B entry points of libcdc_b200.so.
 *
 * NOT part of the drop-in boundary (include/cdc_b200.h): nothing here is needed to decode, and nothing here can change
 * what cdc_decode computes.  tests/ and tools/ bind these through ctypes next to the product symbols.
 * (The measurement hook that DOES alter results -- leaving op classes out of the captured graph -- and the environment
 * switches exist only in the separate tools build, libcdc_b200_tools.so, compiled with -DCDC_TOOLS by
 * `csrc/build.sh tools`.)
 * Every op of every sequence the plan builds (the denoise step, the context net, the analysis encoder, the hyper-encoder
 * and the hyper-decoder) can be described and run alone (cdc_seq_*): tests/test_gpu_step_ops.py and
 * tests/test_gpu_codec_ops.py check each one against a float64 reference of that one operation.
 */
#ifndef CDC_B200_TOOLS_H
#define CDC_B200_TOOLS_H

#include "cdc_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- plan options (A/B of planner decisions; set BEFORE cdc_bind_io, a change re-plans at the next bind) ---------- */
typedef enum {
    CDC_OPT_FUSE_APPLY = 0,     /* N tiles a conv may have for the input-GroupNorm fusion; 0 = never fuse.  default 2 */
    CDC_OPT_KF = 1,             /* 0: every conv through the general kernel (conv_tc.cu).  default 1 */
    CDC_OPT_PLAN_SMS = 2,       /* SMs the conv grids and the GroupNorm apply grid are laid out for; 0 (default) or more
                                   than the device has: the device's count.  A test lever: a few SMs put several strips
                                   (and images) on one strip-conv CTA at small shapes */
    CDC_OPT_COUNT = 3
} cdc_plan_option;
int cdc_set_plan_option(cdc_ctx* ctx, int option, int value);

/* ---- per-layer access ------------------------------------------------------------------------------------------- */
/* The op sequences of the bound plan.  The codec sequences exist when their weights were loaded (context.*: CONTEXT;
 * codec.*: ENCODER, HYPER_ENC, HYPER_DEC); they take no schedule. */
typedef enum {
    CDC_SEQ_STEP = 0,       /* one denoise step (cdc_denoise_step) */
    CDC_SEQ_CONTEXT = 1,    /* the context net (cdc_set_latent) */
    CDC_SEQ_ENCODER = 2,    /* the analysis encoder (cdc_encode_analysis) */
    CDC_SEQ_HYPER_ENC = 3,  /* the hyper-encoder (cdc_hyper_encode) */
    CDC_SEQ_HYPER_DEC = 4,  /* the hyper-decoder (cdc_hyper_decode) */
    CDC_SEQ_COUNT = 5
} cdc_seq;
/* An unknown seq fails with CDC_ERR_SHAPE, a sequence whose weights were not loaded with CDC_ERR_WEIGHT (cdc_last_error
 * says which): cdc_seq_num_ops returns that code, cdc_seq_op_name "" and the flops / bytes 0. */
int cdc_seq_num_ops(cdc_ctx* ctx, int seq);
const char* cdc_seq_op_name(cdc_ctx* ctx, int seq, int i);
double cdc_seq_op_flops(cdc_ctx* ctx, int seq, int i);
double cdc_seq_op_bytes(cdc_ctx* ctx, int seq, int i);
/* runs op i of sequence seq alone on s; k is the sampler step (checked against the schedule for CDC_SEQ_STEP only, the
 * other sequences ignore it) */
int cdc_run_seq_op(cdc_ctx* ctx, int seq, int i, int k, cdc_stream s);
/* the same for CDC_SEQ_STEP */
int cdc_num_step_ops(cdc_ctx* ctx);
const char* cdc_step_op_name(cdc_ctx* ctx, int i);
double cdc_step_op_flops(cdc_ctx* ctx, int i);
double cdc_step_op_bytes(cdc_ctx* ctx, int i);
int cdc_run_step_op(cdc_ctx* ctx, int i, int k, cdc_stream s);

/* Read-only description of op i of a sequence of the bound plan: what it computes, from which tensors into which, and which
 * kernel instantiation runs it.  Metadata recorded when the plan was built; reading it changes nothing. */
typedef enum {
    CDC_OPK_MEMSET = 0,     /* clears the step's GroupNorm accumulator slots (gn_out_acc, gn_slots of them) */
    CDC_OPK_CONV = 1,
    CDC_OPK_GN_STATS = 2,   /* GroupNorm statistics of src[0] into gn_out_acc */
    CDC_OPK_GN_APPLY = 3,   /* out = act(GroupNorm(src[0]; gn_in_acc) [* (1 + s) + sh]) [+ residual] */
    CDC_OPK_ATTENTION = 4   /* out = softmax(q k^T / 8) v per head, src[0] = qkv [B][HW][3C] */
} cdc_op_kind;
typedef struct {
    void* p;  /* NHWC 16-bit activation; NULL: not used */
    int C, Cphys, H, W;  /* Cphys: channels stored per pixel (the stem's x_t copy stores fewer than its C) */
} cdc_tensor_desc;
typedef struct {
    int kind;            /* cdc_op_kind */
    char weight[64];     /* parameter prefix of the conv / GroupNorm ("down.0.rb1.conv2", "mid.attn.gn", "final") or "" */
    char res_weight[64]; /* 1x1 residual conv computed in the same launch ("down.1.rb1.res") or "" */
    char in_gn[64];      /* GroupNorm + SiLU applied to the conv's input rows ("down.0.rb1.gn1") or "" */
    int film_off;        /* offset of the (scale | shift) FiLM pair in a step's FiLM vector (cdc_get_film), -1: none */
    int mode, ksize, epi, silu;  /* conv: mode 0 stride 1, 1 stride 2, 2 nearest-x2 input, 3 transposed 5x5 stride 2
                                    (ConvTranspose2d(5, stride 2, padding 2, output_padding 1), weight [in][out][5][5]);
                                    epi 0 store, 1 GroupNorm statistics, 2 sampler update (final conv); gn_apply: silu */
    int kernel;          /* conv: 1 = conv_tc.cu (general), 2 = conv_kf.cu (strip); 0 otherwise */
    int bn, cpg, ch, staged, xk16, tr, res1, apply;  /* the instantiation / walk that runs (ch: 64-channel input chunks) */
    cdc_tensor_desc src[2], residual, out, res_out;
    void* gn_in_acc;     /* GroupNorm accumulator slot read ([B][32][4] int64, csrc/gn_sums.cuh) or NULL */
    void* gn_out_acc;    /* slot accumulated into (memset: first slot cleared) or NULL */
    int gn_slots;        /* memset: slots cleared */
    float* x;            /* final conv: sampler state, NHWC fp32 [B][H][W][3], read as x_t and overwritten with x_prev */
    float* x0_out;       /* final conv: x0 estimate, NHWC fp32 */
    void* xpad;          /* final conv: the stem's 16-bit x_t copy, rewritten with x_prev */
    float act_slope;     /* conv: LeakyReLU slope applied after the bias (the hyper networks' 0.2), 0: none */
    /* conv launch geometry.  conv_kf.cu: n_tiles N tiles (output-parity tiles included) of g1 CTAs each; the kernel-space
     * grid (image rows, or image columns for the transposed walk) has `rows` rows, split into nseg 128-pixel segment
     * columns per image and `strips` strips per column; CTA c of a tile runs the units (image, segment, strip)
     * u = c, c + g1, ... < B * nseg * strips.  conv_tc.cu: n_tiles output tiles (N tiles x phases x images x pixel
     * tiles) over `grid` persistent CTAs (g1, nseg, strips, rows 0).  grid: CTAs launched (both kernels). */
    int n_tiles, g1, nseg, strips, rows, grid;
} cdc_step_op_desc;
int cdc_seq_op_describe(cdc_ctx* ctx, int seq, int i, cdc_step_op_desc* out);
int cdc_step_op_describe(cdc_ctx* ctx, int i, cdc_step_op_desc* out);  /* CDC_SEQ_STEP */
/* in-stream device time (microseconds) of every op of step k, after `warm` untimed steps; us_out[cdc_num_step_ops] */
int cdc_profile_step(cdc_ctx* ctx, int k, int warm, float* us_out, cdc_stream s);
/* In-graph timing: captures the same K-step graph with every kernel writing (earliest CTA start, latest CTA end) in
 * globaltimer nanoseconds, replays it `reps` times after one warm replay, and returns per op of every step the MEDIAN
 * over the replays of start (relative to the first kernel of the replay) and duration, in microseconds:
 * start_us / dur_us [steps][cdc_num_step_ops] (the memset node reports 0).  x / cond must be bound.  Synchronises. */
int cdc_profile_graph(cdc_ctx* ctx, int reps, float* start_us, float* dur_us, cdc_stream s);

/* ---- single-op entry points for kernel-level parity tests --------------------------------------------------------- */
/* conv: x NHWC 16-bit (cdc_act_dtype) sources (1 or 2), w OIHW fp32 (device), bias fp32; mode 0 = stride 1,
 * 1 = stride 2, 2 = nearest-x2 input; out NHWC 16-bit; gn_sums (optional, ZERO on entry): GroupNorm statistics of the
 * output, [B][32 groups][4] int64 = (sum * 2^20, (squares mod 1024) * 2^20, floor(squares / 1024), 0)
 * (csrc/gn_sums.cuh). */
int cdc_test_conv(int device, const void* src0, int c0, const void* src1, int c1, int B, int H, int W,
                  const float* w_oihw, const float* bias, int cout, int ksize, int mode, int force_bn,
                  const void* residual, void* out, int64_t* gn_sums, cdc_stream s);
int cdc_test_attention(const void* qkv, void* out, int B, int N, int heads, cdc_stream s);
int cdc_test_gn(const void* x, const void* r, void* y, const float* gamma, const float* beta, const float* film,
                int B, int HW, int C, int silu, float eps, cdc_stream s);
/* The byte-boundary kernels of cdc_compress_rgb8 / cdc_decompress_rgb8, each alone on device buffers (no context;
 * CDC_ERR_SHAPE on bad arguments):
 *   scale_rows: idx NCHW int32 [B][C][HW] = the CDF row of max(sigma, min_sigma), sigma = channels [c_off, c_off + C) of
 *               the NHWC 16-bit sigma_act (ldc channels per pixel); scale_table fp32 [64]
 *   dequant:    dst NHWC 16-bit [B][HW][C] = 16-bit of float(q) + mu, q NCHW int32; mu = mu_vec[c] (fp32 [C]) or channel c of
 *               the NHWC 16-bit mu_act (mu_ldc channels per pixel): exactly one of the two
 *   rgb8_in:    8-bit interleaved RGB [npix][3] (16-byte aligned) -> channels 0..2 of dst64 (64 channels per pixel) =
 *               16-bit of 2 * (v / 255) - 1, channel 3 = 0, channels 4..63 untouched; npix a multiple of 16
 *   rgb8_out:   xs fp32 [npix][3] -> rgb [npix][3] = round_half_even(255 * (clamp(x, -1, 1) + 1) / 2); both 16-byte
 *               aligned, npix a multiple of 16 */
int cdc_test_scale_rows(const void* sigma_act, int ldc, int c_off, float min_sigma, const float* scale_table, int32_t* idx, int B,
                        int C, int HW, cdc_stream s);
int cdc_test_dequant(const int32_t* q, const float* mu_vec, const void* mu_act, int mu_ldc, void* dst, int B, int C, int HW,
                     cdc_stream s);
int cdc_test_rgb8_in(const uint8_t* rgb, void* dst64, int64_t npix, cdc_stream s);
int cdc_test_rgb8_out(const float* xs, uint8_t* rgb, int64_t npix, cdc_stream s);

#ifdef CDC_TOOLS
/* tools build only: leave a class of ops out of the captured graph (0 none, 1 tcgen05 convs, 2 elementwise/GroupNorm,
 * 3 attention); while a class is skipped cdc_get_x / cdc_decode_host fail with CDC_ERR_STATE (the image is garbage) */
int cdc_debug_graph_skip(cdc_ctx* ctx, int op_class);
#endif

#ifdef __cplusplus
}
#endif
#endif /* CDC_B200_TOOLS_H */
