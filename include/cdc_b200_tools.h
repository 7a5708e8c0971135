/* cdc_b200_tools -- test, profiling and A/B entry points of libcdc_b200.so.
 *
 * NOT part of the drop-in boundary (include/cdc_b200.h): nothing here is needed to decode, and nothing here can change
 * what cdc_decode computes.  tests/ and tools/ bind these through ctypes next to the product symbols.
 * (The measurement hooks that DO alter results -- leaving op classes out of the captured graph, environment switches,
 * the mma.sync attention kernel -- exist only in the separate tools build, libcdc_b200_tools.so, compiled with
 * -DCDC_TOOLS by `csrc/build.sh tools`.)
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
    CDC_OPT_KF_S2 = 2,          /* 0: stride-2 convs through the general kernel.  default 1 */
    CDC_OPT_KF_MIN_PIXELS = 3,  /* levels with fewer pixels per image use the general kernel.  default 0 */
    CDC_OPT_KF_RING = 4,        /* input-ring slots of the one-chunk strip convs.  default 6 */
    CDC_OPT_COUNT = 5
} cdc_plan_option;
int cdc_set_plan_option(cdc_ctx* ctx, int option, int value);

/* ---- per-layer access ------------------------------------------------------------------------------------------- */
int cdc_num_step_ops(cdc_ctx* ctx);
const char* cdc_step_op_name(cdc_ctx* ctx, int i);
double cdc_step_op_flops(cdc_ctx* ctx, int i);
double cdc_step_op_bytes(cdc_ctx* ctx, int i);
int cdc_run_step_op(cdc_ctx* ctx, int i, int k, cdc_stream s);

/* Read-only description of step op i of the bound plan: what it computes, from which tensors into which, and which
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
    int mode, ksize, epi, silu;  /* conv: mode 0 stride 1, 1 stride 2, 2 nearest-x2 input; epi 0 store, 1 GroupNorm
                                    statistics, 2 sampler update (final conv); gn_apply: silu */
    int kernel;          /* conv: 1 = conv_tc.cu (general), 2 = conv_kf.cu (strip); 0 otherwise */
    int bn, cpg, ch, staged, xk16, tr, res1, apply;  /* the instantiation / walk that runs (ch: 64-channel input chunks) */
    cdc_tensor_desc src[2], residual, out, res_out;
    void* gn_in_acc;     /* GroupNorm accumulator slot read ([B][32][4] int64, csrc/gn_sums.cuh) or NULL */
    void* gn_out_acc;    /* slot accumulated into (memset: first slot cleared) or NULL */
    int gn_slots;        /* memset: slots cleared */
    float* x;            /* final conv: sampler state, NHWC fp32 [B][H][W][3], read as x_t and overwritten with x_prev */
    float* x0_out;       /* final conv: x0 estimate, NHWC fp32 */
    void* xpad;          /* final conv: the stem's 16-bit x_t copy, rewritten with x_prev */
} cdc_step_op_desc;
int cdc_step_op_describe(cdc_ctx* ctx, int i, cdc_step_op_desc* out);
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

#ifdef CDC_TOOLS
/* tools build only: leave a class of ops out of the captured graph (0 none, 1 tcgen05 convs, 2 elementwise/GroupNorm,
 * 3 attention); while a class is skipped cdc_get_x / cdc_decode_host fail with CDC_ERR_STATE (the image is garbage) */
int cdc_debug_graph_skip(cdc_ctx* ctx, int op_class);
#endif

#ifdef __cplusplus
}
#endif
#endif /* CDC_B200_TOOLS_H */
