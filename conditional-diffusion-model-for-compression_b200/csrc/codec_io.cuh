// What the host runtime (runner.cu) lends the byte-level codec entry points (bitstream.cu: cdc_compress_rgb8,
// cdc_decompress_rgb8): the bound plan's codec tensors and op sequences, and a slot for the state bitstream.cu owns.
#pragma once
#include <cuda_runtime.h>

#include "../../include/cdc_b200.h"
#include "kernels.cuh"

namespace cdc {

// Every entry point that takes a cdc_ctx runs on the context's device and restores the caller's current device on
// exit (ADVICE r1: a Decoder on cuda:1 must work -- and must not move the process -- while cuda:0 is current).
struct DevGuard {
    int prev = -1, dev;
    explicit DevGuard(int d) : dev(d) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DevGuard() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};

constexpr float kMinSigma = 0.11f;  // the hyper-decoder's sigma = max(sigma_raw, kMinSigma) (oracle/codec.py HyperDecoder)

// bitstream.cu's state in a context: the entropy tables (kept across binds) and the work buffers of the bound shape
struct ByteCodec;
void byte_codec_release_buffers(ByteCodec* bc);  // the bound shape's buffers (the plan is released); null is fine
void byte_codec_destroy(ByteCodec* bc);          // everything (cdc_destroy); null is fine

struct BoundCodec {
    int B = 0, H = 0, W = 0, latent_ch = 0, num_sms = 0, device = 0;
    int K = 0;              // steps of the set schedule (0: none)
    bool has_ctx = false;   // the context net's weights were loaded
    bool seeded = false;    // per-image seeds are bound (cdc_set_image_seeds)
    bool graph_skip = false;  // tools build: ops are left out of the decode graph, its image is garbage
    act_t* img64 = nullptr;           // [B*H*W][64]: the analysis encoder's input, channels 3..63 zero
    const act_t* enc_y = nullptr;     // [B*(H/16)*(W/16)][latent_ch]: its output
    act_t* hdec_in = nullptr;         // [B*(H/64)*(W/64)][latent_ch]: the hyper-decoder's input
    const act_t* hdec_out = nullptr;  // [B*(H/16)*(W/16)][2*latent_ch]: mu | raw sigma
    act_t* latent = nullptr;          // [B*(H/16)*(W/16)][latent_ch]: the context net's input
    const float* xs = nullptr;        // [B*H*W][3]: the sampler state
    ByteCodec** state = nullptr;      // the context's slot (created by bitstream.cu on first use)
};
// CDC_OK with *out filled, or CDC_ERR_STATE (no bound shape) / CDC_ERR_WEIGHT (no codec weights) with the message set
int bound_codec(cdc_ctx* ctx, BoundCodec* out);
// the context's slot only (no bound shape needed: cdc_set_entropy_tables)
ByteCodec** byte_codec_slot(cdc_ctx* ctx);
int ctx_device(cdc_ctx* ctx);
int ctx_latent_ch(cdc_ctx* ctx);

enum CodecSeq { CODEC_SEQ_ENCODER, CODEC_SEQ_HYPER_DEC, CODEC_SEQ_CONTEXT };
int run_codec_seq(cdc_ctx* ctx, CodecSeq q, cudaStream_t s);
// sets cdc_last_error and returns code
int ctx_fail(cdc_ctx* ctx, int code, const char* fmt, ...);

}  // namespace cdc
