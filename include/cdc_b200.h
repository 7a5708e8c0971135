/* cdc_b200 -- C ABI of the B200-native CDC decode hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  The reference repository ships no code
 * (/root/reference/README.md is 0 bytes, /root/reference/.gitignore:1-27 is a stock template), so
 * there is no reference FFI to cite line by line; each entry point below names the ORACLE
 * function it replaces (the parity source pinned by BASELINE.json `north_star`), which is what a
 * maintainer of the reference would bind through ctypes (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; all tensor pointers are DEVICE pointers unless the
 * name says `_host`; tensors cross the boundary as contiguous NCHW fp32 (the layout of the
 * oracle's torch tensors) and are converted to the internal NHWC 16-bit layout (fp16 by default, see csrc/act.cuh) on the device.
 * Every call returns 0 on success or a negative cdc_status; the message is available from
 * cdc_last_error().  Nothing throws across the ABI.  There is NO CPU fallback: a device that is
 * not sm_100 is CDC_ERR_ARCH.  One cdc_ctx per (process, device); not thread-safe; all work is
 * enqueued on the caller's stream (pass 0 for the legacy default stream).
 */
#ifndef CDC_B200_H
#define CDC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cdc_ctx cdc_ctx;
typedef void* cdc_stream; /* cudaStream_t */

typedef enum {
    CDC_OK = 0,
    CDC_ERR_SHAPE = -1,
    CDC_ERR_ARCH = -2,
    CDC_ERR_CUDA = -3,
    CDC_ERR_UNIMPLEMENTED = -4,
    CDC_ERR_STATE = -5,
    CDC_ERR_WEIGHT = -6,
    CDC_ERR_DATA = -7 /* the bytes are not a valid CDC5 stream for this context */
} cdc_status;

/* oracle/config.py CDCConfig */
typedef struct {
    int32_t base;      /* 64 */
    int32_t mults[4];  /* 1,2,3,4 */
    int32_t groups;    /* 32 */
    int32_t heads;     /* 4 */
    int32_t head_dim;  /* 64 */
    int32_t temb;      /* 256 */
    int32_t T;         /* 1000 */
    int32_t latent_ch; /* 256 */
    float gn_eps;      /* 1e-5 */
} cdc_config;

/* ---- lifetime -------------------------------------------------------------------------------- */
int cdc_create(const cdc_config* cfg, int device, cdc_ctx** out);
void cdc_destroy(cdc_ctx* ctx);
const char* cdc_last_error(cdc_ctx* ctx); /* ctx may be NULL: last error of a failed cdc_create */
int cdc_abi_version(void); /* 2 */
int cdc_act_dtype(void); /* storage / MMA operand type of activations: 1 = fp16 (default build), 0 = bf16 */

/* ---- weights: oracle/unet.py UNet.state_dict() (+ "context." + oracle/codec.py ContextNet) ----
 * `name` is the state-dict key, `dev_ptr` a device fp32 tensor in PyTorch layout (conv OIHW,
 * linear [out][in]).  The data is copied; the caller may free it after the call returns and the
 * stream is synchronised.  cdc_finalize_weights() repacks conv weights to 16-bit [C_out][kh][kw][C_in]
 * and fails with CDC_ERR_WEIGHT naming the first missing tensor. */
int cdc_load_weights(cdc_ctx* ctx, const char* name, const void* dev_ptr, const int64_t* shape, int ndim);
int cdc_finalize_weights(cdc_ctx* ctx);
int cdc_has_context_net(cdc_ctx* ctx);

/* ---- oracle/sampler.py make_schedule / OracleDecoder.set_sample_schedule ---------------------- */
int cdc_set_schedule(cdc_ctx* ctx, int steps);
int cdc_schedule_index(cdc_ctx* ctx, int k);              /* training index idx_k, or <0 */
int cdc_schedule_coeffs(cdc_ctx* ctx, int k, float* c0, float* c1);
/* sampler variant (SURVEY.md section 8 row f4; oracle/sampler.py make_schedule(..., eta, pred)): pred_eps = 0 the network
 * predicts x0 (default), 1 it predicts the noise; eta >= 0 is the DDIM stochasticity (0 = deterministic), seed keys the
 * counter-based noise z(seed, step, pixel).  Takes effect at the next cdc_set_schedule. */
int cdc_set_sampler(cdc_ctx* ctx, int pred_eps, float eta, uint64_t seed);
/* all five coefficients of step k: x0 = e0*x_t + e1*out; x_prev = c0*clamp(x0) + c1*x_t + sigma*z */
int cdc_schedule_coeffs5(cdc_ctx* ctx, int k, float* c0, float* c1, float* e0, float* e1, float* sigma);
/* oracle/unet.py TimeEmbed + RB.film for every step of the schedule: floats per step, and the table
 * [steps][cdc_film_size] (18 ResBlocks x (scale | shift)) copied to a device buffer */
int cdc_film_size(cdc_ctx* ctx);
int cdc_get_film(cdc_ctx* ctx, float* film_dev, cdc_stream s);

/* ---- shape binding: allocates the workspace arena, builds tensor maps and the launch plan ------
 * batch 1 .. 192 (CDC_ERR_SHAPE beyond: the GroupNorm apply kernel holds every image's statistics table in 48 KB of
 * shared memory); height and width multiples of 64. */
int cdc_bind_io(cdc_ctx* ctx, int batch, int height, int width);
/* Batch-invariant plans: on = 1 lays every op sequence (denoise step, context net, analysis encoder, hyper-encoder,
 * hyper-decoder) out per image exactly as for a batch of 1; the launches still cover the whole batch.  on = 0 (the
 * default) plans for the bound batch; any other value is CDC_ERR_SHAPE.  Takes effect at the next cdc_bind_io, which
 * re-plans when the mode changed, also for the bound shape.
 * The guarantee, for any batch 1 .. 192 and any position b: everything computed for image b -- the context maps, x_t and
 * raw x0_hat of every step, the final image, y, z, mu, sigma and the quantised symbols of the codec side, the pixels of
 * cdc_decompress_rgb8 -- is bit for bit what the same call gives for that image bound alone, and what the default mode
 * gives at batch 1.  Conditions: the noise is per image (seeds bound with cdc_set_image_seeds, or a caller-supplied x_T with
 * eta = 0), and both runs use the same SM count (a device of the same model) and the same build (fp16 or bf16).  The cost
 * is throughput at large batches: shorter strips mean more halo rows per image (DESIGN.md). */
int cdc_set_batch_invariant(cdc_ctx* ctx, int on);
int cdc_set_cond(cdc_ctx* ctx, const float* c0, const float* c1, const float* c2, const float* c3, cdc_stream s);
int cdc_set_latent(cdc_ctx* ctx, const float* y_hat, cdc_stream s); /* runs the context net: cond = context_net(y_hat) */
int cdc_set_x(cdc_ctx* ctx, const float* x_nchw, cdc_stream s);
int cdc_get_x(cdc_ctx* ctx, float* x_nchw, int to_image01, cdc_stream s);
int cdc_get_x0(cdc_ctx* ctx, float* x0_nchw, cdc_stream s); /* raw x0_hat of the last step (predict_x0) */
/* the bound context maps (oracle/codec.py ContextNet.forward output, or what cdc_set_cond stored): NCHW fp32
 * c_i [B, C_i, H >> i, W >> i]; any pointer may be NULL to skip that level */
int cdc_get_cond(cdc_ctx* ctx, float* c0, float* c1, float* c2, float* c3, cdc_stream s);

/* ---- codec side of the decode loop (SURVEY.md section 8 row f2; oracle/codec.py Encoder, HyperEncoder, HyperDecoder) --
 * Available when the weights named "codec." + oracle Codec.state_dict() keys (codec.encoder.*, codec.hyper_enc.*,
 * codec.hyper_dec.*) were loaded; shapes follow cdc_bind_io(batch, H, W).  Deterministic: the same input gives the same
 * bits on every run and every B200 (fixed accumulation order), so an encoder and a decoder that both run
 * cdc_hyper_decode on the same z_hat derive identical (mu, sigma) -- what a real bitstream needs. */
int cdc_has_codec(cdc_ctx* ctx);
/* y = encoder(2 * img - 1): img NCHW fp32 [B,3,H,W] in [0,1] -> y NCHW fp32 [B,latent_ch,H/16,W/16] */
int cdc_encode_analysis(cdc_ctx* ctx, const float* img01, float* y, cdc_stream s);
/* z = hyper_enc(y): [B,latent_ch,H/16,W/16] -> [B,latent_ch,H/64,W/64] */
int cdc_hyper_encode(cdc_ctx* ctx, const float* y, float* z, cdc_stream s);
/* (mu, sigma) = hyper_dec(z_hat), sigma = max(sigma_raw, 0.11): [B,latent_ch,H/64,W/64] -> 2 x [B,latent_ch,H/16,W/16] */
int cdc_hyper_decode(cdc_ctx* ctx, const float* z_hat, float* mu, float* sigma, cdc_stream s);

/* ---- oracle/sampler.py OracleDecoder.denoise_step / decode ------------------------------------ */
int cdc_denoise_step(cdc_ctx* ctx, int k, cdc_stream s); /* x <- c0_k*clamp(unet(x, idx_k, cond)) + c1_k*x */
int cdc_decode(cdc_ctx* ctx, cdc_stream s);              /* all K steps: ONE cudaGraphLaunch */
/* All K steps like cdc_decode, also recording the trajectory (oracle/sampler.py OracleDecoder.decode(trajectory=...)).
 * Slot j records step k = j * every, for j < ceil(K / every).
 * x_traj[j]  = x_t entering step k (x_traj[0] = x_T).
 * x0_traj[j] = raw x0_hat of step k, as cdc_get_x0 gives it.
 * Both are NCHW fp32 [slots][B][3][H][W] device buffers. Either may be NULL, but not both.
 * The final state (cdc_get_x / cdc_get_x0) is bit-identical to cdc_decode's.  A second graph, captured on the first call
 * for the current (K, every) and dropped with cdc_decode's; the buffer pointers are not baked into it. */
int cdc_decode_trajectory(cdc_ctx* ctx, float* x_traj, float* x0_traj, int every, cdc_stream s);
/* Blocks the host until slot j of the most recent cdc_decode_trajectory has been written. */
int cdc_trajectory_wait(cdc_ctx* ctx, int j);
/* host-buffer convenience used for end-to-end timing: H2D(latent, x_T) -> context net -> decode ->
 * D2H(image in [0,1]); synchronises the stream before returning. */
int cdc_decode_host(cdc_ctx* ctx, const float* latent_host, const float* xT_host, float* image_host, cdc_stream s);

/* ---- per-image seeds: image b's noise depends only on (seeds[b], pixel within the image, plane), not on its batch ----
 * Philox4x32-10 keyed by seeds[b], counter (p, c2, c3) with p = h*W + w inside the image: x_T uses (c2, c3) = (0, 1),
 * the sampler noise of step k (eta > 0) (k, 0).  Without seeds bound, the noise is the batch-wide one of cdc_set_sampler.
 * cdc_set_image_seeds: n == batch turns per-image mode on with these seeds, n == 0 turns it off; any other n is
 * CDC_ERR_SHAPE.  Written in stream order on `s` (after the last launch that read the previous seeds); the captured graphs
 * are not re-captured.  A cdc_bind_io to a different shape turns the mode off. */
int cdc_set_image_seeds(cdc_ctx* ctx, const uint64_t* seeds_host, int n, cdc_stream s);
/* x_T = gamma * z(seeds[b], pixel) into the sampler state (as cdc_set_x would put it); CDC_ERR_STATE without seeds bound */
int cdc_init_noise(cdc_ctx* ctx, float gamma, cdc_stream s);
/* cdc_decode_host with x_T drawn on the device from the bound seeds (cdc_init_noise) instead of copied from the host */
int cdc_decode_host_seeded(cdc_ctx* ctx, const float* latent_host, float gamma, float* image_host, cdc_stream s);

int cdc_launches_per_step(cdc_ctx* ctx);
int cdc_launches_context(cdc_ctx* ctx);
double cdc_flops_per_step(cdc_ctx* ctx); /* algorithmic, SURVEY.md section 8d rule */
/* fp16 storage diagnostics: number of epilogue passes (thread x tile) that met a value beyond +-65504 and stored it
 * saturated since the context was created or the counter last reset.  0 with the synthetic weights; a trained
 * checkpoint that makes this non-zero is losing accuracy silently otherwise.  Synchronises the stream. */
int cdc_saturation_count(cdc_ctx* ctx, uint64_t* count, int reset, cdc_stream s);

/* ---- oracle/entropy.py quantize_symbols / cdf_lookup (stateless) ------------------------------- */
/* q = rint(y - mu) int32 (half-to-even), y_hat = q + mu.  mu_mod == 0: mu is elementwise;
 * otherwise mu[(i / mu_inner) % mu_mod] (per-channel medians of the factorised prior). */
int cdc_quantize(const float* y, const float* mu, int32_t* q, float* y_hat, int64_t n, int64_t mu_inner,
                 int64_t mu_mod, cdc_stream s);
/* sigma != NULL: idx from the 64-entry scale table; sigma == NULL: idx = (i / inner) % rows. */
int cdc_cdf_lookup(const int32_t* q, const float* sigma, const int32_t* cdf, const int32_t* row_start,
                   const int32_t* cdf_length, const int32_t* offset, const float* scale_table, int rows,
                   int64_t inner, int32_t* idx, int32_t* v, int32_t* lo, int32_t* hi, int32_t* raw, int64_t n,
                   cdc_stream s);

/* ---- oracle/rans.py encode / decode: the on-wire bitstream of the quantised latents (SURVEY.md section 8 row f3) ------
 * 32-bit-state rANS, 16-bit precision, 16-bit words; every channel row of `hw` symbols (n_chan = batch * channels rows) is
 * cut into `spc` interleaved streams (stream j codes symbols j, j + spc, ...).  Byte-exact with the oracle; the container
 * layout is in oracle/rans.py and DESIGN.md.  All pointers are device pointers; stateless, current device. */
int cdc_rans_streams_per_channel(int64_t hw);                       /* the format's choice of spc for hw symbols per row */
int64_t cdc_rans_scratch_bytes(int64_t n_chan, int64_t hw, int spc); /* workspace for cdc_rans_encode */
int64_t cdc_rans_max_bytes(int64_t n_chan, int64_t hw, int spc);     /* upper bound of the container size */
/* (idx, v, lo, hi, raw) as produced by cdc_cdf_lookup + the tables' cdf_length -> container in `out`; its size in bytes
 * is written to *out_bytes_dev (device memory) when the stream reaches that point */
int cdc_rans_encode(const int32_t* idx, const int32_t* v, const int32_t* lo, const int32_t* hi, const int32_t* raw,
                    const int32_t* cdf_length, int64_t n_chan, int64_t hw, int spc, void* scratch, uint8_t* out,
                    int64_t out_capacity, uint64_t* out_bytes_dev, cdc_stream s);
/* container + the CDF row index of every element (from sigma, or the channel) -> q int32; n_chan / hw / spc are the
 * header's values (the caller parses the 24-byte header); scratch: 8 bytes per stream; *status_dev = 1 if the container is
 * truncated or corrupt */
int cdc_rans_decode(const uint8_t* data, int64_t data_bytes, const int32_t* idx, const int32_t* cdf, const int32_t* row_start,
                    const int32_t* cdf_length, const int32_t* offset, int rows, int64_t n_chan, int64_t hw, int spc,
                    void* scratch, int32_t* q, int32_t* status_dev, cdc_stream s);

/* ---- the codec at the byte boundary: 8-bit RGB image <-> CDC5 stream, one call each (Codec.compress / decompress_bytes) --
 * CDC5 = "CDC5" | u32 B, H, W | u64 nz | z container (nz bytes, cdc_rans_*) | y container; seeds and steps are not in it.
 * Images are host [B][H][W][3] uint8, interleaved RGB.  Host buffers work as in cdc_decode_host: page-locked ones are
 * copied directly, pageable ones through pinned staging; a device pointer is CDC_ERR_SHAPE.  The work buffers are
 * allocated on the first compress / decompress for the bound shape and freed with it.  Every byte of a stream is checked
 * on the host before anything runs on it: a stream that does not parse for this context is CDC_ERR_DATA, as is one whose
 * rANS payload does not decode (found on the device; the decode then stops before the diffusion steps). */
/* Entropy tables, host arrays in the layout of entropy_tables.Tables (cdf[n_cdf]; row_start, cdf_length, offset [rows]);
 * copied to the device and validated (row_start + cdf_length inside n_cdf, cdf_length >= 2).
 * which = 0: Gaussian, 64 <= rows <= 256 (row = scale-table entry), scale_table[64], median NULL.
 * which = 1: factorised prior, latent_ch <= rows <= 256 (row = channel), scale_table NULL, median[latent_ch] (NULL: zeros). */
int cdc_set_entropy_tables(cdc_ctx* ctx, int which, const int32_t* cdf, int64_t n_cdf, const int32_t* row_start,
                           const int32_t* cdf_length, const int32_t* offset, int rows, const float* scale_table,
                           const float* median);
/* Host-only parse of a CDC5 stream (no CUDA call): B, H, W, so the caller can cdc_bind_io.  CDC_ERR_DATA if the header,
 * either container header or a size table is malformed or points past the end. */
int cdc_stream_info(const uint8_t* data_host, int64_t nbytes, int* B, int* H, int* W);
/* Largest stream cdc_compress_rgb8 can write for the bound shape: 24 + both containers' cdc_rans_max_bytes (< 0: error) */
int64_t cdc_compress_max_bytes(cdc_ctx* ctx);
/* rgb_host [B][H][W][3] uint8 of the bound shape -> the CDC5 stream in out_host, byte-identical to Codec.compress(rgb / 255),
 * and its size in *nbytes.  Needs both tables.  CDC_ERR_SHAPE if capacity < *nbytes (which still reports the size needed).
 * Synchronises s. */
int cdc_compress_rgb8(cdc_ctx* ctx, const uint8_t* rgb_host, uint8_t* out_host, int64_t capacity, int64_t* nbytes, cdc_stream s);
/* CDC5 stream -> rgb_host [B][H][W][3] uint8 = round_half_even(255 * (clamp(x,-1,1)+1)/2) of the decode of its latent with
 * the set schedule and the bound per-image seeds (x_T = gamma * z; CDC_ERR_STATE without seeds, as cdc_decode_host_seeded),
 * i.e. Decoder.decode(Codec.decompress_bytes(...), seeds=...) in 8 bits.  The stream's B, H, W must be the bound shape
 * (CDC_ERR_SHAPE).  Needs both tables and the context net.  Synchronises s. */
int cdc_decompress_rgb8(cdc_ctx* ctx, const uint8_t* data_host, int64_t nbytes, float gamma, uint8_t* rgb_host, cdc_stream s);

#ifdef __cplusplus
}
#endif
#endif /* CDC_B200_H */
