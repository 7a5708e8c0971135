// The codec at the byte boundary (include/cdc_b200.h cdc_compress_rgb8 / cdc_decompress_rgb8): 8-bit RGB image <-> CDC5
// stream in one call each, the host orchestration of Codec.compress / Codec.decode_symbols (codec.py) on the library's own
// kernels.  Compress runs the kernels Codec.encode runs, in its order, so its bytes are Codec.compress's by construction;
// decompress derives every tensor the Python decoder derives with the same fp32 arithmetic and 16-bit rounding.
//
// Untrusted bytes: every field of the stream is checked on the host before a launch reads it (parse_stream), so the
// kernels never index with a count the context did not bind.  Each rANS container gets its own 16-byte-aligned device slot:
// the size table is read as u32 at container + 24, and in CDC5 the y container starts at 24 + nz with nz only even.
#include <stdarg.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "codec_io.cuh"

namespace cdc {

constexpr int64_t kCdc5Header = 24;  // "CDC5" | u32 B, H, W | u64 nz
constexpr int64_t kCdcrHeader = 24;  // "CDCR" | u32 version, n_chan, hw, spc, reserved

struct DevTables {
    void* mem = nullptr;  // cdf | row_start | cdf_length | offset | scale_table or median, one allocation
    CdfTables t{};
    const float* median = nullptr;  // factorised prior: [latent_ch]
    bool set() const { return mem != nullptr; }
    void release() {
        if (mem) cudaFree(mem);
        *this = DevTables();
    }
};

struct ByteCodec {
    DevTables tab[2];  // 0: Gaussian, 1: factorised prior (cdc_set_entropy_tables `which`)
    // work buffers of the bound shape (B, H, W); B == 0: none
    int B = 0, H = 0, W = 0;
    std::vector<void*> dev;  // every device allocation below
    uint8_t* rgb = nullptr;  // [B*H*W*3]
    float *y = nullptr, *z = nullptr, *z_hat = nullptr, *mu = nullptr, *sigma = nullptr;  // NCHW fp32
    int32_t *qz = nullptr, *q = nullptr, *zidx = nullptr, *yidx = nullptr;
    int32_t *zsym[5] = {}, *ysym[5] = {};  // (idx, v, lo, hi, raw) of cdf_lookup
    void* scratch = nullptr;               // rANS encode / decode workspace
    uint8_t *zslot = nullptr, *yslot = nullptr;
    int64_t zcap = 0, ycap = 0;            // slot sizes: the largest container of any spc
    unsigned long long* sizes = nullptr;   // [2] container sizes written by the encoder
    int32_t* status = nullptr;             // [2] decoder status words
    // page-locked staging for pageable caller buffers, and the readback of sizes / status
    uint8_t* h_rgb = nullptr;
    uint8_t* h_stream = nullptr;  // 24 + zcap + ycap
    unsigned long long* h_small = nullptr;  // sizes[2] | status[2]

    cudaError_t alloc(void** p, size_t bytes) {
        const cudaError_t e = cudaMalloc(p, (bytes + 255) & ~size_t(255));
        if (e == cudaSuccess) dev.push_back(*p);
        return e;
    }
    void release_buffers() {
        for (void* p : dev) cudaFree(p);
        dev.clear();
        if (h_rgb) cudaFreeHost(h_rgb);
        if (h_stream) cudaFreeHost(h_stream);
        if (h_small) cudaFreeHost(h_small);
        const DevTables t0 = tab[0], t1 = tab[1];
        *this = ByteCodec();
        tab[0] = t0;
        tab[1] = t1;
    }
};

void byte_codec_release_buffers(ByteCodec* bc) {
    if (bc) bc->release_buffers();
}
void byte_codec_destroy(ByteCodec* bc) {
    if (!bc) return;
    bc->release_buffers();
    bc->tab[0].release();
    bc->tab[1].release();
    delete bc;
}

// ------------------------------------------------------------------------------------------------ stream layout (host)
static uint32_t get_u32(const uint8_t* p) { return p[0] | (p[1] << 8) | (p[2] << 16) | (static_cast<uint32_t>(p[3]) << 24); }
static uint64_t get_u64(const uint8_t* p) { return get_u32(p) | (static_cast<uint64_t>(get_u32(p + 4)) << 32); }
static void put_u32(uint8_t* p, uint32_t v) {
    for (int i = 0; i < 4; ++i) p[i] = static_cast<uint8_t>(v >> (8 * i));
}

struct Container {
    const uint8_t* p = nullptr;
    uint64_t n_chan = 0, hw = 0, spc = 0;
    int64_t used = 0;  // 24 + 4 * streams + the streams' sizes: the bytes the decoder reads
};
struct StreamLayout {
    uint32_t B = 0, H = 0, W = 0;
    Container z, y;
};

// One CDCR container of `len` bytes holding rows of `hw` symbols.  What oracle/rans.py / rans_decode accept, checked without
// decoding: version 1, 1 <= spc <= 32, and a size table whose streams are whole 16-bit words holding at least the state
// and at most what their symbols can consume (4 bytes of state + 8 per symbol), lying inside the container.
static const char* parse_container(const uint8_t* p, uint64_t len, uint64_t hw, Container* c) {
    if (len < kCdcrHeader) return "container shorter than its header";
    if (memcmp(p, "CDCR", 4) != 0) return "bad container magic";
    if (get_u32(p + 4) != 1) return "unsupported container version";
    c->p = p;
    c->n_chan = get_u32(p + 8);
    c->hw = get_u32(p + 12);
    c->spc = get_u32(p + 16);
    if (c->n_chan < 1) return "container without rows";
    if (c->hw != hw) return "container row length does not match the image size";
    if (c->spc < 1 || c->spc > 32) return "container streams per row outside 1..32";
    const uint64_t ns = c->n_chan * c->spc;
    if (len < kCdcrHeader + 4 * ns) return "container shorter than its size table";
    const uint64_t max_stream = 4 + 8 * ((hw + c->spc - 1) / c->spc);
    uint64_t used = kCdcrHeader + 4 * ns;
    for (uint64_t i = 0; i < ns; ++i) {
        const uint32_t sz = get_u32(p + kCdcrHeader + 4 * i);
        if (sz < 4 || (sz & 1) || sz > max_stream) return "container size table holds an impossible stream size";
        used += sz;
    }
    if (used > len) return "container streams run past its end";
    c->used = static_cast<int64_t>(used);
    return nullptr;
}

// The whole CDC5 stream: header, both containers, and that they describe the same B x latent rows of an H x W image.
static const char* parse_stream(const uint8_t* d, int64_t n, StreamLayout* o) {
    if (!d || n < kCdc5Header) return "shorter than the CDC5 header";
    if (memcmp(d, "CDC5", 4) != 0) return "not a CDC5 stream";
    o->B = get_u32(d + 4);
    o->H = get_u32(d + 8);
    o->W = get_u32(d + 12);
    const uint64_t nz = get_u64(d + 16), rest = static_cast<uint64_t>(n - kCdc5Header);
    if (o->B < 1 || o->B > (1u << 20) || o->H < 64 || o->W < 64 || o->H % 64 || o->W % 64 || o->H > (1u << 16) || o->W > (1u << 16))
        return "header batch / image size out of range";
    if (nz > rest) return "z container runs past the end";
    if (nz == rest) return "no y container";
    const uint64_t hwy = static_cast<uint64_t>(o->H / 16) * (o->W / 16);
    const char* e = parse_container(d + kCdc5Header, nz, hwy / 16, &o->z);
    if (e) return e;
    if ((e = parse_container(d + kCdc5Header + nz, rest - nz, hwy, &o->y))) return e;
    if (o->z.n_chan != o->y.n_chan || o->z.n_chan % o->B) return "container rows do not match the batch";
    return nullptr;
}

// ------------------------------------------------------------------------------------------------ buffers
#define CK(expr)                                                                                               \
    do {                                                                                                       \
        cudaError_t e_ = (expr);                                                                               \
        if (e_ != cudaSuccess) return ctx_fail(ctx, CDC_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

enum HostMem { kPageable, kPinned, kDevice };
static HostMem host_mem(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();  // (unregistered host memory reports an error on old drivers)
        return kPageable;
    }
    return at.type == cudaMemoryTypeDevice ? kDevice : at.type == cudaMemoryTypeHost ? kPinned : kPageable;
}

static int64_t max_container_bytes(int64_t n_chan, int64_t hw) {  // over every spc a stream may declare
    int64_t m = 0;
    for (int spc = 1; spc <= 32; ++spc) m = std::max<int64_t>(m, rans_max_bytes(n_chan, hw, spc));
    return m;
}

struct Dims {
    int64_t npix, nch, hwy, hwz, ny, nz;
    int spc_y, spc_z;  // what the encoder writes (cdc_rans_streams_per_channel)
    explicit Dims(const BoundCodec& v)
        : npix(static_cast<int64_t>(v.B) * v.H * v.W), nch(static_cast<int64_t>(v.B) * v.latent_ch),
          hwy(static_cast<int64_t>(v.H / 16) * (v.W / 16)), hwz(hwy / 16), ny(nch * hwy), nz(nch * hwz),
          spc_y(cdc_rans_streams_per_channel(hwy)), spc_z(cdc_rans_streams_per_channel(hwz)) {}
};

// The bound plan, the context's ByteCodec and its work buffers for the bound shape (allocated here on first use).
static int prepare(cdc_ctx* ctx, BoundCodec* v, ByteCodec** out, cudaStream_t s) {
    int r = bound_codec(ctx, v);
    if (r) return r;
    ByteCodec*& bc = *v->state;
    if (!bc) bc = new ByteCodec();
    *out = bc;
    if (!bc->tab[0].set() || !bc->tab[1].set())
        return ctx_fail(ctx, CDC_ERR_STATE, "set the Gaussian and the factorised-prior tables first (cdc_set_entropy_tables)");
    if (bc->B == v->B && bc->H == v->H && bc->W == v->W) return CDC_OK;
    bc->release_buffers();
    const Dims d(*v);
    bc->zcap = max_container_bytes(d.nch, d.hwz);
    bc->ycap = max_container_bytes(d.nch, d.hwy);
    const int64_t scratch = std::max<int64_t>({rans_scratch_bytes(d.nch, d.hwz, d.spc_z), rans_scratch_bytes(d.nch, d.hwy, d.spc_y),
                                               8 * d.nch * 32 + 8});  // (decode: 8 bytes per stream)
    CK(bc->alloc(reinterpret_cast<void**>(&bc->rgb), d.npix * 3));
    for (float** f : {&bc->y, &bc->mu, &bc->sigma}) CK(bc->alloc(reinterpret_cast<void**>(f), d.ny * 4));
    for (float** f : {&bc->z, &bc->z_hat}) CK(bc->alloc(reinterpret_cast<void**>(f), d.nz * 4));
    for (int32_t** i : {&bc->q, &bc->yidx}) CK(bc->alloc(reinterpret_cast<void**>(i), d.ny * 4));
    for (int32_t** i : {&bc->qz, &bc->zidx}) CK(bc->alloc(reinterpret_cast<void**>(i), d.nz * 4));
    for (int k = 0; k < 5; ++k) {
        CK(bc->alloc(reinterpret_cast<void**>(&bc->ysym[k]), d.ny * 4));
        CK(bc->alloc(reinterpret_cast<void**>(&bc->zsym[k]), d.nz * 4));
    }
    CK(bc->alloc(&bc->scratch, scratch));
    CK(bc->alloc(reinterpret_cast<void**>(&bc->zslot), bc->zcap));  // (cudaMalloc: 256-byte aligned)
    CK(bc->alloc(reinterpret_cast<void**>(&bc->yslot), bc->ycap));
    CK(bc->alloc(reinterpret_cast<void**>(&bc->sizes), 16));
    CK(bc->alloc(reinterpret_cast<void**>(&bc->status), 8));
    CK(cudaMallocHost(&bc->h_rgb, d.npix * 3));
    CK(cudaMallocHost(&bc->h_stream, kCdc5Header + bc->zcap + bc->ycap));
    CK(cudaMallocHost(&bc->h_small, 32));
    // the z symbols' CDF row is their channel (codec.py decode_symbols)
    std::vector<int32_t> ch(static_cast<size_t>(d.nz));
    for (int64_t i = 0; i < d.nz; ++i) ch[i] = static_cast<int32_t>((i / d.hwz) % v->latent_ch);
    // (pageable source: staged by the driver before the call returns, so ch may go out of scope)
    CK(cudaMemcpyAsync(bc->zidx, ch.data(), ch.size() * 4, cudaMemcpyHostToDevice, s));
    bc->B = v->B;
    bc->H = v->H;
    bc->W = v->W;
    return CDC_OK;
}

}  // namespace cdc

using namespace cdc;

extern "C" {

int cdc_set_entropy_tables(cdc_ctx* ctx, int which, const int32_t* cdf, int64_t n_cdf, const int32_t* row_start,
                           const int32_t* cdf_length, const int32_t* offset, int rows, const float* scale_table,
                           const float* median) {
    if (!ctx) return CDC_ERR_STATE;
    const int latent_ch = ctx_latent_ch(ctx);
    if (which != 0 && which != 1) return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_set_entropy_tables: which must be 0 or 1, got %d", which);
    if (!cdf || !row_start || !cdf_length || !offset || n_cdf < 2 || n_cdf > (1LL << 30))
        return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_set_entropy_tables: null table, or n_cdf outside 2 .. 2^30");
    const int min_rows = which == 0 ? 64 : latent_ch;  // the decoder's rows: a scale-table entry, or the channel
    if (rows < min_rows || rows > 256)
        return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_set_entropy_tables: %d rows, need %d .. 256", rows, min_rows);
    if (which == 0 ? (!scale_table || median) : scale_table != nullptr)
        return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_set_entropy_tables: the Gaussian tables take a scale table and no median, "
                                            "the factorised prior a median (or NULL) and no scale table");
    for (int r = 0; r < rows; ++r)
        if (row_start[r] < 0 || cdf_length[r] < 2 || static_cast<int64_t>(row_start[r]) + cdf_length[r] > n_cdf)
            return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_set_entropy_tables: row %d (start %d, length %d) outside the %lld CDF entries", r,
                            row_start[r], cdf_length[r], static_cast<long long>(n_cdf));
    DevGuard guard(ctx_device(ctx));
    ByteCodec*& bc = *byte_codec_slot(ctx);
    if (!bc) bc = new ByteCodec();
    DevTables& t = bc->tab[which];
    t.release();  // (cudaFree waits for the device: no earlier call still reads the old tables)
    const int nf = which == 0 ? 64 : latent_ch;
    const size_t ints = static_cast<size_t>(n_cdf) + 3 * static_cast<size_t>(rows);
    std::vector<int32_t> hi(ints);
    memcpy(hi.data(), cdf, n_cdf * 4);
    memcpy(hi.data() + n_cdf, row_start, rows * 4);
    memcpy(hi.data() + n_cdf + rows, cdf_length, rows * 4);
    memcpy(hi.data() + n_cdf + 2 * rows, offset, rows * 4);
    std::vector<float> hf(nf, 0.0f);
    if (which == 0) memcpy(hf.data(), scale_table, 64 * 4);
    else if (median) memcpy(hf.data(), median, nf * 4);
    const size_t fofs = (ints * 4 + 15) & ~size_t(15);
    CK(cudaMalloc(&t.mem, fofs + nf * 4));
    int32_t* di = static_cast<int32_t*>(t.mem);
    float* df = reinterpret_cast<float*>(static_cast<uint8_t*>(t.mem) + fofs);
    CK(cudaMemcpyAsync(di, hi.data(), ints * 4, cudaMemcpyHostToDevice, 0));
    CK(cudaMemcpyAsync(df, hf.data(), nf * 4, cudaMemcpyHostToDevice, 0));
    CK(cudaStreamSynchronize(0));
    t.t = CdfTables{di, di + n_cdf, di + n_cdf + rows, di + n_cdf + 2 * rows, which == 0 ? df : nullptr, rows};
    t.median = which == 1 ? df : nullptr;
    return CDC_OK;
}

int cdc_stream_info(const uint8_t* data_host, int64_t nbytes, int* B, int* H, int* W) {
    StreamLayout L;
    if (parse_stream(data_host, nbytes, &L)) return CDC_ERR_DATA;
    if (B) *B = static_cast<int>(L.B);
    if (H) *H = static_cast<int>(L.H);
    if (W) *W = static_cast<int>(L.W);
    return CDC_OK;
}

int64_t cdc_compress_max_bytes(cdc_ctx* ctx) {
    BoundCodec v;
    const int r = bound_codec(ctx, &v);
    if (r) return r;
    const Dims d(v);
    return kCdc5Header + rans_max_bytes(d.nch, d.hwz, d.spc_z) + rans_max_bytes(d.nch, d.hwy, d.spc_y);
}

int cdc_compress_rgb8(cdc_ctx* ctx, const uint8_t* rgb_host, uint8_t* out_host, int64_t capacity, int64_t* nbytes, cdc_stream s) {
    if (!ctx) return CDC_ERR_STATE;
    if (!rgb_host || !out_host || !nbytes) return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_compress_rgb8: null buffer");
    BoundCodec v;
    int r = bound_codec(ctx, &v);
    if (r) return r;
    DevGuard guard(v.device);
    const HostMem in_mem = host_mem(rgb_host), out_mem = host_mem(out_host);
    if (in_mem == kDevice || out_mem == kDevice) return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_compress_rgb8: takes host buffers, got a device pointer");
    const cudaStream_t st = reinterpret_cast<cudaStream_t>(s);
    ByteCodec* bc = nullptr;
    if ((r = prepare(ctx, &v, &bc, st))) return r;
    const Dims d(v);
    const DevTables &gauss = bc->tab[0], &fact = bc->tab[1];
    const int Cl = v.latent_ch;
    // image -> y (cdc_encode_analysis with the 8-bit input)
    const uint8_t* src = rgb_host;
    if (in_mem == kPageable) {
        memcpy(bc->h_rgb, rgb_host, d.npix * 3);
        src = bc->h_rgb;
    }
    CK(cudaMemcpyAsync(bc->rgb, src, d.npix * 3, cudaMemcpyHostToDevice, st));
    CK(launch_rgb8_in(bc->rgb, v.img64, d.npix, st));
    if ((r = run_codec_seq(ctx, CODEC_SEQ_ENCODER, st))) return r;
    CK(launch_nhwc_act_to_nchw_f32(v.enc_y, bc->y, v.B, Cl, static_cast<int>(d.hwy), st));
    // Codec.encode: z, its symbols against the factorised prior, (mu, sigma) from z_hat, y's symbols
    if ((r = cdc_hyper_encode(ctx, bc->y, bc->z, s))) return r;
    CK(launch_quantize(bc->z, fact.median, bc->qz, bc->z_hat, d.nz, d.hwz, Cl, v.num_sms, st));
    CK(launch_cdf_lookup(bc->qz, nullptr, fact.t, d.hwz, bc->zsym[0], bc->zsym[1], bc->zsym[2], bc->zsym[3], bc->zsym[4], d.nz,
                         v.num_sms, st));
    if ((r = cdc_hyper_decode(ctx, bc->z_hat, bc->mu, bc->sigma, s))) return r;
    CK(launch_quantize(bc->y, bc->mu, bc->q, nullptr, d.ny, 0, 0, v.num_sms, st));
    CK(launch_cdf_lookup(bc->q, bc->sigma, gauss.t, 1, bc->ysym[0], bc->ysym[1], bc->ysym[2], bc->ysym[3], bc->ysym[4], d.ny,
                         v.num_sms, st));
    // the two containers, each into its own slot
    CK(launch_rans_encode(bc->zsym[0], bc->zsym[1], bc->zsym[2], bc->zsym[3], bc->zsym[4], fact.t.cdf_length, d.nch, d.hwz, d.spc_z,
                          bc->scratch, bc->zslot, bc->sizes, st));
    CK(launch_rans_encode(bc->ysym[0], bc->ysym[1], bc->ysym[2], bc->ysym[3], bc->ysym[4], gauss.t.cdf_length, d.nch, d.hwy, d.spc_y,
                          bc->scratch, bc->yslot, bc->sizes + 1, st));
    CK(cudaMemcpyAsync(bc->h_small, bc->sizes, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const int64_t nz = static_cast<int64_t>(bc->h_small[0]), ny = static_cast<int64_t>(bc->h_small[1]);
    *nbytes = kCdc5Header + nz + ny;
    if (capacity < *nbytes)
        return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_compress_rgb8: the stream is %lld bytes, the buffer holds %lld",
                        static_cast<long long>(*nbytes), static_cast<long long>(capacity));
    uint8_t* dst = out_mem == kPinned ? out_host : bc->h_stream;
    memcpy(dst, "CDC5", 4);
    put_u32(dst + 4, static_cast<uint32_t>(v.B));
    put_u32(dst + 8, static_cast<uint32_t>(v.H));
    put_u32(dst + 12, static_cast<uint32_t>(v.W));
    put_u32(dst + 16, static_cast<uint32_t>(static_cast<uint64_t>(nz)));
    put_u32(dst + 20, static_cast<uint32_t>(static_cast<uint64_t>(nz) >> 32));
    CK(cudaMemcpyAsync(dst + kCdc5Header, bc->zslot, nz, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(dst + kCdc5Header + nz, bc->yslot, ny, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (dst != out_host) memcpy(out_host, dst, *nbytes);
    return CDC_OK;
}

int cdc_decompress_rgb8(cdc_ctx* ctx, const uint8_t* data_host, int64_t nbytes, float gamma, uint8_t* rgb_host, cdc_stream s) {
    if (!ctx) return CDC_ERR_STATE;
    if (!data_host || !rgb_host) return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_decompress_rgb8: null buffer");
    BoundCodec v;
    int r = bound_codec(ctx, &v);
    if (r) return r;
    DevGuard guard(v.device);
    const HostMem in_mem = host_mem(data_host), out_mem = host_mem(rgb_host);
    if (in_mem == kDevice || out_mem == kDevice) return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_decompress_rgb8: takes host buffers, got a device pointer");
    if (!v.has_ctx) return ctx_fail(ctx, CDC_ERR_WEIGHT, "cdc_decompress_rgb8: context-net weights (context.*) were not loaded");
    if (v.K < 1) return ctx_fail(ctx, CDC_ERR_STATE, "cdc_decompress_rgb8: call cdc_set_schedule first");
    if (!v.seeded) return ctx_fail(ctx, CDC_ERR_STATE, "cdc_decompress_rgb8: no per-image seeds bound (cdc_set_image_seeds)");
    if (v.graph_skip) return ctx_fail(ctx, CDC_ERR_STATE, "ops are being left out of the graph (tools build, graph skip): x is garbage");
    // every field, before anything is launched on it
    StreamLayout L;
    if (const char* e = parse_stream(data_host, nbytes, &L)) return ctx_fail(ctx, CDC_ERR_DATA, "cdc_decompress_rgb8: %s", e);
    if (static_cast<int>(L.B) != v.B || static_cast<int>(L.H) != v.H || static_cast<int>(L.W) != v.W)
        return ctx_fail(ctx, CDC_ERR_SHAPE, "cdc_decompress_rgb8: the stream is %u x %u x %u, the bound shape %d x %d x %d", L.B, L.H, L.W,
                        v.B, v.H, v.W);
    if (L.z.n_chan != static_cast<uint64_t>(v.B) * v.latent_ch)
        return ctx_fail(ctx, CDC_ERR_DATA, "cdc_decompress_rgb8: %llu container rows, the context codes %d per image",
                        static_cast<unsigned long long>(L.z.n_chan), v.latent_ch);
    const cudaStream_t st = reinterpret_cast<cudaStream_t>(s);
    ByteCodec* bc = nullptr;
    if ((r = prepare(ctx, &v, &bc, st))) return r;
    const Dims d(v);
    const DevTables &gauss = bc->tab[0], &fact = bc->tab[1];
    const int Cl = v.latent_ch;
    if (L.z.used > bc->zcap || L.y.used > bc->ycap) return ctx_fail(ctx, CDC_ERR_DATA, "cdc_decompress_rgb8: container larger than any valid one");
    // each container into its own aligned slot
    const uint8_t *zsrc = L.z.p, *ysrc = L.y.p;
    if (in_mem == kPageable) {
        memcpy(bc->h_stream, L.z.p, L.z.used);
        memcpy(bc->h_stream + bc->zcap, L.y.p, L.y.used);
        zsrc = bc->h_stream;
        ysrc = bc->h_stream + bc->zcap;
    }
    CK(cudaMemcpyAsync(bc->zslot, zsrc, L.z.used, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(bc->yslot, ysrc, L.y.used, cudaMemcpyHostToDevice, st));
    // z (row = channel) -> z_hat = qz + median -> hyper-decoder -> y's rows from sigma -> y
    CK(launch_rans_decode(bc->zslot, L.z.used, bc->zidx, fact.t, d.nch, d.hwz, static_cast<int>(L.z.spc), bc->scratch, bc->qz,
                          bc->status, st));
    CK(launch_dequant_to_act(bc->qz, fact.median, nullptr, 0, v.hdec_in, v.B, Cl, static_cast<int>(d.hwz), st));
    if ((r = run_codec_seq(ctx, CODEC_SEQ_HYPER_DEC, st))) return r;
    CK(launch_scale_rows(v.hdec_out, 2 * Cl, Cl, kMinSigma, gauss.t.scale_table, bc->yidx, v.B, Cl, static_cast<int>(d.hwy), st));
    CK(launch_rans_decode(bc->yslot, L.y.used, bc->yidx, gauss.t, d.nch, d.hwy, static_cast<int>(L.y.spc), bc->scratch, bc->q,
                          bc->status + 1, st));
    int32_t* h_status = reinterpret_cast<int32_t*>(bc->h_small + 2);
    CK(cudaMemcpyAsync(h_status, bc->status, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (h_status[0] || h_status[1])
        return ctx_fail(ctx, CDC_ERR_DATA, "cdc_decompress_rgb8: the %s container is truncated or corrupt", h_status[0] ? "z" : "y");
    // y_hat = q + mu -> context net -> x_T from the seeds -> K steps -> 8-bit image
    CK(launch_dequant_to_act(bc->q, nullptr, v.hdec_out, 2 * Cl, v.latent, v.B, Cl, static_cast<int>(d.hwy), st));
    if ((r = run_codec_seq(ctx, CODEC_SEQ_CONTEXT, st))) return r;
    if ((r = cdc_init_noise(ctx, gamma, s))) return r;
    if ((r = cdc_decode(ctx, s))) return r;
    CK(launch_rgb8_out(v.xs, bc->rgb, d.npix, st));
    uint8_t* dst = out_mem == kPinned ? rgb_host : bc->h_rgb;
    CK(cudaMemcpyAsync(dst, bc->rgb, d.npix * 3, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (dst != rgb_host) memcpy(rgb_host, dst, d.npix * 3);
    return CDC_OK;
}

}  // extern "C"
