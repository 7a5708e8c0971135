// Sampler update applied in the final conv's epilogue, and the counter-based noise it may add.
//
//   x0     = e0 * x_t + e1 * out          (X-parameterisation: e0 = 0, e1 = 1;  eps-parameterisation: out = eps_hat,
//                                           e0 = 1/sqrt(abar_t), e1 = -sqrt(1 - abar_t)/sqrt(abar_t))
//   x_prev = c0 * clamp(x0, -1, 1) + c1 * x_t + sg * z
//
// with (c0, c1, sg) from the schedule (eta = 0: sg = 0 and the update is the deterministic DDIM step of SURVEY.md A.4).
// z ~ N(0, 1) is a pure function of (seed, step, pixel, channel): Philox4x32-10 keyed by the seed, counter =
// (pixel index, step, 0, 0); words 0/1 -> Box-Muller pair (channels 0, 1), words 2/3 -> channel 2.  The oracle
// (oracle/sampler.py philox_normal) restates the same function in numpy, so a teacher-forced stochastic step can be
// compared within the float tolerance.
// Per-image mode (cdc_set_image_seeds): the key is image b's own seed and the counter's pixel is the index h*W + w
// WITHIN the image, so image b's noise does not depend on the batch it is decoded in.  Step k's plane uses counter words
// (k, 0), the x_T plane (init_noise_kernel) (0, 1): the two never share a counter.
// Oracle counterpart: oracle/sampler.py ddim_update / make_schedule (the reference ships no code).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cdc {

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t (&out)[4]) {
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
        const uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0;
        c1 = lo1;
        c2 = n2;
        c3 = lo0;
        k0 += W0;
        k1 += W1;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}

// Philox words -> three standard normals (shared by every noise plane)
__device__ __forceinline__ void philox_words_normal3(const uint32_t (&w)[4], float (&z)[3]) {
    const float u0 = (static_cast<float>(w[0] >> 9) + 0.5f) * (1.0f / 8388608.0f);   // (0, 1): 23 bits + 1/2, exact in fp32
    const float u2 = (static_cast<float>(w[2] >> 9) + 0.5f) * (1.0f / 8388608.0f);
    const float t1 = static_cast<float>(w[1] >> 8) * (1.0f / 16777216.0f);           // [0, 1)
    const float t3 = static_cast<float>(w[3] >> 8) * (1.0f / 16777216.0f);
    const float r0 = sqrtf(-2.0f * logf(u0)), r2 = sqrtf(-2.0f * logf(u2));
    float s1, c1;
    sincospif(2.0f * t1, &s1, &c1);
    const float c3 = cospif(2.0f * t3);
    z[0] = r0 * c1;
    z[1] = r0 * s1;
    z[2] = r2 * c3;
}

// three standard normals of counter (pix, c2, c3) under key `seed`
__device__ __forceinline__ void philox_normal3(unsigned long long seed, unsigned long long pix, uint32_t c2, uint32_t c3,
                                               float (&z)[3]) {
    uint32_t w[4];
    philox4x32_10(static_cast<uint32_t>(pix), static_cast<uint32_t>(pix >> 32), c2, c3, static_cast<uint32_t>(seed),
                  static_cast<uint32_t>(seed >> 32), w);
    philox_words_normal3(w, z);
}

struct SamplerCoef {
    float c0, c1, e0, e1, sg;
    unsigned long long seed;
    int step;
    const unsigned long long* img_seeds;  // kernels.cuh ImageSeeds block, or null; read only when sg != 0
    unsigned int hw;                      // pixels per image
};

// one pixel's three channels: returns x_prev in xn, the (unclamped) x0 estimate in x0
__device__ __forceinline__ void sampler_update3(const SamplerCoef& s, const float (&outv)[3], const float (&xt)[3],
                                                unsigned long long pix, float (&x0)[3], float (&xn)[3]) {
    float z[3] = {0.f, 0.f, 0.f};
    if (s.sg != 0.0f) {
        if (s.img_seeds && s.img_seeds[0]) {  // per-image mode: image b's seed, pixel within the image
            const unsigned long long b = pix / s.hw;
            philox_normal3(s.img_seeds[1 + b], pix - b * s.hw, static_cast<uint32_t>(s.step), 0u, z);
        } else {
            philox_normal3(s.seed, pix, static_cast<uint32_t>(s.step), 0u, z);
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        // (e0 = 0, e1 = 1 reproduces out exactly: 0 * x_t is +-0 for finite x_t and 1 * out + 0 = out)
        x0[c] = fmaf(s.e1, outv[c], s.e0 * xt[c]);
        const float v = s.c0 * fminf(fmaxf(x0[c], -1.0f), 1.0f) + s.c1 * xt[c];
        xn[c] = s.sg != 0.0f ? fmaf(s.sg, z[c], v) : v;
    }
}

}  // namespace cdc
