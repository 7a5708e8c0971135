"""Reference of the per-image seeded noise (include/cdc_b200.h cdc_set_image_seeds; csrc/sampler.cuh), in numpy on top of
oracle/sampler.py's Philox, and an OracleDecoder that decodes with it.  Test infrastructure only.

Image b's noise is Philox4x32-10 keyed by seeds[b] (64-bit), counter (p_lo, p_hi, c2, c3) with p = h*W + w the pixel
index WITHIN the image; the words become three normals exactly as oracle/sampler.py philox_normal converts them.
Planes: x_T is (c2, c3) = (0, 1) and x_T = gamma * z; the sampler noise of step k is (k, 0)."""
import numpy as np
import torch

from oracle.sampler import OracleDecoder, ddim_update, philox4x32_10

XT_PLANE = (0, 1)


def step_plane(k):
    return (int(k), 0)


def philox_normal_images(seeds, c2, c3, H, W) -> torch.Tensor:
    """z [len(seeds), 3, H, W] fp32: image b keyed by seeds[b], counter (pixel within the image, c2, c3)."""
    p = np.arange(H * W, dtype=np.uint64)
    lo, hi = p & np.uint64(0xFFFFFFFF), p >> np.uint64(32)
    out = []
    for s in seeds:
        s = int(s)
        w0, w1, w2, w3 = philox4x32_10(lo, hi, np.full(p.shape, c2, dtype=np.uint64), np.full(p.shape, c3, dtype=np.uint64),
                                       s & 0xFFFFFFFF, (s >> 32) & 0xFFFFFFFF)
        u0 = ((w0 >> np.uint32(9)).astype(np.float64) + 0.5) / 8388608.0
        u2 = ((w2 >> np.uint32(9)).astype(np.float64) + 0.5) / 8388608.0
        t1 = (w1 >> np.uint32(8)).astype(np.float64) / 16777216.0
        t3 = (w3 >> np.uint32(8)).astype(np.float64) / 16777216.0
        r0, r2 = np.sqrt(-2.0 * np.log(u0)), np.sqrt(-2.0 * np.log(u2))
        z = np.stack([r0 * np.cos(2.0 * np.pi * t1), r0 * np.sin(2.0 * np.pi * t1), r2 * np.cos(2.0 * np.pi * t3)], axis=0)
        out.append(z.reshape(3, H, W))
    return torch.from_numpy(np.ascontiguousarray(np.stack(out, axis=0)).astype(np.float32))


class SeededOracleDecoder(OracleDecoder):
    """OracleDecoder with per-image seeds: decode(..., seeds=[...]) draws x_T per image and, while it runs, denoise_step
    adds per-image sampler noise.  Without seeds it is the OracleDecoder."""

    image_seeds = None

    @torch.no_grad()
    def denoise_step(self, x_t, t, cond):
        if self.image_seeds is None:
            return super().denoise_step(x_t, t, cond)
        k = self._k_of(t)
        out = self.network_out(x_t, t, cond)
        sc = self.sched
        z = None
        if float(sc.sg[k]) != 0.0:
            z = philox_normal_images(self.image_seeds, *step_plane(k), x_t.shape[2], x_t.shape[3])
        return ddim_update(x_t, out, sc.c0[k], sc.c1[k], sc.e0[k], sc.e1[k], sc.sg[k], z)

    @torch.no_grad()
    def decode(self, latent, steps, *, init=None, gamma=0.8, seed=0, seeds=None, cond=None, trajectory=None):
        if seeds is None:
            return super().decode(latent, steps, init=init, gamma=gamma, seed=seed, cond=cond, trajectory=trajectory)
        if init is not None:
            raise ValueError("give init or seeds, not both")
        B, _, h, w = latent.shape
        if len(seeds) != B:
            raise ValueError(f"{len(seeds)} seeds for a batch of {B}")
        x_T = gamma * philox_normal_images(seeds, *XT_PLANE, h * 16, w * 16)
        self.image_seeds = [int(s) for s in seeds]
        try:
            return super().decode(latent, steps, init=x_T, cond=cond, trajectory=trajectory)
        finally:
            self.image_seeds = None
