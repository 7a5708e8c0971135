"""CPU checks of the per-image seeded noise reference (tests/seeded_reference.py): an image's noise does not depend on the
batch around it, planes and seeds are distinct, the definition is tied to the batch-wide philox_normal, and an oracle
decode with per-image seeds gives each image the result it gets alone."""
import pytest
import torch

from oracle.sampler import philox_normal
from tests.seeded_reference import XT_PLANE, SeededOracleDecoder, philox_normal_images, step_plane

SEEDS = [7, 2 ** 64 - 1, 0x0123456789ABCDEF]


def test_image_noise_is_independent_of_the_batch():
    H, W = 32, 48
    for plane in (XT_PLANE, step_plane(0), step_plane(5)):
        z = philox_normal_images(SEEDS, *plane, H, W)
        assert z.shape == (3, 3, H, W) and z.dtype == torch.float32
        for b, s in enumerate(SEEDS):
            assert torch.equal(z[b], philox_normal_images([s], *plane, H, W)[0]), (plane, b)


def test_seeds_and_planes_differ():
    H, W = 32, 32
    z = philox_normal_images(SEEDS, *XT_PLANE, H, W)
    for i in range(3):
        for j in range(i + 1, 3):
            assert (z[i] - z[j]).abs().mean() > 0.5
    for s in SEEDS:
        xt = philox_normal_images([s], *XT_PLANE, H, W)
        s0 = philox_normal_images([s], *step_plane(0), H, W)
        s1 = philox_normal_images([s], *step_plane(1), H, W)
        assert (xt - s0).abs().mean() > 0.5 and (s0 - s1).abs().mean() > 0.5
    # roughly standard normal
    big = philox_normal_images([3], *XT_PLANE, 128, 128)
    assert abs(big.mean().item()) < 0.02 and abs(big.std().item() - 1.0) < 0.02


def test_single_image_step_plane_is_the_batch_wide_noise():
    """For one image the per-image pixel index is the global one, so step k's plane under seed s is philox_normal(s, k)."""
    for s, k in ((0, 0), (11, 3), (2 ** 64 - 1, 16)):
        assert torch.equal(philox_normal_images([s], *step_plane(k), 24, 40), philox_normal(s, k, 1, 24, 40))


@pytest.mark.parametrize("seed,pix,plane,want", [
    (0, 0, (0, 1), (1.6511781215667725, 0.8456454873085022, -0.10209861397743225)),
    (1, 5, (0, 0), (-0.5405268669128418, 1.8356248140335083, -0.13882915675640106)),
    (2 ** 64 - 1, 1234, (3, 0), (0.6664711236953735, -0.868420422077179, -2.316354513168335)),
    (0xDEADBEEFCAFEF00D, 77, (0, 1), (-1.4397529363632202, -0.1696407049894333, -0.02612435445189476)),
])
def test_known_answers(seed, pix, plane, want):
    z = philox_normal_images([seed], *plane, 64, 64)[0].reshape(3, -1)[:, pix]
    assert torch.allclose(z, torch.tensor(want), rtol=0, atol=1e-6), z


def test_oracle_decode_with_seeds_is_batch_invariant():
    from oracle.config import CDCConfig
    from oracle.weights import build_unet, synthetic_cond
    cfg = CDCConfig()
    orc = SeededOracleDecoder(cfg, build_unet(cfg, seed=0))
    orc.set_sample_schedule(3, eta=1.0)
    B, H, W = 3, 64, 64
    cond = synthetic_cond(cfg, B, H, W, index=1)
    lat = torch.zeros(B, cfg.latent_ch, H // 16, W // 16)
    seeds = [5, 2 ** 63 + 9, 42]
    traj = []
    img = orc.decode(lat, 3, seeds=seeds, cond=cond, trajectory=traj)
    assert torch.equal(traj[0], 0.8 * philox_normal_images(seeds, *XT_PLANE, H, W))
    traj1 = []
    img1 = orc.decode(lat[1:2], 3, seeds=seeds[1:2], cond=[c[1:2] for c in cond], trajectory=traj1)
    for k in range(3):
        assert (traj[k][1:2] - traj1[k]).abs().max().item() < 1e-5, k
    e = (img[1:2] - img1).abs().max().item()
    print(f"image 1 of 3 vs alone: max diff {e:.3g}")
    assert e < 1e-5
    assert orc.image_seeds is None  # nothing left bound: the next decode without seeds is the plain oracle's
    with pytest.raises(ValueError):
        orc.decode(lat, 3, seeds=seeds[:2], cond=cond)
    with pytest.raises(ValueError):
        orc.decode(lat, 3, seeds=seeds, init=traj[0], cond=cond)
