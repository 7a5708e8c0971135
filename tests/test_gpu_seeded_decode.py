"""Per-image seeds on a real B200 (Decoder.decode(..., seeds=...), cdc_set_image_seeds / cdc_init_noise /
cdc_decode_host_seeded): x_T and the eta > 0 sampler noise match the numpy reference (tests/seeded_reference.py), an image
decodes the same alone and inside a batch, the graph, eager, host and device paths agree bit for bit, and decodes without
seeds are untouched."""
import ctypes as C

import pytest
import torch

from tests.seeded_reference import XT_PLANE, SeededOracleDecoder, philox_normal_images, step_plane

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
DEV = "cuda:0"
GAMMA = 0.8

_cache = {}


def _weights():
    if "w" not in _cache:
        from cdc_b200 import CDCConfig
        from cdc_b200.synthetic import random_weights
        _cache["w"] = random_weights(CDCConfig(), seed=0, with_context=True)
    return _cache["w"]


def _decoder():
    if "dec" not in _cache:
        from cdc_b200 import CDCConfig, Decoder
        _cache["dec"] = Decoder(CDCConfig(), _weights(), device=DEV)
    return _cache["dec"]


def _latent(B, H, W, index=0):
    from cdc_b200.synthetic import latent
    return latent(B, H, W, index=index).to(DEV)


def _device_xT(dec, lat, seeds):
    dec.set_latent(lat)
    dec.set_image_seeds(seeds)
    dec.init_noise(GAMMA)
    return dec._get_x()


def test_device_xT_matches_the_reference():
    dec = _decoder()
    B, H, W = 3, 128, 192
    seeds = [1, 2 ** 64 - 2, 0x5EED]
    dec.set_sample_schedule(4)
    x = _device_xT(dec, _latent(B, H, W), seeds)
    ref = GAMMA * philox_normal_images(seeds, *XT_PLANE, H, W)
    e = (x.cpu() - ref).abs().max().item()
    print(f"x_T vs reference: max diff {e:.3g}")
    assert e < 1e-5


def test_xT_is_batch_invariant_bitwise():
    dec = _decoder()
    H, W = 128, 192
    dec.set_sample_schedule(4)
    x3 = _device_xT(dec, _latent(3, H, W), [10, 11, 12]).clone()
    x1 = _device_xT(dec, _latent(1, H, W), [12])
    assert torch.equal(x3[2:3], x1)


def test_per_image_sampler_noise_matches_the_reference():
    """z_k recovered from the trajectory, z_k = (x_{k+1} - c0 clamp(x0_hat_k) - c1 x_k) / sigma_k, is the reference's."""
    dec = _decoder()
    B, H, W, K = 3, 128, 192, 4
    seeds = [3, 2 ** 40 + 1, 99]
    dec.set_sample_schedule(K, eta=1.0, seed=123)
    try:
        xt, x0 = [], []
        dec.decode(_latent(B, H, W, index=1), K, seeds=seeds, trajectory=xt, x0_trajectory=x0)
        checked = 0
        for k in range(K - 1):
            c0, c1, e0, e1, sg = dec.coeffs5(k)
            if sg == 0.0:
                continue
            z = (xt[k + 1] - c0 * x0[k].clamp(-1.0, 1.0) - c1 * xt[k]) / sg
            ref = philox_normal_images(seeds, *step_plane(k), H, W)
            e = (z.cpu() - ref).abs().max().item()
            # the recovery divides fp32 rounding of the x's (a few ulp of |x|) by sigma: sigma is 0.006 at t = 999
            tol = 1e-4 + 8 * 2.0 ** -23 * (xt[k + 1].abs().max().item() + abs(c0) + c1 * xt[k].abs().max().item()) / sg
            print(f"step {k}: sigma {sg:.4f}, max |z - reference| = {e:.3g} (tolerance {tol:.3g})")
            assert e < tol, k
            checked += 1
        assert checked == K - 1
    finally:
        dec.set_sample_schedule(17)


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_image_decodes_the_same_alone_and_in_a_batch(eta):
    dec = _decoder()
    H, W, K = 128, 192, 5
    seeds = [21, 22, 23]
    lat = _latent(3, H, W, index=2)
    dec.set_sample_schedule(K, eta=eta, seed=5)
    try:
        t3, t30 = [], []
        img3 = dec.decode(lat, K, seeds=seeds, trajectory=t3, x0_trajectory=t30)
        t3, t30, img3 = [t[1:2].clone() for t in t3], [t[1:2].clone() for t in t30], img3[1:2].clone()
        t1, t10 = [], []
        img1 = dec.decode(lat[1:2], K, seeds=seeds[1:2], trajectory=t1, x0_trajectory=t10)
        worst, bitwise = 0.0, True
        for k in range(K):
            for a, b in ((t3[k], t1[k]), (t30[k], t10[k])):
                worst = max(worst, (a - b).abs().max().item())
                bitwise = bitwise and torch.equal(a, b)
        e = (img3 - img1).abs().max().item()
        bitwise = bitwise and torch.equal(img3, img1)
        print(f"eta {eta}: image 1 of 3 vs alone: max diff trajectory {worst:.3g}, image {e:.3g}, bitwise {bitwise}")
        assert worst < 1e-2 and e < 1e-2
    finally:
        dec.set_sample_schedule(17)


def test_free_running_seeded_decode_tracks_the_oracle():
    from cdc_b200 import CDCConfig, Decoder
    from oracle.config import CDCConfig as OCfg
    from oracle.weights import build_unet, synthetic_cond
    ocfg = OCfg()
    net = build_unet(ocfg, seed=0)
    dec = Decoder(CDCConfig(), dict(net.state_dict()), device=DEV)
    orc = SeededOracleDecoder(ocfg, net)
    B, H, W, K = 2, 128, 192, 5
    seeds = [8, 2 ** 64 - 9]
    dec.set_sample_schedule(K, eta=1.0)
    orc.set_sample_schedule(K, eta=1.0)
    cond = synthetic_cond(ocfg, B, H, W, index=4)
    lat = torch.zeros(B, 256, H // 16, W // 16)
    ref = []
    img_ref = orc.decode(lat, K, seeds=seeds, cond=cond, trajectory=ref)
    got = []
    img = dec.decode(lat, K, seeds=seeds, cond=cond, trajectory=got)
    for k in range(K):
        e = (got[k].cpu() - ref[k]).abs().max().item()
        print(f"k={k}: max|x_t - oracle| = {e:.5f}")
        assert e < 0.1, f"step {k}: {e}"
    e = (img.cpu() - img_ref).abs().max().item()
    print(f"image: {e:.5f}")
    assert e < 0.1


def test_graph_equals_eager_steps_bitwise():
    """decode(seeds=) == set_image_seeds + init_noise, x_T read back and fed in again, then K eager denoise_steps."""
    dec = _decoder()
    B, H, W, K = 2, 128, 192, 5
    seeds = [31, 32]
    lat = _latent(B, H, W, index=3)
    dec.set_sample_schedule(K, eta=1.0, seed=7)
    try:
        traj = []
        img = dec.decode(lat, K, seeds=seeds, trajectory=traj).clone()
        x = _device_xT(dec, lat, seeds).clone()
        assert torch.equal(x, traj[0])
        for k in range(K):
            assert torch.equal(x, traj[k]), f"x_t of step {k}"
            x = dec.denoise_step(x, dec.idx[k])
        assert torch.equal(dec._get_x(to_image=True), img)
        # decode_progressive with the same seeds yields the same slots
        for k, xt, _ in dec.decode_progressive(lat, K, seeds=seeds):
            assert torch.equal(xt, traj[k]), f"progressive slot {k}"
    finally:
        dec.set_sample_schedule(17)


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_host_path_equals_device_path(eta):
    dec = _decoder()
    B, H, W, K = 2, 128, 192, 4
    seeds = torch.tensor([2 ** 63 + 1, 77], dtype=torch.uint64)
    lat = _latent(B, H, W, index=4)
    dec.set_sample_schedule(K, eta=eta, seed=1)
    try:
        img_d = dec.decode(lat, K, seeds=seeds).cpu()
        img_h = dec.decode(lat.cpu(), K, seeds=seeds)
        assert not img_h.is_cuda and torch.equal(img_h, img_d)
        out = torch.empty(B, 3, H, W).pin_memory()
        assert dec.decode(lat.cpu(), K, seeds=[2 ** 63 + 1, 77], out=out) is out and torch.equal(out, img_d)
        # int64 tensors are accepted too
        assert torch.equal(dec.decode(lat, K, seeds=torch.tensor([5, 6])).cpu(), dec.decode(lat.cpu(), K, seeds=[5, 6]))
    finally:
        dec.set_sample_schedule(17)


def test_codec_decompress_passes_seeds_through():
    from cdc_b200 import CDCConfig, Codec, Decoder
    from oracle.config import CDCConfig as OCfg
    from oracle.weights import build_codec, build_unet, synthetic_image
    ocfg = OCfg()
    oc = build_codec(ocfg, seed=1)
    w = dict(build_unet(ocfg, seed=0).state_dict())
    for k, v in oc.state_dict().items():
        w[("context." + k[len("context."):]) if k.startswith("context.") else ("codec." + k)] = v
    dec = Decoder(CDCConfig(), w, device=DEV)
    gauss, fact = oc.tables()
    codec = Codec(dec, gauss_tables=gauss, fact_tables=fact, median=oc.prior.median)
    B, H, W, K = 2, 128, 128, 4
    data, enc = codec.compress(synthetic_image(B, H, W, index=3))
    dec.set_sample_schedule(K, eta=0.5, seed=2)
    img = codec.decompress_bytes(data, K, seeds=[4, 5])
    assert img.shape == (B, 3, H, W)
    y_hat = codec.latent_from_symbols(enc["qz"], enc["q"])[0]
    assert torch.equal(img, dec.decode(y_hat, K, seeds=[4, 5]))
    assert torch.equal(codec.decompress(enc["qz"], enc["q"], K, seeds=[4, 5]), img)
    assert not torch.equal(codec.decompress_bytes(data, K, seeds=[4, 6])[1], img[1])


def test_decodes_without_seeds_are_untouched():
    dec = _decoder()
    B, H, W, K = 2, 128, 192, 4
    from cdc_b200.synthetic import init_noise
    lat = _latent(B, H, W, index=5)
    x = init_noise(B, H, W, index=5).to(DEV)
    dec.set_sample_schedule(K)
    a = dec.decode(lat, K, init=x).clone()
    b = dec.decode(lat.cpu(), K, seed=0).clone()
    ops, launches = dec.step_ops(), dec.launches_per_step()
    dec.decode(lat, K, seeds=[1, 2])
    assert torch.equal(dec.decode(lat, K, init=x), a)
    assert torch.equal(dec.decode(lat.cpu(), K, seed=0), b)
    assert dec.step_ops() == ops and dec.launches_per_step() == launches
    # eta > 0 without seeds: the batch-wide seed keys the noise, as before
    try:
        imgs = []
        for s in (1, 1, 2):
            dec.set_sample_schedule(K, eta=1.0, seed=s)
            dec.decode(lat, K, seeds=[3, 4])  # a seeded decode in between leaves nothing bound
            imgs.append(dec.decode(lat, K, init=x).clone())
        assert torch.equal(imgs[0], imgs[1]) and not torch.equal(imgs[0], imgs[2])
    finally:
        dec.set_sample_schedule(17)


def test_errors():
    from cdc_b200 import CDCConfig, Decoder
    dec = Decoder(CDCConfig(), _weights(), device=DEV)
    L, ctx = dec.L, dec.ctx
    B, H, W, K = 2, 64, 64, 3
    lat = _latent(B, H, W)
    dec.set_sample_schedule(K)
    with pytest.raises(ValueError):
        dec.decode(lat, K, seeds=[1])  # wrong length
    with pytest.raises(ValueError):
        dec.decode(lat, K, seeds=[1, 2], init=torch.zeros(B, 3, H, W))
    for bad in ([-1, 2], [1, 2 ** 64], [1.5, 2], [True, 2]):
        with pytest.raises(ValueError):
            dec.decode(lat, K, seeds=bad)
    with pytest.raises(ValueError):
        dec.decode(lat, K, seeds=torch.tensor([1.0, 2.0]))
    dec.set_latent(lat)
    with pytest.raises(ValueError):
        dec.set_image_seeds([1, 2, 3])
    assert L.cdc_init_noise(ctx, C.c_float(GAMMA), None) != 0 and b"no per-image seeds" in L.cdc_last_error(ctx)
    out = torch.empty(B, 3, H, W)
    lh = lat.cpu().contiguous()
    assert L.cdc_decode_host_seeded(ctx, C.c_void_p(lh.data_ptr()), C.c_float(GAMMA), C.c_void_p(out.data_ptr()), None) != 0
    arr = (C.c_uint64 * 3)(1, 2, 3)
    assert L.cdc_set_image_seeds(ctx, arr, 3, None) != 0 and b"batch of 2" in L.cdc_last_error(ctx)
    assert L.cdc_set_image_seeds(ctx, arr, 2, None) == 0
    assert L.cdc_init_noise(ctx, C.c_float(GAMMA), None) == 0
    dec.set_image_seeds(None)
    assert L.cdc_init_noise(ctx, C.c_float(GAMMA), None) != 0
    # a bind to another shape drops the seeds
    dec.set_image_seeds([1, 2])
    dec.set_latent(_latent(1, H, W))
    assert L.cdc_init_noise(ctx, C.c_float(GAMMA), None) != 0 and b"no per-image seeds" in L.cdc_last_error(ctx)
    del dec
