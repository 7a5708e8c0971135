"""Batch-invariant plans on a real B200 (include/cdc_b200.h cdc_set_batch_invariant, Decoder(..., batch_invariant=True)):
every op of every sequence is laid out per image as for a batch of 1, and everything computed for an image -- context maps,
the trajectory, the final image, the encoder's y / z / mu / sigma / q / qz, the CDC5 symbols and the 8-bit pixels -- is bit
for bit what the same image gives alone, at any position of any batch, in any shard of a data-parallel run, and what the
default plan gives at batch 1."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# the geometry of an op that decides how its images' sums are ordered (grid sizes may differ with the batch)
FIELDS = ("kind", "kernel", "bn", "tr", "nseg", "strips", "rows", "ch", "staged", "res1", "apply")
SHAPES = [(128, 192), (512, 768)]

_cache = {}


def _parts():
    if "p" not in _cache:
        from tests.test_gpu_codec import _setup
        _, oc, _, w = _setup()
        _cache["p"] = (oc, w, oc.tables())
    return _cache["p"]


def _codec(invariant):
    key = ("codec", invariant)
    if key not in _cache:
        from cdc_b200 import CDCConfig, Codec, Decoder
        oc, w, (gauss, fact) = _parts()
        dec = Decoder(CDCConfig(), w, device=DEV, batch_invariant=invariant)
        _cache[key] = Codec(dec, gauss_tables=gauss, fact_tables=fact, median=oc.prior.median)
    return _cache[key]


def _latent(B, H, W, index):
    from cdc_b200.synthetic import latent
    return latent(B, H, W, index=index).to(DEV)


def _describe(dec):
    """{sequence: [(op name, geometry)]} of the bound plan"""
    from cdc_b200 import _ffi
    out = {}
    for seq in (_ffi.SEQ_STEP, _ffi.SEQ_CONTEXT, _ffi.SEQ_ENCODER, _ffi.SEQ_HYPER_ENC, _ffi.SEQ_HYPER_DEC):
        n = dec.L.cdc_seq_num_ops(dec.ctx, seq)
        assert n > 0, seq
        out[seq] = [(dec.L.cdc_seq_op_name(dec.ctx, seq, i).decode(),
                     tuple(getattr(dec.step_op_desc(i, seq), f) for f in FIELDS)) for i in range(n)]
    return out


def _plan(dec, B, H, W):
    dec.bind(B, H, W)
    return _describe(dec)


def _multi_strip_ops(dec, B):
    """strip-conv ops of the bound step plan in which some CTA runs more than one strip"""
    n = dec.L.cdc_seq_num_ops(dec.ctx, 0)
    return [i for i in range(n) if dec.step_op_desc(i).kernel == 2 and
            B * dec.step_op_desc(i).nseg * dec.step_op_desc(i).strips > dec.step_op_desc(i).g1]


def _decode(dec, lat, K, eta, seeds):
    """(image, x_t trajectory, raw x0_hat trajectory), [B, 3, H, W] and [K, B, 3, H, W]"""
    if dec.steps != K or dec.sampler != (eta, "x", 5):
        dec.set_sample_schedule(K, eta=eta, seed=5)
    xt, x0 = [], []
    img = dec.decode(lat, K, seeds=seeds, trajectory=xt, x0_trajectory=x0)
    return img.clone(), torch.stack([t.clone() for t in xt]), torch.stack([t.clone() for t in x0])


def _assert_same(batch, b, alone):
    img, xt, x0 = batch
    i1, t1, z1 = alone
    assert torch.equal(img[b:b + 1], i1), f"image {b}: final image"
    assert torch.equal(xt[:, b:b + 1], t1), f"image {b}: x_t trajectory"
    assert torch.equal(x0[:, b:b + 1], z1), f"image {b}: x0_hat trajectory"


@pytest.mark.parametrize("H,W", SHAPES)
def test_every_op_is_laid_out_as_for_batch_1(H, W):
    inv, dflt = _codec(True).dec, _codec(False).dec
    ref = _plan(dflt, 1, H, W)
    assert _plan(inv, 1, H, W) == ref
    for B in (2, 3, 8):
        assert _plan(inv, B, H, W) == ref, f"batch {B}"


@pytest.mark.parametrize("H,W,K,eta", [(128, 192, 5, 0.0), (128, 192, 5, 1.0), (512, 768, 17, 0.0)])
def test_decode_is_bitwise_per_image(H, W, K, eta):
    dec = _codec(True).dec
    seeds = [11, 2 ** 63 + 5, 77]
    lat = _latent(3, H, W, index=4)
    batch = _decode(dec, lat, K, eta, seeds)
    assert _multi_strip_ops(dec, 3), "no CTA runs several strips: the test would not exercise the phantom rows"
    for b in range(3):
        _assert_same(batch, b, _decode(dec, lat[b:b + 1], K, eta, [seeds[b]]))


@pytest.mark.parametrize("H,W,B", [(128, 192, 5), (512, 768, 8)])
def test_same_image_first_and_last_in_the_batch(H, W, B):
    dec = _codec(True).dec
    K = 5
    lat = _latent(B, H, W, index=6)
    lat[B - 1] = lat[0]
    seeds = [100 + i for i in range(B)]
    seeds[B - 1] = seeds[0]
    batch = _decode(dec, lat, K, 0.0, seeds)
    if B == 8:  # every level-0 strip conv's CTAs run several rounds of strips
        assert len(_multi_strip_ops(dec, B)) >= 4
    img, xt, x0 = batch
    assert torch.equal(img[0], img[B - 1]) and torch.equal(xt[:, 0], xt[:, B - 1]) and torch.equal(x0[:, 0], x0[:, B - 1])
    alone = _decode(dec, lat[:1], K, 0.0, seeds[:1])
    _assert_same(batch, 0, alone)
    _assert_same(batch, B - 1, alone)


@pytest.mark.parametrize("H,W,K", [(128, 192, 5), (512, 768, 17)])
def test_invariant_batch_1_is_the_default_batch_1(H, W, K):
    lat = _latent(1, H, W, index=8)
    for eta in (0.0, 1.0):
        _assert_same(_decode(_codec(False).dec, lat, K, eta, [21]), 0, _decode(_codec(True).dec, lat, K, eta, [21]))


def test_ctas_that_span_images():
    """16 SMs: the strip convs' CTAs run several strips each, of both images (B = 2) or of one (B = 1)."""
    from cdc_b200 import _ffi
    dec = _codec(True).dec
    H, W, K = 128, 192, 4
    seeds = [5, 6]
    lat = _latent(2, H, W, index=9)
    dec.set_plan_option(_ffi.OPT_PLAN_SMS, 16)
    try:
        batch = _decode(dec, lat, K, 1.0, seeds)
        assert len(_multi_strip_ops(dec, 2)) >= 4
        for b in range(2):
            _assert_same(batch, b, _decode(dec, lat[b:b + 1], K, 1.0, [seeds[b]]))
    finally:
        dec.set_plan_option(_ffi.OPT_PLAN_SMS, 0)


@pytest.mark.parametrize("H,W", SHAPES)
def test_context_net_and_encoder_are_bitwise_per_image(H, W):
    from oracle.weights import synthetic_image
    codec = _codec(True)
    dec = codec.dec
    B = 3
    lat = _latent(B, H, W, index=10)
    dec.set_latent(lat)
    cond = [c.clone() for c in dec.get_cond()]
    img = synthetic_image(B, H, W, index=2)
    keys = ("y", "z", "mu", "sigma", "q", "qz")
    enc = {k: v.clone() for k, v in codec.encode(img).items() if k in keys}
    for b in range(B):
        dec.set_latent(lat[b:b + 1])
        for i, c in enumerate(dec.get_cond()):
            assert torch.equal(cond[i][b:b + 1], c), f"image {b}: c{i}"
        e1 = codec.encode(img[b:b + 1])
        for k in keys:
            assert torch.equal(enc[k][b:b + 1], e1[k]), f"image {b}: {k}"


def test_bytes_and_pixels_do_not_depend_on_the_batch():
    from tests.test_gpu_bitstream_cabi import _rgb8
    codec = _codec(True)
    H, W, K = 128, 192, 5
    u8 = _rgb8(3, H, W, index=5)
    data3 = codec.compress_rgb8(u8)
    data1 = codec.compress_rgb8(u8[1:2].contiguous())
    qz3, q3 = codec.decode_symbols(data3)
    qz1, q1 = codec.decode_symbols(data1)
    assert torch.equal(qz3[1:2], qz1) and torch.equal(q3[1:2], q1)
    px3 = codec.decompress_rgb8(data3, K, seeds=[3, 4, 5])
    px1 = codec.decompress_rgb8(data1, K, seeds=[4])
    assert px3.dtype == torch.uint8 and torch.equal(px3[1:2], px1)


def test_sharded_decode_is_the_same_for_every_world_size():
    """dp.shard_indices on one GPU: each rank's images decoded as one batch, assembled by index."""
    from cdc_b200.dp import shard_indices
    dec = _codec(True).dec
    H, W, K, N = 128, 192, 5, 5
    lat = _latent(N, H, W, index=12)
    seeds = [1000 + 7 * i for i in range(N)]
    dec.set_sample_schedule(K, eta=1.0, seed=5)
    images = {}
    for world in (1, 2, 3):
        out = torch.empty(N, 3, H, W)
        for rank in range(world):
            idx = shard_indices(N, rank, world)
            out[idx] = dec.decode(lat[idx], K, seeds=[seeds[i] for i in idx]).cpu()
        images[world] = out
    assert torch.equal(images[1], images[2]) and torch.equal(images[1], images[3])


def test_mode_switch_replans_at_the_next_bind_and_bad_values_are_refused():
    from cdc_b200 import _ffi
    dec = _codec(True).dec
    L = dec.L
    assert L.cdc_set_batch_invariant(dec.ctx, 2) == _ffi.ERR_SHAPE
    assert L.cdc_set_batch_invariant(dec.ctx, -1) == _ffi.ERR_SHAPE
    B, H, W = 8, 128, 192
    inv = _plan(dec, B, H, W)
    try:
        assert L.cdc_set_batch_invariant(dec.ctx, 0) == 0
        assert _describe(dec) == inv  # the bound plan stands until the next bind ...
        assert L.cdc_bind_io(dec.ctx, B, H, W) == 0  # ... which re-plans for the same shape
        dflt = _describe(dec)
        assert dflt != inv
        assert dflt == _plan(_codec(False).dec, B, H, W)
    finally:
        assert L.cdc_set_batch_invariant(dec.ctx, 1) == 0
        assert L.cdc_bind_io(dec.ctx, B, H, W) == 0
    assert _describe(dec) == inv
