"""Trajectory recording from the captured decode graph (cdc_decode_trajectory / cdc_trajectory_wait, Decoder.decode(...,
trajectory=...), Decoder.decode_progressive): every recorded slot equals the eager step-by-step state bit for bit, the
free-running graph tracks the oracle's trajectory, and the plain decode path is untouched."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
DEV = "cuda:0"

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


def _inputs(B, H, W, index=0):
    from cdc_b200.synthetic import init_noise, latent
    return latent(B, H, W, index=index).to(DEV), init_noise(B, H, W, index=index).to(DEV)


def _buf(dec, every=1):
    B, H, W = dec.shape
    return torch.full((dec.trajectory_slots(every), B, 3, H, W), float("nan"), device=DEV)


def _eager(dec, lat, x, K):
    """set_latent, then per step: record x_t, run the step's ops eagerly, read x0_hat."""
    xs, x0s = [], []
    dec.set_latent(lat)
    for k in range(K):
        xs.append(x.clone())
        x = dec.denoise_step(x, dec.idx[k])
        x0s.append(dec._get_x0())
    return xs, x0s


@pytest.mark.parametrize("pred,eta", [("x", 0.0), ("x", 1.0), ("eps", 0.5)])
def test_graph_trajectory_equals_eager_bitwise(pred, eta):
    dec = _decoder()
    B, H, W, K = 2, 128, 192, 6
    lat, x = _inputs(B, H, W, index=2)
    try:
        dec.set_sample_schedule(K, eta=eta, pred=pred, seed=11)
        img = dec.decode(lat, K, init=x).clone()
        traj, traj0 = [], []
        img_t = dec.decode(lat, K, init=x, trajectory=traj, x0_trajectory=traj0)
        assert len(traj) == len(traj0) == K and all(t.shape == (B, 3, H, W) and t.is_cuda for t in traj + traj0)
        assert traj[0].untyped_storage().data_ptr() == traj0[-1].untyped_storage().data_ptr()  # one allocation
        assert torch.equal(img_t, img)
        xs, x0s = _eager(dec, lat, x, K)
        for k in range(K):
            assert torch.equal(traj[k], xs[k]), f"x_t of step {k}"
            assert torch.equal(traj0[k], x0s[k]), f"x0_hat of step {k}"
        # only one of the two lists: the same slots
        only = []
        dec.decode(lat, K, init=x, x0_trajectory=only)
        assert all(torch.equal(a, b) for a, b in zip(only, traj0))
    finally:
        dec.set_sample_schedule(17)


def test_free_running_trajectory_tracks_the_oracle():
    from cdc_b200 import CDCConfig, Decoder
    from oracle.config import CDCConfig as OCfg
    from oracle.sampler import OracleDecoder
    from oracle.weights import build_unet, synthetic_cond, synthetic_init
    ocfg = OCfg()
    net = build_unet(ocfg, seed=0)
    dec = Decoder(CDCConfig(), dict(net.state_dict()), device=DEV)
    orc = OracleDecoder(ocfg, net)
    B, H, W, K = 1, 128, 192, 5
    cond, x = synthetic_cond(ocfg, B, H, W, index=4), synthetic_init(B, H, W, index=4)
    lat = torch.zeros(B, 256, H // 16, W // 16)
    ref = []
    img_ref = orc.decode(lat, K, init=x, cond=cond, trajectory=ref)
    got = []
    img = dec.decode(lat, K, init=x, cond=cond, trajectory=got)
    assert len(got) == len(ref) == K
    for k in range(K):
        e = (got[k].cpu() - ref[k]).abs().max().item()
        print(f"k={k}: max|x_t - oracle| = {e:.5f}")
        assert e < 0.1, f"step {k}: {e}"
    assert torch.equal(got[0].cpu(), x)
    e = (img.cpu() - img_ref).abs().max().item()
    print(f"image: {e:.5f}")
    assert e < 0.1


def test_sparse_recording_picks_every_fourth_slot():
    dec = _decoder()
    B, H, W, K = 1, 128, 128, 17
    lat, x = _inputs(B, H, W, index=5)
    dec.set_sample_schedule(K)
    dec.set_latent(lat)
    full, full0 = _buf(dec), _buf(dec)
    dec._set_x(x)
    dec.decode_trajectory(full, full0, every=1)
    img = dec._get_x(to_image=True)
    assert dec.trajectory_slots(4) == 5
    sp, sp0 = _buf(dec, 4), _buf(dec, 4)
    dec._set_x(x)
    dec.decode_trajectory(sp, sp0, every=4)
    assert torch.equal(dec._get_x(to_image=True), img)
    for j, k in enumerate((0, 4, 8, 12, 16)):
        assert torch.equal(sp[j], full[k]) and torch.equal(sp0[j], full0[k]), f"slot {j} (step {k})"
    # every > K: slot 0 alone
    one = _buf(dec, 40)
    dec._set_x(x)
    dec.decode_trajectory(None, one, every=40)
    assert one.shape[0] == 1 and torch.equal(one[0], full0[0])


def test_plain_path_is_untouched():
    dec = _decoder()
    B, H, W, K = 1, 128, 192, 4
    lat, x = _inputs(B, H, W, index=6)
    dec.set_sample_schedule(K)
    img = dec.decode(lat, K, init=x).clone()
    ops, launches = dec.step_ops(), dec.launches_per_step()
    traj = []
    dec.decode(lat, K, init=x, trajectory=traj)
    assert dec.step_ops() == ops and dec.launches_per_step() == launches
    assert torch.equal(dec.decode(lat, K, init=x), img)
    # host inputs with a trajectory: the device path, the image returned on the host like cdc_decode_host's
    out = torch.empty(B, 3, H, W)
    traj_h = []
    got = dec.decode(lat.cpu(), K, init=x.cpu(), out=out, trajectory=traj_h)
    assert got is out and torch.equal(out, img.cpu()) and all(torch.equal(a, b) for a, b in zip(traj, traj_h))
    assert torch.equal(dec.decode(lat.cpu(), K, init=x.cpu()), img.cpu())


def test_rebinding_and_buffers_are_stateless():
    from cdc_b200 import CDCConfig, Decoder
    dec = _decoder()
    K = 3
    plan = [(1, 128, 192), (2, 64, 128), (1, 128, 192)]
    got = []
    for i, (B, H, W) in enumerate(plan):
        lat, x = _inputs(B, H, W, index=i % 2)
        t, t0 = [], []
        img = dec.decode(lat, K, init=x, trajectory=t, x0_trajectory=t0)
        got.append((torch.stack(t).clone(), torch.stack(t0).clone(), img.clone()))
    for i, (B, H, W) in enumerate(plan):
        fresh = Decoder(CDCConfig(), _weights(), device=DEV)
        lat, x = _inputs(B, H, W, index=i % 2)
        t, t0 = [], []
        img = fresh.decode(lat, K, init=x, trajectory=t, x0_trajectory=t0)
        assert torch.equal(got[i][0], torch.stack(t)) and torch.equal(got[i][1], torch.stack(t0)), f"plan entry {i}"
        assert torch.equal(got[i][2], img)
        del fresh
    # two calls at one shape, two pairs of buffers: each call writes its own (no pointer is baked into the graph)
    B, H, W = plan[0]
    lat, x = _inputs(B, H, W, index=0)
    dec.set_latent(lat)
    a, a0, b, b0 = _buf(dec), _buf(dec), _buf(dec), _buf(dec)
    dec._set_x(x)
    dec.decode_trajectory(a, a0)
    a_copy, a0_copy = a.clone(), a0.clone()
    dec._set_x(x)
    dec.decode_trajectory(b, b0)
    torch.cuda.synchronize()
    assert torch.equal(a, a_copy) and torch.equal(a0, a0_copy)
    assert torch.equal(a, got[0][0]) and torch.equal(b, got[0][0])
    assert torch.equal(a0, got[0][1]) and torch.equal(b0, got[0][1])


def test_progressive_decode_at_768x512():
    dec = _decoder()
    B, H, W, K = 1, 512, 768, 17
    lat, x = _inputs(B, H, W, index=0)
    dec.set_sample_schedule(K)
    img = dec.decode(lat, K, init=x).clone()
    bufs = []
    alloc = dec._traj_buffers

    def nan_buffers(*a):  # pre-filled with NaN: a slot read before it is written shows up
        xt, x0 = alloc(*a)
        for t in (xt, x0):
            t.fill_(float("nan"))
        bufs.append((xt, x0))
        return xt, x0

    dec._traj_buffers = nan_buffers
    try:
        seen, clones = [], []
        for k, xt, x0 in dec.decode_progressive(lat, K, init=x):
            clones.append((xt.clone(), x0.clone()))  # on the caller's stream, while the graph still runs on its own
            seen.append(k)
        torch.cuda.synchronize()
        assert seen == list(range(K))
        xt_all, x0_all = bufs[0]
        for k, (c, c0) in enumerate(clones):
            assert torch.isfinite(c).all() and torch.isfinite(c0).all(), f"slot {k} read before it was written"
            assert torch.equal(c, xt_all[k]) and torch.equal(c0, x0_all[k]), f"slot {k}"
        dec.denoise_step(xt_all[K - 1], dec.idx[K - 1])
        assert torch.equal(dec._get_x(to_image=True), img)
        # sparse, stopped early: the caller's stream waits for the graph, the next decode is exact
        for k, xt, x0 in dec.decode_progressive(lat, K, every=4, init=x):
            if k == 4:
                break
        assert torch.equal(dec.decode(lat, K, init=x), img)
        # a suspended generator: the decoder's next call waits for its graph instead of racing it on the workspace
        g = dec.decode_progressive(lat, K, init=x)
        k, xt, _ = next(g)
        assert k == 0
        assert torch.equal(dec.decode(lat, K, init=x), img)
        g.close()
        torch.cuda.synchronize()
        assert torch.equal(bufs[-1][0], xt_all) and torch.equal(bufs[-1][1], x0_all)
    finally:
        del dec._traj_buffers


def test_errors_launch_nothing():
    from cdc_b200 import CDCConfig, Decoder
    dec = Decoder(CDCConfig(), _weights(), device=DEV)
    L, ctx = dec.L, dec.ctx
    nan = torch.full((4,), float("nan"), device=DEV)
    p = C.c_void_p(nan.data_ptr())
    assert L.cdc_decode_trajectory(ctx, p, p, 1, None) != 0 and b"bind" in L.cdc_last_error(ctx)  # nothing bound
    assert L.cdc_trajectory_wait(ctx, 0) != 0 and b"no cdc_decode_trajectory" in L.cdc_last_error(ctx)
    B, H, W = 1, 64, 64
    lat, x = _inputs(B, H, W)
    dec.set_latent(lat)
    assert L.cdc_decode_trajectory(ctx, p, p, 1, None) != 0 and b"schedule" in L.cdc_last_error(ctx)
    dec.set_sample_schedule(3)
    dec._set_x(x)
    a, a0 = _buf(dec), _buf(dec)
    pa, pa0 = C.c_void_p(a.data_ptr()), C.c_void_p(a0.data_ptr())
    x_before = dec._get_x()
    assert L.cdc_decode_trajectory(ctx, pa, pa0, 0, None) != 0 and b"every" in L.cdc_last_error(ctx)
    assert L.cdc_decode_trajectory(ctx, None, None, 1, None) != 0 and b"null" in L.cdc_last_error(ctx)
    assert L.cdc_trajectory_wait(ctx, 0) != 0 and b"no cdc_decode_trajectory" in L.cdc_last_error(ctx)
    torch.cuda.synchronize()
    assert torch.isnan(a).all() and torch.isnan(a0).all() and torch.isnan(nan).all()
    assert torch.equal(dec._get_x(), x_before)  # no step ran
    dec.decode_trajectory(a, a0)
    assert L.cdc_trajectory_wait(ctx, 2) == 0
    for j in (3, -1):
        assert L.cdc_trajectory_wait(ctx, j) != 0 and b"outside" in L.cdc_last_error(ctx)
    torch.cuda.synchronize()
    assert torch.isfinite(a).all() and torch.isfinite(a0).all()
    with pytest.raises(ValueError):
        dec.decode_trajectory(a[:2], a0)  # 2 slots for a 3-step schedule
    with pytest.raises(ValueError):
        dec.decode_trajectory(a.double())
    with pytest.raises(ValueError):
        dec.decode_trajectory(a.cpu())
    with pytest.raises(ValueError):
        dec.decode_trajectory(None, None)
    with pytest.raises(ValueError):
        dec.decode_trajectory(a, every=0)
    with pytest.raises(ValueError):
        next(dec.decode_progressive(lat, 3, init=x, every=0))
    del dec
