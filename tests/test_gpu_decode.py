"""Step- and decode-level parity of the CUDA path against the CPU oracle on a real B200
(SURVEY.md A.7: teacher-forced per-step max-abs <= 1e-2; graph replay == eager launches)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False  # the torch checker must be true fp32
torch.backends.cuda.matmul.allow_tf32 = False
DEV = "cuda:0"
TOL = 1e-2  # BASELINE.json north_star: reconstructions within 1e-2 max-abs of the fp32 oracle per step

_cache = {}


def _setup(with_context=False):
    key = ("ctx" if with_context else "unet")
    if key in _cache:
        return _cache[key]
    from cdc_b200 import CDCConfig, Decoder
    from oracle.config import CDCConfig as OCfg
    from oracle.sampler import OracleDecoder
    from oracle.weights import build_codec, build_unet
    ocfg = OCfg()
    net = build_unet(ocfg, seed=0)
    weights = dict(net.state_dict())
    codec = None
    if with_context:
        codec = build_codec(ocfg, seed=1)
        weights.update({"context." + k: v for k, v in codec.context.state_dict().items()})
    dec = Decoder(CDCConfig(), weights, device=DEV)
    orc = OracleDecoder(ocfg, net, context_net=codec.context if codec else None)
    _cache[key] = (dec, orc, ocfg)
    return _cache[key]


@pytest.mark.parametrize("shape", [(1, 256, 256), (2, 128, 192), (1, 64, 64), (1, 128, 384), (3, 64, 128)])
def test_teacher_forced_step_parity(shape):
    from oracle.weights import synthetic_cond, synthetic_init
    dec, orc, ocfg = _setup()
    B, H, W = shape
    dec.set_sample_schedule(17)
    orc.set_sample_schedule(17)
    assert dec.idx == orc.sched.idx
    for k in range(17):
        c0, c1 = dec.coeffs(k)
        assert c0 == float(orc.sched.c0[k]) and c1 == float(orc.sched.c1[k])
    cond = synthetic_cond(ocfg, B, H, W)
    x = synthetic_init(B, H, W)
    worst = 0.0
    for t in (999, 500, 0):
        x0_ref = orc.predict_x0(x, t, cond)
        xp_ref = orc.denoise_step(x, t, cond)
        xp = dec.denoise_step(x, t, cond).cpu()
        x0 = dec._get_x0().cpu()
        e0 = (x0 - x0_ref).abs().max().item()
        e1 = (xp - xp_ref).abs().max().item()
        print(f"shape {shape} t={t}: max|x0-x0_ref|={e0:.5f} max|xprev-ref|={e1:.5f}")
        worst = max(worst, e1)
        assert torch.isfinite(xp).all()
        assert e1 <= TOL, f"t={t}: x_prev max-abs {e1}"
        # (raw x0_hat: 1e-2 on the last step, where it IS the image; 3e-2 at noisy steps, where it is multiplied by
        # c0 <= 0.3 before it reaches x_prev -- the same gate as the headline test in test_gpu_parity_r2.py)
        assert e0 <= (TOL if t == 0 else 3 * TOL), f"t={t}: x0_hat max-abs {e0}"
    try:
        dec.denoise_step(x, 998, cond)
        assert False, "t outside the schedule must raise"
    except ValueError:
        pass


def test_full_trajectory_teacher_forced_and_graph_equals_eager():
    from oracle.weights import synthetic_cond, synthetic_init
    dec, orc, ocfg = _setup()
    B, H, W, K = 1, 128, 128, 5
    cond = synthetic_cond(ocfg, B, H, W, index=3)
    x = synthetic_init(B, H, W, index=3)
    traj = []
    img_ref = orc.decode(torch.zeros(B, 256, H // 16, W // 16), K, init=x, cond=cond, trajectory=traj)
    dec.set_sample_schedule(K)
    for k in range(K):  # teacher forcing: feed the oracle's x_t
        xp = dec.denoise_step(traj[k], orc.sched.idx[k], cond).cpu()
        ref = traj[k + 1] if k + 1 < K else (img_ref * 2 - 1)
        if k + 1 == K:
            xp = xp.clamp(-1, 1)
        e = (xp - ref).abs().max().item()
        print(f"k={k}: {e:.5f}")
        assert e <= TOL
    # eager free-running vs one graph launch: bitwise identical
    xe = x.clone()
    for k in range(K):
        xe = dec.denoise_step(xe, orc.sched.idx[k])
    img_e = ((xe.clamp(-1, 1) + 1) / 2).cpu()
    img_g = dec.decode(torch.zeros(B, 256, H // 16, W // 16), K, init=x.to(DEV), cond=cond).cpu()
    assert torch.equal(img_e, img_g)
    img_g2 = dec.decode(torch.zeros(B, 256, H // 16, W // 16), K, init=x.to(DEV), cond=cond).cpu()
    assert torch.equal(img_g, img_g2)
    fr = (img_g - img_ref).abs().max().item()
    print(f"free-running decode max-abs vs oracle: {fr:.5f}")
    assert fr < 0.1


def test_context_net_and_host_decode():
    from oracle.weights import synthetic_init, synthetic_latent
    dec, orc, ocfg = _setup(with_context=True)
    B, H, W, K = 1, 128, 192, 3
    lat = synthetic_latent(B, H, W)
    x = synthetic_init(B, H, W)
    with torch.no_grad():
        cond_ref = orc.context_net(lat)
    img_ref = orc.decode(lat, K, init=x, cond=cond_ref)
    img = dec.decode(lat, K, init=x)  # host tensors -> cdc_decode_host
    assert img.device.type == "cpu" and img.shape == (B, 3, H, W)
    e = (img - img_ref).abs().max().item()
    print(f"host decode (context net on GPU) max-abs vs oracle: {e:.5f}")
    assert e < 0.1
    img2 = dec.decode(lat.to(DEV), K, init=x.to(DEV)).cpu()
    assert torch.equal(img, img2)
    # page-locked caller buffers are copied from / to directly (no staging copies): same result, returned in `out`
    out = torch.empty_like(img).pin_memory()
    img3 = dec.decode(lat.pin_memory(), K, init=x.pin_memory(), out=out)
    assert img3 is out and torch.equal(img, img3)


def test_flops_and_launch_accounting():
    from oracle.unet import unet_flops
    dec, orc, ocfg = _setup()
    dec.set_sample_schedule(17)
    dec.bind(1, 256, 256)
    assert abs(dec.flops_per_step() / unet_flops(ocfg, 1, 256, 256) - 1.0) < 1e-6
    # every op is one kernel of ours except the memset node that clears the GroupNorm accumulators
    assert dec.launches_per_step() == len(dec.step_ops()) - 1 > 60
    # GroupNorm 1 of the ResBlocks whose conv2 runs the kh-fused kernel is applied inside that conv: no pass of its own
    names = [o[0] for o in dec.step_ops()]
    assert any(n.endswith("conv2+gn_in") for n in names)
    assert not any(n.startswith("down.0.rb1.gn1") for n in names) and any(n.startswith("down.0.rb1.gn2") for n in names)


@pytest.mark.parametrize("shape", [(1, 256, 384), (2, 128, 192), (3, 64, 128), (1, 512, 768)])
def test_fused_input_groupnorm_is_bit_identical(shape):
    """conv2 applying GroupNorm 1 + FiLM + SiLU to its input rows in shared memory (default) must reproduce, bit for bit,
    the plan that runs the same arithmetic as a pass of its own (plan option FUSE_APPLY = 0): same fp16 activations, same
    MMA order."""
    from cdc_b200 import CDCConfig, Decoder, _ffi
    from cdc_b200.synthetic import init_noise, latent, random_weights
    B, H, W = shape
    w = random_weights(CDCConfig(), seed=0, with_context=True)
    lat, x = latent(B, H, W, index=3), init_noise(B, H, W, index=3)
    outs, n_gn1 = [], []
    for fuse in (2, 0):
        d = Decoder(CDCConfig(), w, device=DEV)
        d.set_plan_option(_ffi.OPT_FUSE_APPLY, fuse)
        outs.append(d.decode(lat, 3, init=x).clone())
        n_gn1.append(sum(1 for o in d.step_ops() if ".gn1." in o[0]))
        del d
    assert n_gn1[0] < n_gn1[1] == 18  # (levels too small for the kh-fused kernel keep the pass)
    assert torch.isfinite(outs[0]).all()
    assert torch.equal(outs[0], outs[1]), f"max diff {(outs[0].float() - outs[1].float()).abs().max().item()}"


def test_wrong_shapes_fail_loudly():
    dec, _, _ = _setup()
    with pytest.raises(RuntimeError):
        dec.bind(1, 100, 256)


def test_batch_beyond_the_groupnorm_table_is_refused_at_bind():
    """193 images need a 49 KB GroupNorm statistics table: cdc_bind_io refuses the batch (instead of a later CUDA error
    from the first step), and the context then binds and decodes a valid shape as a fresh one does."""
    from cdc_b200 import CDCConfig, Decoder
    from cdc_b200.synthetic import init_noise, latent, random_weights
    w = random_weights(CDCConfig(), seed=0, with_context=True)
    a = Decoder(CDCConfig(), w, device=DEV)
    a.bind(2, 64, 128)
    with pytest.raises(RuntimeError, match="GroupNorm"):
        a.bind(193, 64, 64)
    out = a.decode(latent(2, 64, 128, index=1), 3, init=init_noise(2, 64, 128, index=1))
    ref = Decoder(CDCConfig(), w, device=DEV).decode(latent(2, 64, 128, index=1), 3, init=init_noise(2, 64, 128, index=1))
    assert torch.isfinite(ref).all() and torch.equal(out, ref)


def test_rebinding_shapes_and_schedules_is_stateless():
    """One context decodes different shapes / step counts back to back (workspace, tensor maps, pinned staging and the
    graph are rebuilt); every result equals the one a fresh context produces."""
    from cdc_b200 import CDCConfig, Decoder
    from cdc_b200.synthetic import init_noise, latent, random_weights
    w = random_weights(CDCConfig(), seed=0, with_context=True)
    a = Decoder(CDCConfig(), w, device=DEV)
    outs = []
    plan = [(1, 64, 64, 5), (2, 128, 192, 7), (1, 64, 64, 5), (1, 64, 128, 3)]
    for i, (B, H, W, K) in enumerate(plan):
        outs.append(a.decode(latent(B, H, W, index=i), K, init=init_noise(B, H, W, index=i)).clone())
    for i, (B, H, W, K) in enumerate(plan):
        b = Decoder(CDCConfig(), w, device=DEV)
        ref = b.decode(latent(B, H, W, index=i), K, init=init_noise(B, H, W, index=i))
        assert torch.isfinite(ref).all() and torch.equal(outs[i], ref), f"plan entry {i} differs after re-binding"
        del b
