"""Teacher-forced per-op parity of one denoise step on a real B200.

Every op of the bound step plan runs alone (cdc_run_step_op) on the GPU's own outputs of the ops before it; its outputs
are compared with a float64 reference of that one operation, computed on the GPU from a snapshot of exactly what the
kernel read.  A failure therefore names one kernel instance.  The op descriptions (cdc_step_op_describe) say which
tensors an op reads and writes and which kernel instantiation runs it; everything an op does not declare as its output
must stay bitwise unchanged.

Conv weights are rounded to a fixed-point grid (multiples of 2^-m, every sum of four weights below 2^11 grid steps), so
the fp16 repack and the pre-summed nearest-x2 parity weights are exact and the only conv error left is the fp32
accumulation order: the tolerances (tests/op_reference.py, shared with the codec sequences' check) are derived from that,
op by op.

With B > 1, image b's x_t and cond maps are scaled by 2^((b mod 4) - 1), so that a kernel that takes another image's
GroupNorm statistics, coefficients or seed is off by a factor.  The op descriptions carry the launch geometry; the coverage
test requires that the configurations ran the strip kernel's unit loop in every regime where state carries from one unit
(one strip of one image) to the next: several units per CTA, units of two images in one CTA, one-row and uneven strips,
ragged segments and strips longer than the accumulator ring.
"""
import time

import pytest
import torch

from tests.op_reference import (DEV, SUB16, U16, SeqBuffers, _check_conv, _check_gn_apply, _check_gn_stats,
                                GeometrySeen, _fixed_point_unet, _geom, _inst, _kf_cases, _kf_key, _ratio, image_scale)

pytestmark = pytest.mark.gpu

# (name, (B, H, W), steps K, eta, steps k checked, plan options; "seeds": bind per-image seeds)
CONFIGS = [
    ("headline_768x512", (1, 512, 768), 17, 0.0, (0, 16), {}),
    ("two_images_128x192", (2, 128, 192), 17, 0.0, (8,), {}),
    ("three_images_64x128", (3, 64, 128), 17, 0.0, (8,), {}),
    ("tall_64x1024", (1, 1024, 64), 17, 0.0, (8,), {}),
    ("ragged_704x256", (1, 256, 704), 17, 0.0, (8,), {}),
    ("general_kernel_768x512", (1, 512, 768), 17, 0.0, (16,), {"OPT_KF": 0}),
    ("ddim_noise_128x192", (2, 128, 192), 17, 1.0, (3,), {}),
    ("cfg1_256x256", (1, 256, 256), 17, 0.0, (8,), {}),
    ("cfg3_16x256x256", (16, 256, 256), 100, 0.0, (50,), {}),
    ("cfg5_2048x2048", (1, 2048, 2048), 17, 0.0, (8,), {}),
    # level 0: 192 strip columns on 148 CTAs, so every level-0 conv (the final conv's DDIM epilogue, with each image's
    # own seed, included) runs units of several images on one CTA
    ("max_batch_192x64x64", (192, 64, 64), 17, 1.0, (3,), {"seeds": True}),
    ("one_row_64x1024", (1, 64, 1024), 17, 0.0, (8,), {}),  # one-row strips at levels 2 and 3
    # planned for a few SMs: several units per CTA (of two images) for the level-1 and level-2 instantiations too, and
    # transposed-walk strips longer than the accumulator ring
    ("plan_sms4_2x64x1024", (2, 64, 1024), 17, 0.0, (8,), {"OPT_PLAN_SMS": 4}),
    ("plan_sms12_2x256x64", (2, 256, 64), 17, 0.0, (8,), {"OPT_PLAN_SMS": 12}),
]
KF_MODE = {0: 0, 2: 1, 1: 2}  # conv mode (0 stride 1, 1 stride 2, 2 nearest-x2) -> conv_kf.cu MODE
EPI = {"EPI_STORE": 0, "EPI_STATS": 1, "EPI_DDIM": 2}
# conv_kf.cu instantiations the denoise step never selects, as (bn, cpg, epi, ch, staged, xk16, mode, res1, apply)
KF_NOT_IN_STEP = {
    (64, 1, 0, 1, True, False, 0, False, False): "codec encoder stem (the image's 3 channels in one 64-channel chunk)",
    (64, 4, 1, 1, True, False, 0, False, False): "codec encoder level-1 conv1, 64 -> 128 channels",
    (64, 1, 0, 2, False, False, 0, False, False): "two-chunk store conv without the x_t shortcut: the step's stem always "
                                                  "has it; kernel-level tests (cdc_test_conv) use this one",
    # the step's stats convs with these shapes all have a 1x1 residual conv, and its fused instantiation exists for the
    # same (bn, ch), so the plan always takes that one (conv_uses_kf); kernel-level tests use the plain ones
    (64, 2, 1, 2, False, False, 0, False, False): "128 -> 64 stats conv without a fused residual conv",
    (32, 4, 1, 3, False, False, 0, False, False): "192 -> 128 stats conv without a fused residual conv",
    (32, 4, 1, 4, False, False, 0, False, False): "256 -> 128 stats conv without a fused residual conv",
}

GEOM_CLASSES = [(0, 0), (1, 0), (0, 1), (0, 2)]  # (tr, MODE): the transposed walk exists for MODE 0 only
GEOM_WANT = ("one_row", "uneven", "ragged", "ring_wrap")

_seen_kf, _seen_tr, _seen_tc, _done = set(), set(), set(), set()
_geo = GeometrySeen()


class _Step(SeqBuffers):
    """One configuration: the decoder with the fixed-point weights, the step descriptions and views of every buffer."""

    def __init__(self, shape, K, eta, opts):
        from cdc_b200 import CDCConfig, Decoder, _ffi
        from oracle.config import CDCConfig as OCfg
        from oracle.weights import synthetic_cond, synthetic_init
        self.ocfg = OCfg()
        net = _fixed_point_unet(self.ocfg)
        sd = dict(net.state_dict())
        self.W = {k: v.double().to(DEV) for k, v in sd.items()}
        self.dec = Decoder(CDCConfig(), sd, device=DEV)
        for name, v in opts.items():
            if name.startswith("OPT_"):
                self.dec.set_plan_option(getattr(_ffi, name), v)
        self.eta, self.seed = eta, 5
        self.dec.set_sample_schedule(K, eta=eta, seed=self.seed)
        B, H, W = shape
        self.B, self.H, self.W_ = B, H, W
        sc = image_scale(B) if B > 1 else 1.0
        self.dec.set_cond([c * sc for c in synthetic_cond(self.ocfg, B, H, W)])
        self.dec._set_x(synthetic_init(B, H, W) * sc)
        self.image_seeds = [7919 * b + 11 for b in range(B)] if opts.get("seeds") else None
        if self.image_seeds:
            self.dec.set_image_seeds(self.image_seeds)
        n = len(self.dec.step_ops())
        self.names = [o[0] for o in self.dec.step_ops()]
        self.desc = [self.dec.step_op_desc(i) for i in range(n)]
        self._bind_views()


def _check_attention(st, d, snap):
    qkv = snap[d.src[0].p].double()  # [B, H, W, 3C]
    B, C = qkv.shape[0], d.out.C
    t = qkv.reshape(B, -1, 3 * C)
    heads = C // 64
    q, kk, v = (t[..., i * C:(i + 1) * C].reshape(B, -1, heads, 64).transpose(1, 2) for i in range(3))
    p = torch.softmax(q @ kk.transpose(-1, -2) / 8.0, dim=-1)
    ref = (p @ v).transpose(1, 2).reshape(B, -1, C)
    pv = (p @ v.abs()).transpose(1, 2).reshape(B, -1, C)
    got = st.views[d.out.p].double().reshape(B, -1, C)
    # probabilities rounded to 16 bits for the P.V product (2^-11 relative each), the softmax normaliser accumulated
    # from unrounded terms (another 2^-11 of sum p |v|), exp2 / fp32 accumulation far below that; 2x headroom; one fp16
    # rounding of the output
    tol = U16 * ref.abs() + 4 * U16 * pv + SUB16
    return {"out": _ratio((got - ref).abs(), tol)}


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_step_ops_match_float64(cfg):
    name, shape, K, eta, ks, opts = cfg
    t0 = time.perf_counter()
    st = _Step(shape, K, eta, opts)
    st.film = st.dec.film_table().double()
    film0 = st.dec.film_table().clone()
    st.dec.saturation_count(reset=True)
    bad, worst_r, worst_s = [], (0.0, ""), (0.0, "")
    for k in ks:
        snap = {p: v.clone() for p, v in st.views.items()}
        for i, d in enumerate(st.desc):
            op = st.names[i]
            st.dec.run_step_op(i, k)
            torch.cuda.synchronize()
            st.check_writes(op, d, snap)
            if d.kind == 0:
                worst = {}
            elif d.kind == 1:
                worst = _check_conv(st, d, snap, k)
            elif d.kind == 2:
                worst = _check_gn_stats(st, d, snap)
            elif d.kind == 3:
                worst = _check_gn_apply(st, d, snap, k)
            elif d.kind == 4:
                worst = _check_attention(st, d, snap)
            else:
                pytest.fail(f"{op}: op kind {d.kind} has no float64 reference")
            shown = " ".join(f"{key}={val:.3g}" for key, val in worst.items())
            print(f"[{name} k={k}] {i:3d} {op:28s} {_inst(d):84s} {shown}  [{_geom(d, st.B)}]")
            for key, val in worst.items():
                if key == "err/S":
                    worst_s = max(worst_s, (val, op))
                else:
                    worst_r = max(worst_r, (val, f"{op} {key}"))
                    if not val <= 1.0:
                        bad.append(f"k={k} op {i} {op} ({_inst(d)}): {key} err/tol = {val:.3g}")
            if d.kind == 1:
                (_seen_tc if d.kernel == 1 else _seen_kf).add(_kf_key(d) if d.kernel == 2 else (d.bn, d.cpg, d.epi))
                if d.kernel == 2:
                    _seen_tr.add(d.tr)
            _geo.add(d, st.B)
            st.advance(d, snap)
        assert torch.equal(st.dec.film_table(), film0), "the FiLM table changed"
        assert st.dec.saturation_count() == 0, "an epilogue saturated to the fp16 range"
    print(f"[{name}] worst err/tol {worst_r[0]:.3g} ({worst_r[1]}), worst conv err/S {worst_s[0]:.3g} ({worst_s[1]}), "
          f"{time.perf_counter() - t0:.1f} s")
    assert not bad, f"{name}: " + "; ".join(bad)
    _done.add(name)


def check_geometry_coverage(want, geo):
    """The unit-loop regimes of kf_geometry the checked ops reached: every instantiation of want with several units
    per CTA, the APPLY and DDIM ones with units of two images in one CTA, every (walk, MODE) class of GEOM_CLASSES with
    one-row strips, uneven strips, ragged segments and ring wrap, and the general kernel with more tiles than CTAs.
    (Every one of these is reachable by the denoise step and by the codec sequences.)"""
    single = sorted(k for k in want if "several_units" not in geo.kf.get(k, ()))
    assert not single, f"instantiations never checked with several units per CTA: {single}"
    one_img = sorted(k for k in want if (k[8] or k[2] == 2) and "two_images" not in geo.kf.get(k, ()))
    assert not one_img, f"APPLY / DDIM instantiations never checked with two images' units on one CTA: {one_img}"
    missing = [(c, g) for c in GEOM_CLASSES for g in GEOM_WANT if (c, g) not in geo.cls]
    assert not missing, f"(walk, MODE) geometry never checked: {missing}"
    assert geo.tc_waves, "conv_tc.cu never checked with more tiles than CTAs"


def test_step_op_coverage():
    """Every conv_kf.cu instantiation the step plan can select was checked above at least once, with both walks, and in
    the unit-loop regimes check_geometry_coverage lists."""
    missing_cfg = [c[0] for c in CONFIGS if c[0] not in _done]
    assert not missing_cfg, f"configurations not run (or failed): {missing_cfg}"
    print("conv_tc.cu instantiations checked:", sorted(_seen_tc))
    want = _kf_cases() - set(KF_NOT_IN_STEP)
    assert not (set(KF_NOT_IN_STEP) - _kf_cases()), "stale exclusion"
    assert want <= _seen_kf, f"conv_kf.cu instantiations never checked: {sorted(want - _seen_kf)}"
    assert _seen_tr == {0, 1}, f"walks checked: {_seen_tr}"
    print("conv_tc.cu instantiations checked with more tiles than CTAs:", sorted(_geo.tc_waves))
    check_geometry_coverage(want, _geo)
