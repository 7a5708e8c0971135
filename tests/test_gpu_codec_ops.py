"""Teacher-forced per-op parity of the context net, the analysis encoder, the hyper-encoder and the hyper-decoder on a
real B200.

Each configuration calls the sequence's public entry once (cdc_set_latent, cdc_encode_analysis, cdc_hyper_encode,
cdc_hyper_decode) with a driven input and checks its boundary conversions bitwise: the sequence's input tensor is fp16 of
the caller's input, y / z / mu are fp32 of the last op's output, sigma = max(sigma_raw, 0.11f).  Then every op of the
sequence runs alone (cdc_run_seq_op) on the buffers the ops before it wrote, and its outputs are compared with a float64
reference of that one operation (tests/op_reference.py, as tests/test_gpu_step_ops.py does for the denoise step), so a
failure names one kernel instance; nothing an op does not declare as its output may change.  The op-by-op replay must end
with the same bits in every buffer as the entry left: the entry runs exactly these ops in this order.

The sequences decide the bitstream (y, z, and from z_hat the mu / sigma of every y symbol, on both sides of the stream),
and they run code the denoise step never takes: the 5x5 stride-2 convs, the 5x5 transposed convs, the LeakyReLU epilogue,
the 256 -> 512 output conv, the encoder's strip-kernel instantiations, and the input GroupNorm without FiLM.

With B > 1, image b's input is scaled by 2^((b mod 4) - 1) (per-image GroupNorm statistics), and the coverage test
requires the strip kernel's unit-loop regimes of tests/test_gpu_step_ops.py check_geometry_coverage here too.
"""
import time

import pytest
import torch

from tests.op_reference import (DEV, GeometrySeen, SeqBuffers, _bits, _check_conv, _check_gn_apply, _check_gn_stats,
                                _fixed_point_unet, _geom, _inst, _kf_key, _nhwc, _view, fixed_point_, image_scale)
from tests.test_gpu_step_ops import KF_NOT_IN_STEP, check_geometry_coverage

pytestmark = pytest.mark.gpu

CONTEXT, ENCODER, HYPER_ENC, HYPER_DEC = 1, 2, 3, 4  # include/cdc_b200_tools.h cdc_seq
SIGMA_MIN = torch.tensor(0.11, dtype=torch.float32)  # the hyper-decoder's sigma clamp, as the fp32 the kernel compares
# convs followed by LeakyReLU(0.2) in oracle/codec.py (every other conv has no activation in its epilogue)
LEAKY = {"codec.hyper_enc.c1", "codec.hyper_enc.c2", "codec.hyper_dec.t1", "codec.hyper_dec.t2"}

# (name, sequence, (B, H, W), plan options)
CONFIGS = [
    ("context_768x512", CONTEXT, (1, 512, 768), {}),
    ("context_two_images_128x192", CONTEXT, (2, 128, 192), {}),
    ("context_three_images_64x128", CONTEXT, (3, 64, 128), {}),
    ("context_tall_64x1024", CONTEXT, (1, 1024, 64), {}),  # the strip kernel's transposed walk
    ("context_general_kernel_768x512", CONTEXT, (1, 512, 768), {"OPT_KF": 0}),
    ("context_2048x2048", CONTEXT, (1, 2048, 2048), {}),
    ("context_16x256x256", CONTEXT, (16, 256, 256), {}),
    ("context_one_row_64x1024", CONTEXT, (1, 64, 1024), {}),
    # planned for a few SMs: several units per CTA, of two images, for every strip instantiation
    ("context_plan_sms4_2x64x1024", CONTEXT, (2, 64, 1024), {"OPT_PLAN_SMS": 4}),
    ("context_plan_sms4_2x384x128", CONTEXT, (2, 384, 128), {"OPT_PLAN_SMS": 4}),  # the transposed walk
    ("encoder_64x64", ENCODER, (1, 64, 64), {}),
    ("encoder_three_images_64x128", ENCODER, (3, 64, 128), {}),
    ("encoder_two_images_192x256", ENCODER, (2, 192, 256), {}),
    ("encoder_tall_64x1024", ENCODER, (1, 1024, 64), {}),
    ("encoder_768x512", ENCODER, (1, 512, 768), {}),
    ("encoder_2048x2048", ENCODER, (1, 2048, 2048), {}),
    ("encoder_plan_sms4_2x64x1024", ENCODER, (2, 64, 1024), {"OPT_PLAN_SMS": 4}),  # the encoder's own instantiations
    ("hyper_enc_64x64", HYPER_ENC, (1, 64, 64), {}),  # z is 1 x 1: every tap reads padding or sits at an edge
    ("hyper_enc_two_images_192x256", HYPER_ENC, (2, 192, 256), {}),
    ("hyper_enc_1024x64", HYPER_ENC, (1, 64, 1024), {}),  # z 1 x 16
    ("hyper_enc_2048x2048", HYPER_ENC, (1, 2048, 2048), {}),  # y 128 x 128, z 32 x 32
    ("hyper_dec_64x64", HYPER_DEC, (1, 64, 64), {}),
    ("hyper_dec_two_images_192x256", HYPER_DEC, (2, 192, 256), {}),
    ("hyper_dec_1024x64", HYPER_DEC, (1, 64, 1024), {}),
    ("hyper_dec_2048x2048", HYPER_DEC, (1, 2048, 2048), {}),
]

_cache = {}
_seen, _done = set(), set()
_geo = GeometrySeen()


def _setup():
    """One decoder for every configuration: fixed-point UNet, context-net and codec weights (tests/op_reference.py
    fixed_point_), and a Codec over it."""
    if "s" in _cache:
        return _cache["s"]
    from cdc_b200 import CDCConfig, Codec, Decoder
    from oracle.config import CDCConfig as OCfg
    from oracle.weights import build_codec
    ocfg = OCfg()
    w = dict(_fixed_point_unet(ocfg).state_dict())
    oc = fixed_point_(build_codec(ocfg, seed=1))
    for k, v in oc.state_dict().items():
        w[k if k.startswith("context.") else "codec." + k] = v
    dec = Decoder(CDCConfig(), w, device=DEV)
    codec = Codec(dec, median=oc.prior.median)
    W = {k: v.double().to(DEV) for k, v in w.items() if k.startswith(("context.", "codec."))}
    _cache["s"] = (ocfg, dec, codec, W)
    return _cache["s"]


class _Seq(SeqBuffers):
    """One sequence of the bound plan: its op descriptions and views of every buffer they name."""

    def __init__(self, ocfg, dec, W, seq, shape):
        self.ocfg, self.dec, self.W, self.seq = ocfg, dec, W, seq
        self.B, self.H, self.W_ = shape
        self.film = None  # (no op of these sequences has FiLM)
        self.names = [o[0] for o in dec.step_ops(seq)]
        self.desc = [dec.step_op_desc(i, seq) for i in range(len(self.names))]
        self._bind_views()

    def first(self):
        """The first op that is not the GroupNorm-slot memset: its source is the sequence's input tensor."""
        return next(d for d in self.desc if d.kind != 0)


def _driven_input(seq, B, H, W):
    """The caller's input of the sequence's public entry (NCHW fp32, host); image b scaled by image_scale when B > 1."""
    from oracle.weights import synthetic_image, synthetic_latent
    g = torch.Generator().manual_seed(17)
    if seq == CONTEXT:
        x = synthetic_latent(B, H, W)
    elif seq == ENCODER:
        x = synthetic_image(B, H, W, index=3)
    elif seq == HYPER_ENC:  # y of realistic magnitude, bf16-exact
        x = (8.0 * torch.randn(B, 256, H // 16, W // 16, generator=g)).bfloat16().float()
    else:
        x = torch.round(4.0 * torch.randn(B, 256, H // 64, W // 64, generator=g))  # z_hat
    return x * image_scale(B) if B > 1 else x


def _entry(dec, codec, seq, x):
    """Runs the sequence's public entry on x; returns its fp32 outputs (none for the context net: its outputs are the
    bound cond maps)."""
    if seq == CONTEXT:
        dec.set_latent(x)
        return ()
    if seq == ENCODER:
        return (codec.analysis(x),)
    if seq == HYPER_ENC:
        return (codec.hyper_encode(x),)
    return codec.hyper_decode(x)


def _input_stored(seq, x):
    """What the entry's boundary conversion must store for input x: NHWC fp16, NaN kept, beyond the fp16 range (and
    +-inf) saturated to +-65504; the encoder's image as 2 * img - 1 in channels 0-2 of 64."""
    v = 2.0 * x - 1.0 if seq == ENCODER else x
    h = _nhwc(v.clamp(-65504.0, 65504.0).to(DEV)).half()
    if seq == ENCODER:
        h = torch.cat([h, h.new_zeros(*h.shape[:3], 61)], dim=3)
    return h


def _same_bits(a, b):
    """Bitwise equality, any NaN matching any NaN."""
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(_bits(a)[~na], _bits(b)[~nb])


def _check_boundaries(st, x, outs):
    seq = st.seq
    d0 = st.first()
    got_in = st.views[d0.src[0].p]
    conv_in = "img_in_kernel" if seq == ENCODER else "nchw_to_nhwc_kernel"
    assert _same_bits(got_in, _input_stored(seq, x)), \
        f"{conv_in} (the input of {st.names[st.desc.index(d0)]}): not fp16 of the caller's input"
    last = st.views[st.desc[-1].out.p]
    if seq in (ENCODER, HYPER_ENC):
        assert torch.equal(_bits(outs[0]), _bits(last.permute(0, 3, 1, 2).float())), f"nhwc_to_nchw_kernel: y / z != fp32 of {st.names[-1]}'s output"
    elif seq == HYPER_DEC:
        mu, sigma = outs
        raw = last.permute(0, 3, 1, 2).float()
        assert torch.equal(_bits(mu), _bits(raw[:, :256])), "nhwc_slice_to_nchw_kernel: mu != channels 0-255 of hdec.c3"
        assert torch.equal(_bits(sigma), _bits(torch.maximum(raw[:, 256:], SIGMA_MIN.to(DEV)))), \
            "nhwc_slice_to_nchw_kernel: sigma != max(channels 256-511 of hdec.c3, 0.11f)"
    else:  # the context maps through cdc_get_cond
        cond = st.dec.get_cond()
        for i in range(4):
            d = next(d for n, d in zip(st.names, st.desc) if n.startswith(f"context.rbs.{i}.gn2"))
            assert torch.equal(_bits(cond[i]), _bits(st.views[d.out.p].permute(0, 3, 1, 2).float())), f"c{i}"


def _features(d):
    """What the coverage test wants checked at least once."""
    f = set()
    if d.kind == 1 and d.kernel == 2:
        f.add(("kf", _kf_key(d)))
        if d.apply and d.film_off == -1:
            f.add("kf apply without FiLM")
    if d.kind == 1 and d.kernel == 1:
        f.add(("tc", d.mode, d.ksize))
        if d.act_slope != 0.0:
            f.add(("slope", round(float(d.act_slope), 6)))
    if d.kind == 3 and d.film_off == -1:
        f.add("gn_apply without FiLM")
    return f


@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_codec_ops_match_float64(cfg):
    from cdc_b200 import _ffi
    name, seq, shape, opts = cfg
    t0 = time.perf_counter()
    ocfg, dec, codec, W = _setup()
    dec.set_plan_option(_ffi.OPT_KF, opts.get("OPT_KF", 1))
    dec.set_plan_option(_ffi.OPT_PLAN_SMS, opts.get("OPT_PLAN_SMS", 0))
    B, H, Wd = shape
    x = _driven_input(seq, B, H, Wd)
    dec.bind(B, H, Wd)
    dec.saturation_count(reset=True)
    outs = _entry(dec, codec, seq, x)
    torch.cuda.synchronize()
    st = _Seq(ocfg, dec, W, seq, shape)
    assert st.desc, f"{name}: the sequence has no ops"
    _check_boundaries(st, x, outs)

    entry = {p: v.clone() for p, v in st.views.items()}
    snap = {p: v.clone() for p, v in st.views.items()}
    bad, worst_r, worst_s = [], (0.0, ""), (0.0, "")
    for i, d in enumerate(st.desc):
        op = st.names[i]
        dec.run_step_op(i, 0, seq)
        torch.cuda.synchronize()
        st.check_writes(op, d, snap)
        if d.kind == 0:
            worst = {}
        elif d.kind == 1:
            slope = 0.2 if d.weight.decode() in LEAKY else 0.0
            assert abs(d.act_slope - slope) < 1e-7, f"{op}: LeakyReLU slope {d.act_slope}, the oracle's is {slope}"
            worst = _check_conv(st, d, snap, 0)
        elif d.kind == 2:
            worst = _check_gn_stats(st, d, snap)
        elif d.kind == 3:
            worst = _check_gn_apply(st, d, snap, 0)
        else:
            pytest.fail(f"{op}: op kind {d.kind} has no float64 reference here")
        shown = " ".join(f"{key}={val:.3g}" for key, val in worst.items())
        print(f"[{name}] {i:3d} {op:32s} {_inst(d):84s} {shown}  [{_geom(d, B)}]")
        for key, val in worst.items():
            if key == "err/S":
                worst_s = max(worst_s, (val, op))
            else:
                worst_r = max(worst_r, (val, f"{op} {key}"))
                if not val <= 1.0:
                    bad.append(f"op {i} {op} ({_inst(d)}): {key} err/tol = {val:.3g}")
        _seen.update(_features(d))
        _geo.add(d, B)
        st.advance(d, snap)
    for p, v in st.views.items():
        assert _same_bits(v, entry[p]), f"{name}: the op-by-op replay left other bits than the public entry"
    assert dec.saturation_count() == 0, "an epilogue saturated to the fp16 range"
    if seq == ENCODER:  # the decoder side re-derives (y_hat, mu, sigma) from the symbols alone, bit for bit
        enc = codec.encode(x)
        y_hat, mu, sigma = codec.latent_from_symbols(enc["qz"].cpu(), enc["q"].cpu())
        for k_, got in (("y_hat", y_hat), ("mu", mu), ("sigma", sigma)):
            assert torch.equal(_bits(got), _bits(enc[k_])), f"{name}: latent_from_symbols re-derives another {k_}"
    print(f"[{name}] worst err/tol {worst_r[0]:.3g} ({worst_r[1]}), worst conv err/S {worst_s[0]:.3g} ({worst_s[1]}), "
          f"{time.perf_counter() - t0:.1f} s")
    assert not bad, f"{name}: " + "; ".join(bad)
    _done.add(name)


def test_boundary_conversions_keep_nan():
    """Every NCHW fp32 -> NHWC fp16 conversion at the library's boundary (set_cond, set_x, set_latent, the encoder's
    image, hyper_encode, hyper_decode) stores NaN as NaN and saturates +-inf and finite values beyond the fp16 range to
    +-65504."""
    from oracle.weights import synthetic_cond, synthetic_init
    ocfg, dec, codec, W = _setup()
    B, H, Wd = 2, 64, 128
    special = torch.tensor([float("nan"), float("inf"), -float("inf"), 7e4, -7e4, 65519.0, 1.0])

    def poke(t, vals):
        t = t.clone()
        t.view(-1)[:vals.numel()] = vals
        t.view(-1)[-vals.numel():] = vals
        return t

    c = [poke(t, special) for t in synthetic_cond(ocfg, B, H, Wd)]
    dec.set_cond(c)
    got = dec.get_cond()
    for i in range(4):
        assert _same_bits(got[i], c[i].clamp(-65504.0, 65504.0).half().float().to(DEV)), f"set_cond c{i}"
    x = poke(synthetic_init(B, H, Wd), special)
    dec._set_x(x)
    assert dec.step_ops()[1][0] == "stem"
    xpad = dec.step_op_desc(1).src[0]  # the stem's first source: the 16-channel x_t copy
    xp = _view(xpad.p, (B, H, Wd, 16), torch.float16)
    assert _same_bits(xp[..., :3], _nhwc(x.clamp(-65504.0, 65504.0).to(DEV)).half()), "set_x"
    for seq in (CONTEXT, ENCODER, HYPER_ENC, HYPER_DEC):
        v = _driven_input(seq, B, H, Wd)
        if seq == ENCODER:  # 2 * img - 1 hits the special values
            v = poke(v, (special + 1.0) / 2.0)
        else:
            v = poke(v, special)
        _entry(dec, codec, seq, v)
        torch.cuda.synchronize()
        st = _Seq(ocfg, dec, W, seq, (B, H, Wd))
        assert _same_bits(st.views[st.first().src[0].p], _input_stored(seq, v)), f"sequence {seq}: input conversion"


def test_codec_op_coverage():
    """The configurations above checked every kernel path the codec sequences add to those of the denoise step."""
    missing_cfg = [c[0] for c in CONFIGS if c[0] not in _done]
    assert not missing_cfg, f"configurations not run (or failed): {missing_cfg}"
    want = {("kf", k) for k, why in KF_NOT_IN_STEP.items() if why.startswith("codec encoder")}
    assert len(want) == 2, "KF_NOT_IN_STEP names the encoder's two strip instantiations"
    want |= {"kf apply without FiLM", "gn_apply without FiLM", ("tc", 1, 5), ("tc", 3, 5), ("slope", 0.2)}
    assert want <= _seen, f"never checked: {sorted(map(str, want - _seen))}"
    # every strip instantiation the codec sequences ran, in the unit-loop regimes the step's coverage test requires
    check_geometry_coverage(set(_geo.kf), _geo)
