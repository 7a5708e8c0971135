"""Teacher-forced per-op parity of one denoise step on a real B200.

Every op of the bound step plan runs alone (cdc_run_step_op) on the GPU's own outputs of the ops before it; its outputs
are compared with a float64 reference of that one operation, computed on the GPU from a snapshot of exactly what the
kernel read.  A failure therefore names one kernel instance.  The op descriptions (cdc_step_op_describe) say which
tensors an op reads and writes and which kernel instantiation runs it; everything an op does not declare as its output
must stay bitwise unchanged.

Conv weights are rounded to a fixed-point grid (multiples of 2^-m, every sum of four weights below 2^11 grid steps), so
the fp16 repack and the pre-summed nearest-x2 parity weights are exact and the only conv error left is the fp32
accumulation order: the tolerances below are derived from that, op by op.
"""
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# fp32 accumulation in the tensor cores: |conv - ref| <= C_ACC * S, S = conv(|x|, |w|) + |b| (+ |residual|).
# Measured on a B200 (1000 W power limit) over every conv of every configuration below: worst err/S 3.3e-7 (the final
# conv, whose fp32 output is not rounded to 16 bits), 1.5e-7 for the others.  C_ACC = 2^-19 (1.9e-6) is 5.8x that.
# (A dropped tap or a wrong bias is an error of order S: hundreds of thousands of C_ACC.)
C_ACC = 2.0 ** -19
U16 = 2.0 ** -11          # unit roundoff of fp16: one rounding to nearest of the stored value
SUB16 = 2.0 ** -25        # half the spacing of fp16 subnormals: the rounding error floor near zero
U32 = 2.0 ** -24
TANH_APPROX = 2.0 ** -10.98  # max relative error of tanh.approx.f32 (PTX ISA), used by the GroupNorm + SiLU transform

# (name, (B, H, W), steps K, eta, steps k checked, plan options)
CONFIGS = [
    ("headline_768x512", (1, 512, 768), 17, 0.0, (0, 16), {}),
    ("two_images_128x192", (2, 128, 192), 17, 0.0, (8,), {}),
    ("three_images_64x128", (3, 64, 128), 17, 0.0, (8,), {}),
    ("tall_64x1024", (1, 1024, 64), 17, 0.0, (8,), {}),
    ("ragged_704x256", (1, 256, 704), 17, 0.0, (8,), {}),
    ("general_kernel_768x512", (1, 512, 768), 17, 0.0, (16,), {"OPT_KF": 0}),
    ("ddim_noise_128x192", (2, 128, 192), 17, 1.0, (3,), {}),
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

_seen_kf, _seen_tr, _seen_tc, _done = set(), set(), set(), set()


def _kf_cases():
    """The KF_ALL_CASES() list of csrc/conv_kf.cu as coverage keys (bn, cpg, epi, ch, staged, xk16, mode, res1, apply)."""
    src = open(os.path.join(ROOT, "conditional-diffusion-model-for-compression_b200", "csrc", "conv_kf.cu")).read()
    body = src[src.index("#define KF_ALL_CASES()"):]
    body = body[:body.index("\n\n")]
    cases = set()
    for m in re.finditer(r"KF_CASE\((\d+), (\d+), (EPI_\w+), (\d+), (\w+), (\w+), (\d), (\w+), (\w+)\)", body):
        bn, cpg, epi, ch, st, xk, mode, res, app = m.groups()
        e = EPI[epi]
        cases.add((int(bn), int(cpg) if e == 1 else 1, e, int(ch), st == "true", xk == "true", int(mode), res == "true",
                   app == "true"))
    return cases


def _kf_key(d):
    return (d.bn, d.cpg if d.epi == 1 else 1, d.epi, d.ch, bool(d.staged), bool(d.xk16), KF_MODE[d.mode], bool(d.res1),
            bool(d.apply))


def _inst(d):
    if d.kind != 1:
        return "-"
    if d.kernel == 1:
        return f"conv_tc bn{d.bn} cpg{d.cpg} epi{d.epi}"
    return (f"conv_kf bn{d.bn} cpg{d.cpg} epi{d.epi} ch{d.ch} staged{d.staged} xk16{d.xk16} mode{KF_MODE[d.mode]} "
            f"res1{d.res1} apply{d.apply} tr{d.tr}")


def _fixed_point_unet(ocfg):
    """Oracle UNet (seed 0) with every conv weight on a per-layer grid 2^-m, m the largest with 4 * max|w| * 2^m < 2^11."""
    from oracle.weights import build_unet
    net = build_unet(ocfg, seed=0)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.endswith(".weight") and p.dim() == 4:
                m = math.floor(math.log2(2.0 ** 11 / (4.0 * p.abs().max().item())))
                if 4.0 * p.abs().max().item() * 2.0 ** m >= 2.0 ** 11:
                    m -= 1
                p.copy_(torch.round(p * 2.0 ** m) / 2.0 ** m)
    return net


class _DevPtr:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 3,
                                         "strides": None}


def _view(ptr, shape, dtype):
    """The library's device buffer at ptr as a torch tensor (no copy)."""
    ts = {torch.float16: "<f2", torch.float32: "<f4", torch.int64: "<i8"}[dtype]
    return torch.as_tensor(_DevPtr(ptr, shape, ts), device=DEV)


def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def _nchw(t, C=None):
    """NHWC fp16 [B, H, W, Cphys] -> NCHW float64 with C logical channels (zeros beyond Cphys)."""
    x = t.permute(0, 3, 1, 2).double()
    if C is not None and C > x.shape[1]:
        x = torch.cat([x, x.new_zeros(x.shape[0], C - x.shape[1], x.shape[2], x.shape[3])], dim=1)
    return x


def _nhwc(x):
    return x.permute(0, 2, 3, 1)


def _conv(x, w, mode, ks):
    if mode == 2:
        x = F.interpolate(x, scale_factor=2, mode="nearest")
    return F.conv2d(x, w, stride=2 if mode == 1 else 1, padding=ks // 2)


def _slot_sums(slot):
    """[B, 32, 4] int64 fixed-point accumulators (csrc/gn_sums.cuh) -> (sum, sum of squares) float64 [B, 32]."""
    s = slot.double()
    return s[..., 0] * 2.0 ** -20, s[..., 1] * 2.0 ** -20 + s[..., 2] * 1024.0


def _gn_transform(x, slot, gamma, beta, film, eps, silu):
    """float64 GroupNorm (+FiLM) (+SiLU) of NCHW x with mean / variance from the accumulator slot (oracle/unet.py RB:
    SiLU((GN(x) * gamma + beta) * (1 + s) + sh)).  Returns (y, pre-activation z, zmag): zmag is the sum of the magnitudes
    of the terms z is made of, |a x| + |a mean| + |beta (1 + s)| + |sh| with a = rstd gamma (1 + s)."""
    B, C, H, W = x.shape
    s, q = _slot_sums(slot)
    n = (C // 32) * H * W
    mu = s / n
    rstd = 1.0 / torch.sqrt(q / n - mu * mu + eps)
    mu_c = mu.repeat_interleave(C // 32, dim=1)[:, :, None, None]
    rstd_c = rstd.repeat_interleave(C // 32, dim=1)[:, :, None, None]
    sc = film[0] + 1.0 if film is not None else torch.ones_like(gamma)
    sh = film[1] if film is not None else torch.zeros_like(gamma)
    a = rstd_c * (gamma * sc)[None, :, None, None]
    z = (x - mu_c) * rstd_c * gamma[None, :, None, None] + beta[None, :, None, None]
    z = z * sc[None, :, None, None] + sh[None, :, None, None]
    zmag = (a * x).abs() + (a * mu_c).abs() + (beta * sc).abs()[None, :, None, None] + sh.abs()[None, :, None, None]
    return (z * torch.sigmoid(z) if silu else z), z, zmag


def _group_sums(y):
    B, C = y.shape[:2]
    g = y.reshape(B, 32, -1)
    return g.sum(-1), (g * g).sum(-1)


class _Step:
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
            self.dec.set_plan_option(getattr(_ffi, name), v)
        self.eta, self.seed = eta, 5
        self.dec.set_sample_schedule(K, eta=eta, seed=self.seed)
        B, H, W = shape
        self.B, self.H, self.W_ = B, H, W
        self.dec.set_cond(synthetic_cond(self.ocfg, B, H, W))
        self.dec._set_x(synthetic_init(B, H, W))
        n = len(self.dec.step_ops())
        self.names = [o[0] for o in self.dec.step_ops()]
        self.desc = [self.dec.step_op_desc(i) for i in range(n)]
        self.views = {}
        for d in self.desc:
            for t in (d.src[0], d.src[1], d.residual, d.out, d.res_out):
                if t.p:
                    self.views.setdefault(t.p, _view(t.p, (B, t.H, t.W, t.Cphys), torch.float16))
            if d.kind == 0:
                self.slots_base, self.nslots = d.gn_out_acc, d.gn_slots
                self.views[d.gn_out_acc] = _view(d.gn_out_acc, (d.gn_slots, B, 32, 4), torch.int64)
            if d.x:
                self.x_p, self.x0_p = d.x, d.x0_out
                self.views[d.x] = _view(d.x, (B, H, W, 3), torch.float32)
                self.views[d.x0_out] = _view(d.x0_out, (B, H, W, 3), torch.float32)
                self.views.setdefault(d.xpad, _view(d.xpad, (B, H, W, 16), torch.float16))
                self.xpad_p = d.xpad

    def slot_of(self, snap, p):
        return snap[self.slots_base][self.slot_index(p)]

    def slot_index(self, p):
        return (p - self.slots_base) // (self.B * 32 * 4 * 8)

    def outputs(self, d):
        """(buffers the op may write, GroupNorm slot it accumulates into or None)."""
        if d.kind == 0:
            return {d.gn_out_acc}, None
        outs = {t.p for t in (d.out, d.res_out) if t.p}
        if d.kind == 1 and d.epi == 2:
            outs |= {d.x, d.x0_out, d.xpad}
        slot = self.slot_index(d.gn_out_acc) if d.gn_out_acc else None
        return outs, slot


def _ratio(err, tol):
    return (err / tol).max().item()


def _check_conv(st, d, snap, k):
    """conv (+fused residual conv, +fused input GroupNorm, +statistics, +sampler update) against float64."""
    w = st.W[d.weight.decode() + ".weight"]
    b = st.W[d.weight.decode() + ".bias"]
    srcs = [_nchw(snap[t.p], t.C) for t in (d.src[0], d.src[1]) if t.p]
    x = torch.cat(srcs, dim=1)
    if w.shape[1] != x.shape[1]:  # the stem: x_t (3 of the first source's 64 channels), then the context channels
        n0 = w.shape[1] - srcs[1].shape[1]
        wf = w.new_zeros(w.shape[0], x.shape[1], *w.shape[2:])
        wf[:, :n0] = w[:, :n0]
        wf[:, srcs[0].shape[1]:] = w[:, n0:]
        w = wf
    stat = None
    if d.apply:  # conv2 + GroupNorm 1 (+FiLM) + SiLU of its input, applied by the kernel to the input rows
        gnp = d.in_gn.decode()
        C = x.shape[1]
        film = None
        if d.film_off >= 0:
            f = st.film[k]
            film = (f[d.film_off:d.film_off + C], f[d.film_off + C:d.film_off + 2 * C])
        a = _gn_transform(x, st.slot_of(snap, d.gn_in_acc), st.W[gnp + ".weight"], st.W[gnp + ".bias"], film,
                          st.ocfg.gn_eps, True)[0]
        x = a.half().double()  # the operand the kernel stores in shared memory: fp16 of the transformed value
        # the kernel's operand may differ by one fp16 ulp (<= 2^-10 |a|) where tanh.approx rounds the other way; those
        # differences are independent from tap to tap: 6 standard deviations of their sum
        stat = 6.0 * 2.0 ** -10 * torch.sqrt(_conv(x * x, w * w, d.mode, d.ksize))
    ref = _conv(x, w, d.mode, d.ksize) + b[None, :, None, None]
    S = _conv(x.abs(), w.abs(), d.mode, d.ksize) + b.abs()[None, :, None, None]
    if d.residual.p:
        r = _nchw(snap[d.residual.p])
        ref, S = ref + r, S + r.abs()
    acc = C_ACC * S + (stat if stat is not None else 0.0)
    worst = {}
    if d.epi == 2:  # final conv + sampler update: fp32 epilogue, no 16-bit rounding of the network output
        c0, c1, e0, e1, sg = st.dec.coeffs5(k)
        xt = snap[d.x].double()  # NHWC [B, H, W, 3]
        out = _nhwc(ref)[..., :3]
        x0 = e0 * xt + e1 * out
        tol_x0 = C_ACC * _nhwc(S)[..., :3] + U32 * x0.abs() + 1e-30
        got_x0 = st.views[d.x0_out].double()
        worst["x0"] = _ratio((got_x0 - x0).abs(), tol_x0)
        xp = c0 * x0.clamp(-1.0, 1.0) + c1 * xt
        tol = abs(c0) * tol_x0 + 2 * U32 * (abs(c0) * x0.abs().clamp(max=1.0) + abs(c1) * xt.abs()) + 1e-30
        if sg != 0.0:
            from oracle.sampler import philox_normal
            z = _nhwc(philox_normal(st.seed, k, st.B, st.H, st.W_).double().to(DEV))
            xp = xp + sg * z
            tol = tol + sg * 2.0 ** -18 * (z.abs() + 1.0)  # fp32 logf / sqrtf / sincospif of the Box-Muller pair
        got_x = st.views[d.x].double()
        worst["x_prev"] = _ratio((got_x - xp).abs(), tol)
        xpad = st.views[d.xpad]
        assert torch.equal(xpad[..., :3], st.views[d.x].half()), "xpad channels 0-2 != fp16(x_prev)"
        assert not xpad[..., 3:].any(), "xpad channels 3-15 not zero"
        worst["err/S"] = (((got_x0 - x0).abs() - U32 * x0.abs()).clamp(min=0) / _nhwc(S)[..., :3]).max().item()
        return worst
    got = _nchw(st.views[d.out.p])[:, :ref.shape[1]]
    tol = U16 * ref.abs() + (1.0 + U16) * acc + SUB16
    worst["out"] = _ratio((got - ref).abs(), tol)
    if not d.apply:  # (measured accumulation error, the basis of C_ACC)
        worst["err/S"] = (((got - ref).abs() - U16 * ref.abs() - SUB16).clamp(min=0) / S).max().item()
    if d.res1:  # the ResBlock's 1x1 residual conv computed in the same launch from the same (raw) input
        rw = st.W[d.res_weight.decode() + ".weight"]
        rb = st.W[d.res_weight.decode() + ".bias"]
        rref = _conv(x, rw, 0, 1) + rb[None, :, None, None]
        rS = _conv(x.abs(), rw.abs(), 0, 1) + rb.abs()[None, :, None, None]
        rgot = _nchw(st.views[d.res_out.p])
        worst["res_out"] = _ratio((rgot - rref).abs(), U16 * rref.abs() + (1.0 + U16) * C_ACC * rS + SUB16)
    if d.epi == 1:  # GroupNorm statistics of the output, fixed point
        s_got, q_got = _slot_sums(st.views[st.slots_base][st.slot_index(d.gn_out_acc)])
        s_ref, q_ref = _group_sums(ref)
        # per value: |v - ref| <= e = 2^-11 |ref| + C_ACC S (whether the epilogue sums the fp32 or the stored value);
        # fp32 sums over at most n sequential terms per thread and partial (a strip column: H or W rows x cpg channels,
        # then a 64-way reduction); every partial loses <= 2^-21 to the 2^-20 fixed-point step (one partial per 64 pixels
        # at most)
        e = U16 * ref.abs() + (1.0 + U16) * acc
        es, eq = _group_sums(e)[0], _group_sums(e * (2.0 * ref.abs() + e))[0]
        nseq = max(st.H, st.W_) * d.cpg + 64
        npart = ref.shape[2] * ref.shape[3] / 64.0 + 1.0
        abs_s, abs_q = _group_sums(ref.abs())[0], q_ref
        tol_s = es + nseq * U32 * abs_s + npart * 2.0 ** -21
        tol_q = eq + nseq * U32 * abs_q + npart * 2.0 ** -21
        worst["gn_sum"] = _ratio((s_got - s_ref).abs(), tol_s)
        worst["gn_sq"] = _ratio((q_got - q_ref).abs(), tol_q)
    return worst


def _check_gn_apply(st, d, snap, k):
    gnp = d.weight.decode()
    x = _nchw(snap[d.src[0].p])
    C = x.shape[1]
    film = None
    if d.film_off >= 0:
        f = st.film[k]
        film = (f[d.film_off:d.film_off + C], f[d.film_off + C:d.film_off + 2 * C])
    y, z, zmag = _gn_transform(x, st.slot_of(snap, d.gn_in_acc), st.W[gnp + ".weight"], st.W[gnp + ".bias"], film,
                               st.ocfg.gn_eps, bool(d.silu))
    res = _nchw(snap[d.residual.p]) if d.residual.p else None
    ref = y + res if res is not None else y
    got = _nchw(st.views[d.out.p])
    # z in fp32: the mean and rstd (< 1 ulp each), the folded coefficients a = gamma rstd (1 + s) and
    # b = (beta - mean a') (1 + s) + sh (two roundings each) and the FMA: <= 6 roundings of the terms of z, and SiLU's
    # slope is below 1.1 -> 8 U32 zmag.  SiLU(2h) = h + h tanh.approx(h), h = z / 2: |error| <= |h tanh(h)| 2^-10.98.
    # The residual add in fp32, one fp16 rounding of the stored value.
    tol = U16 * ref.abs() + SUB16 + 8 * U32 * zmag
    if d.silu:
        tol = tol + TANH_APPROX * (0.5 * z * torch.tanh(0.5 * z)).abs()
    if res is not None:
        tol = tol + U32 * (ref.abs() + res.abs())
    return {"out": _ratio((got - ref).abs(), tol)}


def _check_gn_stats(st, d, snap):
    x = _nchw(snap[d.src[0].p])
    s_ref, q_ref = _group_sums(x)
    s_got, q_got = _slot_sums(st.views[st.slots_base][st.slot_index(d.gn_out_acc)])
    # exact fp16 inputs summed in fp32: at most 64 pixels + 8 rows + cpg channels in sequence per partial; one partial
    # per 64 pixels, each losing <= 2^-21 to the fixed-point step
    n = 64 + 8 + x.shape[1] // 32
    npart = x.shape[2] * x.shape[3] / 64.0 + 1.0
    ts = n * U32 * _group_sums(x.abs())[0] + npart * 2.0 ** -21
    tq = n * U32 * q_ref + npart * 2.0 ** -21
    return {"gn_sum": _ratio((s_got - s_ref).abs(), ts), "gn_sq": _ratio((q_got - q_ref).abs(), tq)}


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
    st = _Step(shape, K, eta, opts)
    st.film = st.dec.film_table().double()
    film0 = st.dec.film_table().clone()
    st.dec.saturation_count(reset=True)
    bad = []
    for k in ks:
        snap = {p: v.clone() for p, v in st.views.items()}
        for i, d in enumerate(st.desc):
            op = st.names[i]
            outs, slot = st.outputs(d)
            st.dec.run_step_op(i, k)
            torch.cuda.synchronize()
            # writes only its own outputs
            for p, v in st.views.items():
                if p in outs:
                    continue
                if p == st.slots_base and slot is not None:
                    keep = [j for j in range(st.nslots) if j != slot]
                    assert torch.equal(v[keep], snap[p][keep]), f"{op}: wrote a GroupNorm slot it does not own"
                else:  # (bit patterns: a buffer no op has written yet may hold NaNs)
                    assert torch.equal(_bits(v), _bits(snap[p])), f"{op}: wrote a buffer it does not declare as output"
            if d.kind == 0:
                assert not st.views[st.slots_base].any(), f"{op}: GroupNorm slots not cleared"
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
            print(f"[{name} k={k}] {i:3d} {op:28s} {_inst(d):84s} {shown}")
            bad += [f"k={k} op {i} {op} ({_inst(d)}): {key} err/tol = {val:.3g}" for key, val in worst.items()
                    if key != "err/S" and not val <= 1.0]
            if d.kind == 1:
                (_seen_tc if d.kernel == 1 else _seen_kf).add(_kf_key(d) if d.kernel == 2 else (d.bn, d.cpg, d.epi))
                if d.kernel == 2:
                    _seen_tr.add(d.tr)
            for p in outs:
                snap[p].copy_(st.views[p])
            if slot is not None:
                snap[st.slots_base][slot].copy_(st.views[st.slots_base][slot])
        assert torch.equal(st.dec.film_table(), film0), "the FiLM table changed"
        assert st.dec.saturation_count() == 0, "an epilogue saturated to the fp16 range"
    assert not bad, f"{name}: " + "; ".join(bad)
    _done.add(name)


def test_step_op_coverage():
    """Every conv_kf.cu instantiation the step plan can select was checked above at least once, with both walks."""
    missing_cfg = [c[0] for c in CONFIGS if c[0] not in _done]
    assert not missing_cfg, f"configurations not run (or failed): {missing_cfg}"
    print("conv_tc.cu instantiations checked:", sorted(_seen_tc))
    want = _kf_cases() - set(KF_NOT_IN_STEP)
    assert not (set(KF_NOT_IN_STEP) - _kf_cases()), "stale exclusion"
    assert want <= _seen_kf, f"conv_kf.cu instantiations never checked: {sorted(want - _seen_kf)}"
    assert _seen_tr == {0, 1}, f"walks checked: {_seen_tr}"
