"""float64 references of the ops the plan builds (include/cdc_b200_tools.h cdc_seq_op_describe), their tolerances, and the
buffers an op may write.  Shared by tests/test_gpu_step_ops.py (the denoise step) and tests/test_gpu_codec_ops.py (the
context net, analysis encoder and hyper networks).  Test infrastructure only.

Conv weights are rounded to a fixed-point grid (multiples of 2^-m, every sum of four weights below 2^11 grid steps), so
the fp16 repack and the pre-summed nearest-x2 parity weights are exact and the only conv error left is the fp32
accumulation order: the tolerances below are derived from that, op by op.
"""
import math
import os
import re

import torch
import torch.nn.functional as F

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# fp32 accumulation in the tensor cores: |conv - ref| <= C_ACC * S, S = conv(|x|, |w|) + |b| (+ |residual|).
# Measured on a B200 (1000 W power limit) over every conv of every step configuration of tests/test_gpu_step_ops.py: worst
# err/S 3.3e-7 (the final conv, whose fp32 output is not rounded to 16 bits), 1.5e-7 for the others.  C_ACC = 2^-19
# (1.9e-6) is 5.8x that.  The codec convs reach K = 6400 (the 5x5 convs of the hyper networks) against at most 4608 in
# the step; over every configuration of tests/test_gpu_codec_ops.py (same B200) their worst err/S is 3.1e-7 (henc.c3 at
# 2048 x 2048, K = 6400), 2.3e-7 for the context net and the encoder: under half of C_ACC, which therefore stays.
# (A dropped tap or a wrong bias is an error of order S: hundreds of thousands of C_ACC.)
C_ACC = 2.0 ** -19
U16 = 2.0 ** -11          # unit roundoff of fp16: one rounding to nearest of the stored value
SUB16 = 2.0 ** -25        # half the spacing of fp16 subnormals: the rounding error floor near zero
U32 = 2.0 ** -24
TANH_APPROX = 2.0 ** -10.98  # max relative error of tanh.approx.f32 (PTX ISA), used by the GroupNorm + SiLU transform

KF_MODE = {0: 0, 2: 1, 1: 2}  # conv mode (0 stride 1, 1 stride 2, 2 nearest-x2) -> conv_kf.cu MODE
EPI = {"EPI_STORE": 0, "EPI_STATS": 1, "EPI_DDIM": 2}


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


def image_scale(B):
    """Per-image input scale 2^((b mod 4) - 1), [B, 1, 1, 1]: every image of a batch gets its own GroupNorm statistics (a
    kernel that used another image's would be off by a factor, not by sampling noise), and a power of two keeps the
    synthetic inputs exact."""
    return (2.0 ** (torch.arange(B, dtype=torch.float64) % 4 - 1)).float().reshape(B, 1, 1, 1)


def kf_acc_ring(key):
    """Accumulator-ring length (logical slots) of the conv_kf.cu instantiation key (_kf_key): 6 with the fused residual
    conv or the aliased ring of the 64-column tiles (BN = 32 with the residual conv likewise), else min(16, 512 / BN)."""
    bn, _, epi, _, _, _, mode, res1, _ = key
    alias = mode == 0 and epi != 2 and ((bn == 64 and not res1) or (bn == 32 and res1))
    return 6 if res1 or alias else min(16, 512 // bn)


def kf_geometry(d, B):
    """Which parts of the strip kernel's unit loop a conv_kf.cu op (description d, batch B) runs: a set of
    "several_units" (a CTA runs more than one unit), "two_images" (one CTA's units belong to two images), "one_row"
    (strips of one row), "uneven" (strips of unequal length), "ragged" (the last 128-pixel segment is partly outside the
    image) and "ring_wrap" (a strip is longer than the accumulator ring).  From the launch geometry of the description."""
    units, per_img = B * d.nseg * d.strips, d.nseg * d.strips
    f = set()
    if units > d.g1:
        f.add("several_units")
        if any(len({u // per_img for u in range(c, units, d.g1)}) > 1 for c in range(d.g1)):
            f.add("two_images")
    if d.strips == d.rows:
        f.add("one_row")
    if d.rows % d.strips:
        f.add("uneven")
    s2 = d.mode == 1  # stride 2: the kernel walks the output grid
    cols = (d.src[0].H if d.tr else d.src[0].W) >> (1 if s2 else 0)
    if cols % 128:
        f.add("ragged")
    if -(-d.rows // d.strips) > kf_acc_ring(_kf_key(d)):
        f.add("ring_wrap")
    return f


class GeometrySeen:
    """The launch geometry of the checked conv ops: kf_geometry per conv_kf.cu instantiation and per (walk, MODE), and the
    conv_tc.cu instantiations that ran more tiles than CTAs."""

    def __init__(self):
        self.kf, self.cls, self.tc_waves = {}, set(), set()

    def add(self, d, B):
        if d.kind != 1:
            return
        if d.kernel == 2:
            geo = kf_geometry(d, B)
            self.kf.setdefault(_kf_key(d), set()).update(geo)
            self.cls.update(((d.tr, _kf_key(d)[6]), g) for g in geo)
        elif d.n_tiles > d.grid:
            self.tc_waves.add((d.bn, d.cpg, d.epi))


def _geom(d, B):
    """The launch geometry of conv op d, for the per-op listings."""
    if d.kind != 1:
        return ""
    if d.kernel == 1:
        return f"{d.n_tiles} tiles / {d.grid} CTAs"
    return (f"{B * d.nseg * d.strips} units / {d.g1} CTAs x {d.n_tiles} tiles, {d.nseg} seg, {d.strips} strips of "
            f"{d.rows} rows")


def fixed_point_(module):
    """Every conv (and transposed-conv) weight of module on a per-layer grid 2^-m, m the largest with
    4 * max|w| * 2^m < 2^11: the weights and every sum of four of them (the nearest-x2 parity weights) are exact in fp16."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if name.endswith(".weight") and p.dim() == 4:
                m = math.floor(math.log2(2.0 ** 11 / (4.0 * p.abs().max().item())))
                if 4.0 * p.abs().max().item() * 2.0 ** m >= 2.0 ** 11:
                    m -= 1
                p.copy_(torch.round(p * 2.0 ** m) / 2.0 ** m)
    return module


def _fixed_point_unet(ocfg):
    """Oracle UNet (seed 0) with its conv weights on the fixed-point grid (fixed_point_)."""
    from oracle.weights import build_unet
    return fixed_point_(build_unet(ocfg, seed=0))


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
    """mode 0 stride 1, 1 stride 2, 2 nearest-x2 input, 3 ConvTranspose2d(5, stride 2, padding 2, output_padding 1) with
    w [in, out, 5, 5]."""
    if mode == 3:
        return F.conv_transpose2d(x, w, stride=2, padding=2, output_padding=1)
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


class SeqBuffers:
    """Views of every buffer the ops of one sequence read or write (from their descriptions), and which of them an op
    may write.  Subclasses set dec, desc, B, H, W_ and call _bind_views()."""

    slots_base, nslots = None, 0

    def _bind_views(self):
        B, H, W = self.B, self.H, self.W_
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

    def check_writes(self, op, d, snap):
        """Everything op (description d, just run) does not declare as its output is bitwise what snap holds."""
        outs, slot = self.outputs(d)
        for p, v in self.views.items():
            if p in outs:
                continue
            if p == self.slots_base and slot is not None:
                keep = [j for j in range(self.nslots) if j != slot]
                assert torch.equal(v[keep], snap[p][keep]), f"{op}: wrote a GroupNorm slot it does not own"
            else:  # (bit patterns: a buffer no op has written yet may hold NaNs)
                assert torch.equal(_bits(v), _bits(snap[p])), f"{op}: wrote a buffer it does not declare as output"
        if d.kind == 0:
            assert not self.views[self.slots_base].any(), f"{op}: GroupNorm slots not cleared"

    def advance(self, d, snap):
        """Copy what op d wrote into snap: the inputs of the ops after it."""
        outs, slot = self.outputs(d)
        for p in outs:
            if p != self.slots_base:
                snap[p].copy_(self.views[p])
        if d.kind == 0:
            snap[self.slots_base].copy_(self.views[self.slots_base])
        elif slot is not None:
            snap[self.slots_base][slot].copy_(self.views[self.slots_base][slot])


def _ratio(err, tol):
    return (err / tol).max().item()


def _check_conv(st, d, snap, k):
    """conv (+fused residual conv, +fused input GroupNorm, +statistics, +LeakyReLU, +sampler update) against float64."""
    w = st.W[d.weight.decode() + ".weight"]
    b = st.W[d.weight.decode() + ".bias"]
    srcs = [_nchw(snap[t.p], t.C) for t in (d.src[0], d.src[1]) if t.p]
    x = torch.cat(srcs, dim=1)
    if d.mode != 3 and w.shape[1] != x.shape[1]:
        # a stem: its image channels are the first of a 64-channel chunk (the step's x_t: 3 of the first source's 64
        # channels, then the context channels; the encoder's image: 3 of its one source's 64)
        n1 = srcs[1].shape[1] if len(srcs) > 1 else 0
        n0 = w.shape[1] - n1
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
            if getattr(st, "image_seeds", None):  # per-image seeds bound (cdc_set_image_seeds)
                from tests.seeded_reference import philox_normal_images, step_plane
                z = philox_normal_images(st.image_seeds, *step_plane(k), st.H, st.W_)
            else:
                from oracle.sampler import philox_normal
                z = philox_normal(st.seed, k, st.B, st.H, st.W_)
            z = _nhwc(z.double().to(DEV))
            xp = xp + sg * z
            tol = tol + sg * 2.0 ** -18 * (z.abs() + 1.0)  # fp32 logf / sqrtf / sincospif of the Box-Muller pair
        got_x = st.views[d.x].double()
        worst["x_prev"] = _ratio((got_x - xp).abs(), tol)
        xpad = st.views[d.xpad]
        assert torch.equal(xpad[..., :3], st.views[d.x].half()), "xpad channels 0-2 != fp16(x_prev)"
        assert not xpad[..., 3:].any(), "xpad channels 3-15 not zero"
        worst["err/S"] = (((got_x0 - x0).abs() - U32 * x0.abs()).clamp(min=0) / _nhwc(S)[..., :3]).max().item()
        return worst
    rnd = U16 * ref.abs()
    if d.act_slope != 0.0:  # LeakyReLU after the bias: 1-Lipschitz, so the accumulation bound carries over; one fp32
        # rounding of slope * x on the negative side
        ref = torch.where(ref >= 0, ref, float(d.act_slope) * ref)
        rnd = (U16 + U32) * ref.abs()
    got = _nchw(st.views[d.out.p])[:, :ref.shape[1]]
    tol = rnd + (1.0 + U16) * acc + SUB16
    worst["out"] = _ratio((got - ref).abs(), tol)
    if not d.apply:  # (measured accumulation error, the basis of C_ACC)
        worst["err/S"] = (((got - ref).abs() - rnd - SUB16).clamp(min=0) / S).max().item()
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
