"""The integer and byte side of the codec on a real B200, over whole input domains, bit for bit.

One wrong bit here makes a stream undecodable, so every check is exact:

- the CDF row of a y symbol: the decoder's scale_rows_kernel on every fp16 sigma against the encoder's cdf_lookup, the
  oracle and the counting rule; cdc_cdf_lookup on every fp32 sigma;
- quantize on every finite fp16 y, dequant_to_act, rgb8_in on every byte at every position of its 16-pixel group, and
  rgb8_out at and around every rounding tie, against numpy float32 emulations of their documented arithmetic;
- the rANS coder at every stream count (spc) from 1 to 32, escapes of every payload length, degenerate CDF rows;
- cdc_decompress_rgb8 on CDC5 streams its encoder never writes: other stream counts, and a y container full of escapes.

Every stream fed to the device here is valid; malformed streams are the host parser's tests (test_gpu_bitstream_cabi.py).
"""
import ctypes as C
import struct
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SENTINEL = 0x5A5A  # int16 bits of the fp16 guard value around / beside the outputs
_spc_seen, _nb_seen = set(), set()


def _p(t):
    return C.c_void_p(t.data_ptr())


def _lib():
    from cdc_b200 import _ffi
    return _ffi.lib()


def _table():
    from oracle import entropy as oe
    return oe.scale_table()  # fp32 [64], ascending


def _rows_rule(s32):
    """The CDF row of a clamped, non-NaN fp32 sigma: #{j <= 62 : tab[j] < s}, compared exactly."""
    return np.searchsorted(_table()[:63].astype(np.float64), s32.astype(np.float64), side="left").astype(np.int32)


@pytest.fixture(scope="module")
def gauss():
    from oracle import entropy as oe
    return oe.build_gaussian_tables()


@pytest.fixture(scope="module")
def gauss_dev(gauss):
    from cdc_b200.decoder import DeviceTables
    return DeviceTables(gauss, DEV)


@pytest.fixture(scope="module")
def codec():
    """The codec of tests/test_gpu_codec.py: seed-0 UNet, seed-1 codec, its Gaussian and factorised-prior tables."""
    from tests.test_gpu_codec import _setup
    return _setup()[0]


# ---------------------------------------------------------------------------------------------------- CDF rows
def test_scale_rows_every_fp16_sigma_matches_the_encoder_side(gauss_dev):
    """Every fp16 bit pattern as the sigma half of the hyper-decoder's NHWC output (ldc = 2C, c_off = C, as
    cdc_decompress_rgb8 uses it), at an HW that is not a multiple of the 32-pixel tile.

    The rows must equal the encoder's (cdf_lookup on the fp32 sigma cdc_hyper_decode makes: fmaxf(fp32(h), 0.11f)),
    oracle.entropy.build_indexes, and #{j <= 62 : tab[j] < s}.  NaN: both product sides give row 0, because fmaxf drops
    the NaN before the search; the oracle keeps the NaN through torch.clamp, no comparison holds, and it gives row 63.
    Encoder and decoder agree, so streams decode; the oracle's row for NaN is the one place the product departs from it."""
    from cdc_b200.decoder import cdf_lookup
    from oracle import entropy as oe
    L = _lib()
    B, Cc, HW = 2, 256, 263
    n = HW * Cc
    pats = np.arange(65536, dtype=np.uint16)
    rng = np.random.default_rng(5)
    img = np.stack([np.resize(pats, n), rng.permutation(np.resize(pats, n))]).reshape(B, HW, Cc)
    buf = np.full((B, HW, 2 * Cc), 0x7E00, dtype=np.uint16)  # the mu half: NaN, never read
    buf[:, :, Cc:] = img
    sig = torch.from_numpy(buf.view(np.int16)).to(DEV)
    tab = torch.from_numpy(_table()).to(DEV)
    idx = torch.full((B, Cc, HW), -1, dtype=torch.int32, device=DEV)
    assert L.cdc_test_scale_rows(_p(sig), 2 * Cc, Cc, 0.11, _p(tab), _p(idx), B, Cc, HW, None) == 0
    torch.cuda.synchronize()
    got = idx.cpu().numpy()
    h = img.transpose(0, 2, 1).copy().view(np.float16)  # NCHW fp16
    f = h.astype(np.float32)
    s = np.fmax(f, np.float32(0.11))  # what cdc_hyper_decode stores as sigma (fmaxf: NaN -> 0.11)
    assert np.array_equal(got, _rows_rule(s)), "scale_rows != #{j <= 62 : tab[j] < max(sigma, 0.11f)}"
    enc = cdf_lookup(torch.zeros(B, Cc, HW, dtype=torch.int32), torch.from_numpy(s), gauss_dev, device=DEV)[0].cpu().numpy()
    assert np.array_equal(got, enc), "decoder rows (scale_rows on fp16) != encoder rows (cdf_lookup on fp32)"
    raw = cdf_lookup(torch.zeros(B, Cc, HW, dtype=torch.int32), torch.from_numpy(f), gauss_dev, device=DEV)[0].cpu().numpy()
    assert np.array_equal(got, raw), "cdf_lookup applies the 0.11 clamp itself: unclamped sigma must give the same rows"
    nan = np.isnan(f)
    orc = oe.build_indexes(torch.from_numpy(f), _table()).numpy()
    assert np.array_equal(got[~nan], orc[~nan])
    assert (got[nan] == 0).all() and (orc[nan] == 63).all()
    # the special values, stated
    bits = img.transpose(0, 2, 1)
    expo, mant, neg = (bits >> 10) & 0x1F, bits & 0x3FF, (bits >> 15) == 1
    assert (got[bits == 0x7C00] == 63).all(), "+inf"
    assert (got[bits == 0x7BFF] == 63).all(), "65504"
    assert (got[bits == 0xFC00] == 0).all(), "-inf"
    assert (got[bits == 0x8000] == 0).all() and (got[bits == 0] == 0).all(), "+-0"
    assert (got[neg & ~nan] == 0).all(), "negative sigma"
    assert (got[(expo == 0) & (mant != 0)] == 0).all(), "denormals"
    assert set(np.unique(got).tolist()) == set(range(64)), "every row is reached by some fp16 sigma"


def test_cdf_lookup_rows_every_fp32_sigma(gauss_dev):
    """cdc_cdf_lookup's row on all 2^32 fp32 sigma patterns, in chunks of 2^28, against
    torch.searchsorted(tab[:63], fmax(s, 0.11f)) on the device (NaN -> row 0, as fmaxf gives)."""
    from cdc_b200.decoder import cdf_lookup
    t0 = time.time()
    chunk = 1 << 28
    tab63 = torch.from_numpy(_table()[:63].copy()).to(DEV)
    lo = torch.tensor(np.float32(0.11), device=DEV)
    base = torch.arange(chunk, dtype=torch.int32, device=DEV)
    q = torch.zeros(chunk, dtype=torch.int32, device=DEV)
    for k in range(1 << 4):
        s = (base + (-(1 << 31) + k * chunk)).view(torch.float32)
        got = cdf_lookup(q, s, gauss_dev, device=DEV)
        exp = torch.searchsorted(tab63, torch.fmax(s, lo)).to(torch.int32)
        bad = (got[0] != exp).nonzero()
        assert bad.numel() == 0, f"chunk {k}: {bad.numel()} rows differ, first sigma bits {int(s[bad[0, 0]].view(torch.int32)):#010x}"
        del got, exp, s
    torch.cuda.synchronize()
    print(f"all 2^32 fp32 sigma patterns checked in {time.time() - t0:.1f} s")


# ---------------------------------------------------------------------------------------------------- quantize
def _finite_fp16():
    h = np.arange(65536, dtype=np.uint16).view(np.float16)
    return h[np.isfinite(h)].astype(np.float32)


def _mu_values():
    """64 fp32 mu: 0 (the prior's medians are 0), +-0.5, +-1.5, +-65504, values whose low bits make y - mu inexact near
    a half-integer, and random ones."""
    f = np.float32
    fixed = [0.0, -0.0, 0.5, -0.5, 1.5, -1.5, 65504.0, -65504.0, 2.0 ** -24, 1e-45, -1e-45, 3 * 2.0 ** -14,
             0.5 + 2.0 ** -10, 0.5 + 2.0 ** -14, 0.5 + 2.0 ** -20, -(0.5 + 2.0 ** -20), 0.5 - 2.0 ** -22, 1000.5 + 2.0 ** -13,
             -(2.5 - 2.0 ** -21), 0.25, -0.75, 12345.678, 0.1, -0.3]
    rng = np.random.default_rng(11)
    rest = np.concatenate([rng.standard_normal(20) * 3, rng.standard_normal(20) * 3000]).astype(np.float32)
    return np.concatenate([np.array(fixed, dtype=f), rest]).astype(f)


def _quantize(y, mu, mu_inner=0, mu_mod=0):
    L = _lib()
    q = torch.full(y.shape, -7, dtype=torch.int32, device=DEV)
    yh = torch.empty_like(y)
    assert L.cdc_quantize(_p(y), _p(mu), _p(q), _p(yh), y.numel(), mu_inner, mu_mod, None) == 0
    torch.cuda.synchronize()
    return q.cpu(), yh.cpu()


def test_quantize_every_finite_fp16_y():
    """q = rint(y - mu) (half-even), y_hat = q + mu on every finite fp16 y against 64 mu, elementwise and per channel
    (mu_mod), through the vector path and (unaligned pointers) the scalar path, against oracle.entropy.quantize_symbols."""
    from oracle import entropy as oe
    y1, mu = _finite_fp16(), _mu_values()
    assert mu.size == 64
    N = y1.size
    y = torch.from_numpy(np.tile(y1, 64))
    mu_e = torch.from_numpy(np.repeat(mu, N))
    q_ref, yh_ref = oe.quantize_symbols(y, mu_e)
    yd, md, mv = y.to(DEV), mu_e.to(DEV), torch.from_numpy(mu).to(DEV)

    def same(got, a, b, what):
        assert torch.equal(got[0], a), f"{what}: q"
        assert torch.equal(got[1].view(torch.int32), b.view(torch.int32)), f"{what}: y_hat"

    same(_quantize(yd, md), q_ref, yh_ref, "elementwise")
    same(_quantize(yd, mv, N, 64), q_ref, yh_ref, "per channel")
    # unaligned: everything through the scalar grid-stride loop
    same(_quantize(yd[1:], md[1:]), q_ref[1:], yh_ref[1:], "elementwise, scalar path")
    i = np.arange(1, 64 * N)
    q2, yh2 = oe.quantize_symbols(y[1:], torch.from_numpy(mu[((i - 1) // N) % 64]))
    same(_quantize(yd[1:], mv, N, 64), q2, yh2, "per channel, scalar path")


# ---------------------------------------------------------------------------------------------------- dequant_to_act
def _q_values(n, rng):
    big = [0, 1, -1, 65504, -65504, 65503, 65505, 65519, 65520, 65521, -65519, -65520, -65521, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1,
           -(2 ** 24 - 1), -(2 ** 24), -(2 ** 24 + 1), 2 ** 24 + 3, -(2 ** 31), 2 ** 31 - 1, -(2 ** 31) + 1, 2 ** 31 - 2,
           2047, 2049, 2051, 4095, 4097, 4099, -2049, -4097, 1023, 1025]
    pool = np.arange(-4200, 4200)
    return np.concatenate([big, rng.choice(pool, max(0, n - len(big)))])[:n].astype(np.int32)


def _mu16(n, rng):
    """fp16 mu: small multiples of 2^-14 (fp32 sums near an fp16 tie), normal values, random finite patterns."""
    a = (rng.integers(-64, 64, n) * 0.25 + rng.integers(0, 1 << 10, n) * 2.0 ** -14).astype(np.float16)
    b = (rng.standard_normal(n) * 64).astype(np.float16)
    c = rng.integers(0, 1 << 16, n).astype(np.uint16).view(np.float16)
    c = np.where(np.isfinite(c), c, np.float16(0))
    pick = rng.integers(0, 3, n)
    return np.where(pick == 0, a, np.where(pick == 1, b, c)).astype(np.float16)


def _act16(x32):
    """cvt.rn.satfinite.f16.f32: round to nearest even, finite values beyond the range to +-65504."""
    with np.errstate(over="ignore"):
        h = x32.astype(np.float16)
    return np.where(np.isinf(h) & np.isfinite(x32), np.copysign(np.float16(65504), x32).astype(np.float16), h)


@pytest.mark.parametrize("Cc", [192, 256])
@pytest.mark.parametrize("HW", [1, 24, 33])
@pytest.mark.parametrize("src", ["mu_vec", "mu_act"])
def test_dequant_to_act_is_fp16_of_the_fp32_sum(Cc, HW, src):
    """dst = fp16(__fadd_rn(float(q), mu)) NHWC, for both mu sources (the prior's median vector; channel c of the
    hyper-decoder's NHWC output with ldc = 2C), and nothing outside dst changes."""
    L = _lib()
    B = 2
    rng = np.random.default_rng(Cc * 100 + HW)
    n = B * Cc * HW
    q = _q_values(n, rng)
    q = np.concatenate([q[:34], rng.permutation(q[34:])]).reshape(B, Cc, HW)
    # channels 0-3: fp32 sums 0.75 fp32 ulp past a midpoint between fp16 values, where a rounding of the add other
    # than to nearest changes the fp16 result
    j = np.arange(B * HW).reshape(B, HW)
    q[:, 0], q[:, 1], q[:, 2], q[:, 3] = 2049 + 2 * j, -(2049 + 2 * j), 4098 + 4 * j, -(4098 + 4 * j)
    tie_mu = np.array([3 * 2.0 ** -14, -3 * 2.0 ** -14, 3 * 2.0 ** -13, -3 * 2.0 ** -13], dtype=np.float32)
    if src == "mu_vec":
        mu_vec = np.concatenate([(rng.integers(-8, 8, Cc // 2) * 0.25 + rng.integers(0, 1 << 12, Cc // 2) * 2.0 ** -14),
                                 rng.standard_normal(Cc - Cc // 2) * 300]).astype(np.float32)
        mu_vec[:4] = tie_mu
        mu = np.broadcast_to(mu_vec[None, None, :], (B, HW, Cc))
        md, ma, ldc = torch.from_numpy(mu_vec).to(DEV), None, 0
    else:
        act = np.full((B, HW, 2 * Cc), np.nan, dtype=np.float16)  # sigma half: NaN, never read
        act[:, :, :Cc] = _mu16(B * HW * Cc, rng).reshape(B, HW, Cc)
        act[:, :, :4] = tie_mu.astype(np.float16)
        mu = act[:, :, :Cc].astype(np.float32)
        md, ma, ldc = None, torch.from_numpy(act.view(np.int16)).to(DEV), 2 * Cc
    qn = q.transpose(0, 2, 1)  # NHWC order
    exp = _act16(qn.astype(np.float32) + mu).view(np.int16)
    guard = 4096
    full = torch.full((2 * guard + n,), SENTINEL, dtype=torch.int16, device=DEV)
    dst = full[guard:guard + n]
    qd = torch.from_numpy(q).to(DEV)
    rc = L.cdc_test_dequant(_p(qd), _p(md) if md is not None else None, _p(ma) if ma is not None else None, ldc, _p(dst), B, Cc, HW, None)
    assert rc == 0
    torch.cuda.synchronize()
    got = full.cpu().numpy()
    assert (got[:guard] == SENTINEL).all() and (got[guard + n:] == SENTINEL).all(), "wrote outside dst"
    bad = np.nonzero(got[guard:guard + n] != exp.reshape(-1))[0]
    assert bad.size == 0, f"{bad.size} values differ, first q = {qn.reshape(-1)[bad[0]]}, mu = {mu.reshape(-1)[bad[0]]!r}"


# ---------------------------------------------------------------------------------------------------- rgb8 in / out
def _byte_groups(ngroups):
    """Group g of 16 pixels (48 bytes) holds byte (g + k) % 256 at position k: 256 groups put every byte at every position."""
    g, k = np.meshgrid(np.arange(ngroups), np.arange(48), indexing="ij")
    return ((g + k) % 256).astype(np.uint8).reshape(-1)


def _rgb8_in_ref(v):
    f = np.float32
    return (f(2) * (v.astype(np.float32) / f(255)) - f(1)).astype(np.float16)


def test_rgb8_in_every_byte_at_every_position():
    """Channels 0-2 = fp16(2 * fp32(v / 255) - 1), channel 3 = +0, channels 4-63 untouched."""
    L = _lib()
    rgb = _byte_groups(256)
    npix = rgb.size // 3
    dst = torch.full((npix, 64), SENTINEL, dtype=torch.int16, device=DEV)
    rd = torch.from_numpy(rgb).to(DEV)
    assert L.cdc_test_rgb8_in(_p(rd), _p(dst), npix, None) == 0
    torch.cuda.synchronize()
    got = dst.cpu().numpy()
    exp = _rgb8_in_ref(rgb).view(np.int16).reshape(npix, 3)
    assert np.array_equal(got[:, :3], exp)
    assert (got[:, 3] == 0).all(), "channel 3 must be +0"
    assert (got[:, 4:] == SENTINEL).all(), "channels 4-63 must stay untouched"
    v = np.arange(256)
    once = (2.0 * v / 255.0 - 1.0).astype(np.float16)
    print(f"rgb8_in: {int((once != _rgb8_in_ref(v.astype(np.uint8))).sum())} of 256 bytes differ from fp16 rounded once "
          "from the float64 value")


def test_rgb8_in_equals_img_in_on_the_fp32_image(codec):
    """The 8-bit entry feeds the analysis encoder exactly what launch_img_in makes of the fp32 image u8 / 255."""
    from tests.op_reference import _view
    L = _lib()
    B, H, W = 2, 128, 192
    rgb = _byte_groups(B * H * W // 16)
    u8 = torch.from_numpy(rgb).reshape(B, H, W, 3)
    codec.analysis(u8.permute(0, 3, 1, 2).float() / 255)
    d = next(codec.dec.step_op_desc(i, 2) for i in range(len(codec.dec.step_ops(2))) if codec.dec.step_op_desc(i, 2).kind != 0)
    img64 = _view(d.src[0].p, (B, H, W, d.src[0].Cphys), torch.float16).clone()
    dst = torch.full((B * H * W, 64), SENTINEL, dtype=torch.int16, device=DEV)
    rd = torch.from_numpy(rgb).to(DEV)
    assert L.cdc_test_rgb8_in(_p(rd), _p(dst), B * H * W, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(dst[:, :3], img64.reshape(B * H * W, -1)[:, :3].view(torch.int16))


def _rgb8_out_inputs():
    """For every byte b the fp32 x nearest to where 255 * image01(x) = b +- 0.5, the x (searched within 64 ulps) where it
    lands on that tie exactly, and +-2 ulps around both; +-1 and values past them; +-inf, NaN, +-0."""
    f = np.float32
    xs = []
    ties = 0
    for b in range(256):
        for d in (-0.5, 0.5):
            x0 = f(2.0 * (b + d) / 255.0 - 1.0)
            near = [x0]
            for _ in range(64):
                near.append(np.nextafter(near[-1], f(-2)))
            hi = [x0]
            for _ in range(64):
                hi.append(np.nextafter(hi[-1], f(2)))
            cand = np.array(near + hi, dtype=f)
            w = _image01_255(cand)
            exact = cand[w == f(b + d)]
            ties += exact.size > 0
            for x in [x0, *exact[:2]]:
                up, dn = np.nextafter(x, f(2)), np.nextafter(x, f(-2))
                xs += [x, up, np.nextafter(up, f(2)), dn, np.nextafter(dn, f(-2))]
    one = [f(1), f(-1), np.nextafter(f(1), f(2)), np.nextafter(f(1), f(0)), np.nextafter(f(-1), f(-2)), np.nextafter(f(-1), f(0)),
           f(1.5), f(-1.5), f(1e30), f(-1e30), f(np.inf), f(-np.inf), f(np.nan), f(-0.0), f(0.0), f(1e-45), f(-1e-45)]
    x = np.array(xs + one, dtype=f)
    return x, ties


def _image01_255(x):
    """fp32 emulation of rgb8_out before the rounding: 255 * ((fminf(fmaxf(x, -1), 1) + 1) / 2)."""
    f = np.float32
    t = np.fmin(np.fmax(x.astype(f), f(-1)), f(1))  # (fmax / fmin drop a NaN, as fmaxf / fminf do)
    return ((t + f(1)) / f(2)) * f(255)


def test_rgb8_out_at_every_rounding_tie(codec):
    """rgb8 = rint(255 * image01(x)) half-even, against the numpy float32 emulation and against cdc_get_x(to_image01)
    followed by torch.round: the contract decompress_rgb8 documents."""
    L = _lib()
    x, ties = _rgb8_out_inputs()
    print(f"rgb8_out: {x.size} inputs; an exact x.5 tie found for {ties} of 512 (byte, side)")
    assert ties >= 300
    B, H, W = 2, 128, 192
    npix = B * H * W
    xs = np.zeros(npix * 3, dtype=np.float32)
    assert x.size <= xs.size
    xs[:x.size] = x
    exp = np.rint(_image01_255(xs)).astype(np.uint8)
    xd = torch.from_numpy(xs).to(DEV)
    out = torch.zeros(npix * 3, dtype=torch.uint8, device=DEV)
    assert L.cdc_test_rgb8_out(_p(xd), _p(out), npix, None) == 0
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    bad = np.nonzero(got != exp)[0]
    assert bad.size == 0, f"{bad.size} bytes differ, first x = {xs[bad[0]]!r}: {got[bad[0]]} != {exp[bad[0]]}"
    dec = codec.dec
    dec.bind(B, H, W)
    dec._set_x(xd.reshape(B, H, W, 3).permute(0, 3, 1, 2))
    img = dec._get_x(to_image=True)
    ref = torch.round(img * 255).to(torch.uint8).permute(0, 2, 3, 1).reshape(-1)
    assert torch.equal(out, ref), "rgb8_out != round(255 * cdc_get_x(to_image01))"


# ---------------------------------------------------------------------------------------------------- rANS
def _symbols(q, sigma, tables):
    from oracle import entropy as oe
    return [t.numpy() for t in oe.cdf_lookup(torch.from_numpy(q), torch.from_numpy(sigma), tables)]


def _gpu_encode(sym, tables_dev, n_chan, hw, spc):
    from cdc_b200.bitstream import rans_encode
    return rans_encode([torch.from_numpy(np.ascontiguousarray(s)) for s in sym], tables_dev, n_chan, hw, DEV, spc=spc).cpu().numpy().tobytes()


def _cdc_rans_decode(data, idx, tables_dev, n_chan, hw, spc):
    """cdc_rans_decode called directly with the stream count."""
    L = _lib()
    d = torch.frombuffer(bytearray(data), dtype=torch.uint8).to(DEV)
    ix = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int32).reshape(-1)).to(DEV)
    q = torch.full((n_chan * hw,), 12345, dtype=torch.int32, device=DEV)
    scratch = torch.empty(8 * n_chan * spc + 8, dtype=torch.uint8, device=DEV)
    status = torch.full((1,), 7, dtype=torch.int32, device=DEV)
    t = tables_dev
    rc = L.cdc_rans_decode(_p(d), d.numel(), _p(ix), _p(t.cdf), _p(t.row_start), _p(t.cdf_length), _p(t.offset), t.rows, n_chan, hw,
                           spc, _p(scratch), _p(q), _p(status), None)
    assert rc == 0
    torch.cuda.synchronize()
    assert int(status.item()) == 0, "cdc_rans_decode reports a corrupt container"
    return q.cpu().numpy()


def _check_coder(q, idx, sym, tables, tables_dev, n_chan, hw, spc):
    """GPU encode byte-exact with oracle.rans.encode at this spc; both GPU decoders give q back from the oracle's bytes."""
    from cdc_b200.bitstream import rans_decode
    from oracle import rans as orans
    ref = orans.encode(*sym, tables.cdf_length, n_chan, hw, spc=spc)
    assert _gpu_encode(sym, tables_dev, n_chan, hw, spc) == ref, f"spc {spc}, hw {hw}: encoded bytes differ from the oracle's"
    qf = q.reshape(-1)
    assert np.array_equal(rans_decode(ref, torch.from_numpy(idx.reshape(-1).astype(np.int32)), tables_dev, DEV).cpu().numpy(), qf)
    assert np.array_equal(_cdc_rans_decode(ref, idx, tables_dev, n_chan, hw, spc), qf)
    _spc_seen.add(spc)
    return ref


@pytest.mark.parametrize("hw", [1, 7, 64, 100, 1536])
def test_rans_every_stream_count(gauss, gauss_dev, hw):
    """spc = 1..32 (powers of two or not, above hw: streams with no symbols), n_chan = 3, some escapes in every row."""
    rng = np.random.default_rng(hw)
    n_chan = 3
    sigma = np.exp(rng.uniform(np.log(0.05), np.log(300.0), n_chan * hw)).astype(np.float32)
    q = np.round(rng.standard_normal(n_chan * hw) * sigma * 1.3).astype(np.int32)
    esc = rng.random(n_chan * hw) < 0.05
    q[esc] = rng.integers(-(1 << 20), 1 << 20, int(esc.sum()))
    sym = _symbols(q, sigma, gauss)
    for spc in range(1, 33):
        _check_coder(q, sym[0], sym, gauss, gauss_dev, n_chan, hw, spc)


def _escape_q(raw, row, tables):
    """The q that lookup_rows turns into escape `raw` in `row`: odd raw below the support, even raw above it."""
    off, max_v = int(tables.offset[row]), int(tables.cdf_length[row]) - 2
    v = -(raw + 1) // 2 if raw & 1 else max_v + raw // 2
    return off + v


@pytest.mark.parametrize("spc", [1, 3, 32])
def test_rans_escapes_of_every_length(gauss, gauss_dev, spc):
    """raw = 2^nb - 1 and min(2^(nb + 1) - 2, 2^31 - 1) for nb = 0..31 in four rows, between ordinary symbols: together
    they reach both ends of the representable q range, [offset - 2^30, offset + max_v + 2^30 - 1]."""
    from cdc_b200.decoder import cdf_lookup
    tab = _table()
    raws = sorted({r for nb in range(32) for r in (2 ** nb - 1, min(2 ** (nb + 1) - 2, 2 ** 31 - 1))})
    rows = [0, 20, 45, 63]
    rng = np.random.default_rng(spc)
    n_chan, hw = 3, 160
    sigma = tab[rng.integers(0, 64, n_chan * hw)].astype(np.float32)
    q = np.round(rng.standard_normal(n_chan * hw) * sigma).astype(np.int64)
    slots = rng.permutation(n_chan * hw)[:len(raws) * len(rows)]
    want = {}
    for k, (raw, row) in enumerate((r, w) for r in raws for w in rows):
        sigma[slots[k]] = tab[row]
        q[slots[k]] = _escape_q(raw, row, gauss)
        want[slots[k]] = raw
    assert q.min() >= -(2 ** 31) and q.max() < 2 ** 31
    q = q.astype(np.int32)
    off, max_v = gauss.offset[rows].astype(np.int64), gauss.cdf_length[rows].astype(np.int64) - 2
    assert q.min() == (off - 2 ** 30).min() and q.max() == (off + max_v + 2 ** 30 - 1).max()
    sym = _symbols(q, sigma, gauss)
    gpu = [t.cpu().numpy() for t in cdf_lookup(torch.from_numpy(q), torch.from_numpy(sigma), gauss_dev, device=DEV)]
    for a, b in zip(gpu, sym):
        assert np.array_equal(a, b), "cdf_lookup != oracle lookup_rows"
    slot_idx = np.array(list(want))
    assert np.array_equal(sym[4][slot_idx], np.array(list(want.values()))), "the planted escapes carry the intended raw"
    _check_coder(q, sym[0], sym, gauss, gauss_dev, n_chan, hw, spc)
    for raw in want.values():
        _nb_seen.add(int(raw + 1).bit_length() - 1)


def _degenerate_tables():
    """Row 0: length 2 (max_v = 0, every symbol escapes).  Row 1: frequency-1 bins first, in the middle, last and as the
    escape bin.  Row 2: one bin of 65535.  Row 3: one bin of 1, the escape bin 65535."""
    from oracle import entropy as oe
    rows = [np.array([0, 65536]), np.concatenate([[0], np.cumsum([1, 32766, 1, 32766, 1, 1])]),
            np.array([0, 65535, 65536]), np.array([0, 1, 65536])]
    for r in rows:
        assert r[-1] == 65536 and (np.diff(r) > 0).all()
    return oe._pack(rows, [0, -2, 0, 5], np.zeros(64, dtype=np.float32))


@pytest.mark.parametrize("spc", [1, 3, 32])
def test_rans_degenerate_cdf_rows(spc):
    from cdc_b200.decoder import DeviceTables, cdf_lookup
    tb = _degenerate_tables()
    tdev = DeviceTables(tb, DEV)
    B, nrow, hw = 2, 4, 300
    rng = np.random.default_rng(100 + spc)
    q = np.zeros((B, nrow, hw), dtype=np.int64)
    for r in range(nrow):
        off, max_v = int(tb.offset[r]), int(tb.cdf_length[r]) - 2
        inside = off + rng.integers(0, max(max_v, 1), (B, hw)) if max_v else np.full((B, hw), off)
        raws = rng.choice([0, 1, 2, 3, 4, 5, 100, 2 ** 16 - 1, 2 ** 16, 2 ** 17 + 3, 2 ** 30, 2 ** 31 - 2, 2 ** 31 - 1], (B, hw))
        out = np.vectorize(lambda x: _escape_q(int(x), r, tb))(raws)
        q[:, r] = np.where(rng.random((B, hw)) < 0.4, out, inside)
    q = q.astype(np.int32)
    idx = np.broadcast_to(np.arange(nrow, dtype=np.int32)[None, :, None], q.shape).copy()
    from oracle import entropy as oe
    sym = [t.numpy() for t in oe.lookup_rows(torch.from_numpy(q), torch.from_numpy(idx), tb)]
    gpu = [t.cpu().numpy() for t in cdf_lookup(torch.from_numpy(q), None, tdev, device=DEV)]
    for a, b in zip(gpu, sym):
        assert np.array_equal(a, b), "cdf_lookup (row = channel) != oracle lookup_rows"
    assert (sym[1][:, 0] == 0).all(), "every symbol of the length-2 row is an escape"
    _check_coder(q, idx, sym, tb, tdev, B * nrow, hw, spc)


# ---------------------------------------------------------------------------------------------------- the C ABI decoder
def _rgb8(B, H, W, index):
    from oracle.weights import synthetic_image
    img = synthetic_image(B, H, W, index=index)
    return (img * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def _reference_image(codec, data, steps, seeds, gamma=0.8):
    img = codec.decompress_bytes(data, steps, seeds=seeds, gamma=gamma)
    return (img * 255).round().to(torch.uint8).permute(0, 2, 3, 1).cpu()


def _cdc5(B, H, W, zs, ys):
    return b"CDC5" + struct.pack("<3IQ", B, H, W, len(zs)) + zs + ys


@pytest.fixture(scope="module")
def canonical(codec):
    B, H, W = 2, 128, 192
    u8 = _rgb8(B, H, W, index=5)
    data, enc = codec.compress(u8.permute(0, 3, 1, 2).float() / 255)
    assert data == codec.compress_rgb8(u8)
    pix = codec.decompress_rgb8(data, 5, seeds=[7, 8])
    return (B, H, W), data, enc, pix


@pytest.mark.parametrize("spc_z,spc_y", [(2, 2), (3, 3), (32, 32), (1, 32)])
def test_decompress_rgb8_at_other_stream_counts(codec, canonical, spc_z, spc_y):
    """The z and y symbols of codec.encode re-encoded at stream counts other than the encoder's (1 for both containers
    at this size; spc_z = 32 > hw_z = 6: streams without symbols); the C ABI decoder must give the canonical stream's
    pixels, decode_symbols its (qz, q)."""
    from cdc_b200.bitstream import parse_header, rans_encode
    (B, H, W), data, enc, pix = canonical
    c, h, w = enc["q"].shape[1:]
    zs = rans_encode(enc["z_sym"], codec.fact, B * c, (h // 4) * (w // 4), DEV, spc=spc_z).cpu().numpy().tobytes()
    ys = rans_encode(enc["y_sym"], codec.gauss, B * c, h * w, DEV, spc=spc_y).cpu().numpy().tobytes()
    assert parse_header(zs)[2] == spc_z and parse_header(ys)[2] == spc_y
    other = _cdc5(B, H, W, zs, ys)
    assert other != data
    qz, q = codec.decode_symbols(other)
    assert torch.equal(qz, enc["qz"]) and torch.equal(q, enc["q"])
    assert torch.equal(codec.decompress_rgb8(other, 5, seeds=[7, 8]), pix)
    _spc_seen.update((spc_z, spc_y))


def test_decompress_rgb8_of_an_escape_heavy_y_container(codec, canonical):
    """Every 7th y symbol moved 1 to 40 past its row's support (q = +-(center + d), center = -offset[idx]), alternating
    sides, re-looked-up and re-encoded: a valid stream that is mostly escapes.  decode_symbols must return exactly the
    modified q, and cdc_decompress_rgb8 must equal decompress_bytes rounded."""
    from cdc_b200.bitstream import rans_encode
    from cdc_b200.decoder import cdf_lookup
    (B, H, W), data, enc, _ = canonical
    c, h, w = enc["q"].shape[1:]
    idx = enc["y_sym"][0].reshape(-1)
    center = -codec.gauss.offset[idx.long()]
    q = enc["q"].clone().reshape(-1)
    sel = torch.arange(0, q.numel(), 7, device=DEV)
    k = torch.arange(sel.numel(), device=DEV)
    d = 1 + k % 40
    q[sel] = torch.where(k % 2 == 0, -(center[sel] + d), center[sel] + d).to(torch.int32)
    q = q.reshape(enc["q"].shape)
    sym = cdf_lookup(q, enc["sigma"], codec.gauss, device=DEV)
    assert torch.equal(sym[0], enc["y_sym"][0])
    esc = sym[1] == codec.gauss.cdf_length[sym[0].long()] - 2
    assert int(esc.sum()) >= sel.numel()
    ys = rans_encode(sym, codec.gauss, B * c, h * w, DEV).cpu().numpy().tobytes()
    nz = struct.unpack_from("<Q", data, 16)[0]
    heavy = _cdc5(B, H, W, data[24:24 + nz], ys)
    qz2, q2 = codec.decode_symbols(heavy)
    assert torch.equal(qz2, enc["qz"]) and torch.equal(q2, q)
    got = codec.decompress_rgb8(heavy, 5, seeds=[7, 8])
    assert torch.equal(got, _reference_image(codec, heavy, 5, [7, 8]))
    print(f"escape-heavy y container: {int(esc.sum())} escapes of {q.numel()} symbols, {len(ys)} bytes")


def test_every_stream_count_and_escape_length_was_checked():
    assert _spc_seen >= set(range(1, 33)), f"stream counts never checked: {sorted(set(range(1, 33)) - _spc_seen)}"
    assert _nb_seen >= set(range(32)), f"escape lengths never checked: {sorted(set(range(32)) - _nb_seen)}"
