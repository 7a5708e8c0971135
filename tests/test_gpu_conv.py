"""K-conv (tcgen05 implicit GEMM) parity on a real B200, every call through the C ABI (kernel-level entry points: include/cdc_b200_tools.h).
Checker: torch fp32 ops for the floating-point kernels, the CPU oracle for the integer path."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False  # the torch checker must be true fp32
torch.backends.cuda.matmul.allow_tf32 = False
DEV = "cuda:0"


def _lib():
    from cdc_b200 import _ffi
    return _ffi.lib()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _act_dtype():
    """Storage / MMA-operand dtype the library was built with (csrc/act.cuh): fp16 by default."""
    return torch.float16 if _lib().cdc_act_dtype() == 1 else torch.bfloat16


def _nhwc_act(t):
    return t.permute(0, 2, 3, 1).contiguous().to(_act_dtype())


def _run_conv(srcs, w, b, ksize, mode, force_bn=0, residual=None, stats=False):
    """srcs: list of NCHW fp32 cuda tensors (bf16-exact).  Returns (out NCHW fp32, GroupNorm sums or None)."""
    L = _lib()
    B, _, H, W = srcs[0].shape
    cout = w.shape[0]
    n_pad = (cout + 63) // 64 * 64
    OH, OW = (H // 2, W // 2) if mode == 1 else ((2 * H, 2 * W) if mode == 2 else (H, W))
    s = [_nhwc_act(t) for t in srcs]
    out = torch.full((B, OH, OW, n_pad), float("nan"), device=DEV, dtype=_act_dtype())
    res = _nhwc_act(residual) if residual is not None else None
    # [B][32][4] = (sum * 2^20, (squares mod 1024) * 2^20, floor(squares / 1024), unused): csrc/gn_sums.cuh
    st = torch.zeros(B, 32, 4, device=DEV, dtype=torch.int64) if stats else None
    rc = L.cdc_test_conv(0, _ptr(s[0]), s[0].shape[-1], _ptr(s[1]) if len(s) > 1 else C.c_void_p(0),
                         s[1].shape[-1] if len(s) > 1 else 0, B, H, W, _ptr(w.contiguous()), _ptr(b.contiguous()),
                         cout, ksize, mode, force_bn, _ptr(res), _ptr(out), _ptr(st), C.c_void_p(0))
    assert rc == 0, L.cdc_last_error(None).decode()
    torch.cuda.synchronize()
    o = out[..., :cout].float().permute(0, 3, 1, 2).contiguous()
    return o, st


def _ref_conv(srcs, w, b, ksize, mode, residual=None):
    x = torch.cat(srcs, dim=1)
    if mode == 2:
        x = F.interpolate(x, scale_factor=2, mode="nearest")
    y = F.conv2d(x, w, b, stride=2 if mode == 1 else 1, padding=ksize // 2)
    if residual is not None:
        y = y + residual
    return y


def _mk(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (scale * torch.randn(*shape, generator=g)).bfloat16().float().to(DEV)


def _check(o, ref, what):
    err = (o - ref).abs()
    # one output rounding: 2^-9 relative for bf16, 2^-12 for fp16 (+ fp32 accumulation-order noise)
    tol = (8e-3 if _act_dtype() == torch.bfloat16 else 1.5e-3) * ref.abs().clamp(min=1.0) + 1e-3
    bad = (err > tol).float().mean().item()
    assert torch.isfinite(o).all(), f"{what}: non-finite output"
    assert bad == 0.0, f"{what}: {bad:.4%} elements off, max err {err.max().item():.4f}, ref max {ref.abs().max().item():.3f}"


CONV_CASES = [
    # name, B, H, W, cins, cout, ksize, mode, force_bn
    ("3x3_c64_n64_row128", 1, 64, 128, [64], 64, 3, 0, 0),
    ("3x3_c128_n128_2x64", 2, 32, 64, [128], 128, 3, 0, 0),
    ("3x3_c192_n192", 1, 32, 32, [192], 192, 3, 0, 0),
    ("3x3_c256_n256", 1, 16, 16, [256], 256, 3, 0, 256),
    ("3x3_c256_n256_split64", 1, 16, 16, [256], 256, 3, 0, 64),
    ("3x3_dual_64+128_n128", 1, 32, 64, [64, 128], 128, 3, 0, 0),
    ("1x1_c256_n768", 1, 16, 16, [256], 768, 1, 0, 0),
    ("1x1_c320_n192", 1, 32, 32, [128, 192], 192, 1, 0, 0),
    ("s2_c64_n64", 1, 64, 128, [64], 64, 3, 1, 0),
    ("s2_c192_n192", 2, 32, 32, [192], 192, 3, 1, 0),
    ("up2_c128_n64", 1, 32, 64, [128], 64, 3, 2, 0),
    ("up2_c256_n256", 1, 8, 8, [256], 256, 3, 2, 0),
    ("ragged_48x24_c64_n64", 1, 24, 48, [64], 64, 3, 0, 0),
    ("ragged_s2_24x40", 1, 24, 40, [64], 128, 3, 1, 0),
    ("big_k4608_n256", 1, 16, 32, [256, 256], 256, 3, 0, 0),
    ("multi_tile_persistent", 4, 64, 128, [64], 64, 3, 0, 0),
    # kh-fused strip variant (conv_kf.cu): W a multiple of 128; one or two N tiles, one to three input chunks
    ("strip_c64_n64_256x256", 1, 256, 256, [64], 64, 3, 0, 0),
    ("strip_rows_not_multiple_of_L", 3, 50, 256, [64], 64, 3, 0, 0),
    ("strip_dual_64+64_n64", 1, 64, 384, [64, 64], 64, 3, 0, 0),
    ("strip_c128_n128", 2, 32, 128, [128], 128, 3, 0, 0),
    ("strip_c64+128_n128_streamed", 1, 48, 256, [64, 128], 128, 3, 0, 0),
    ("same_shape_through_conv_tc", 1, 64, 256, [64], 64, 3, 0, -1),
    # kh-fused strip variant (conv_kf.cu): ragged last segment, 1-row strips, long strips (accumulator ring wraps),
    # several units per CTA, two N tiles with two input chunks
    ("kf_ragged_w640", 1, 20, 640, [64], 64, 3, 0, 0),
    ("kf_two_rows", 1, 2, 256, [64], 64, 3, 0, 0),
    ("kf_long_strips", 8, 40, 1024, [64], 64, 3, 0, 0),
    ("kf_units_gt_ctas", 40, 16, 512, [64], 64, 3, 0, 0),
    ("kf_c128_n128_two_tiles", 1, 96, 384, [128], 128, 3, 0, 0),
    ("kf_dual_64+64_long", 2, 130, 256, [64, 64], 64, 3, 0, 0),
    # long strips (20+ rows per CTA): the six-in-eight accumulator ring of the 64-column tiles goes round several times
    # (rows 0 and 1 of every cycle are summed from two TMEM slots); the 32-column tiles' 16-slot ring wraps
    ("kf_c128_n128_long_strips", 8, 48, 512, [128], 128, 3, 0, 0),
    ("kf_c192_n128_bn32_long_strips", 4, 64, 256, [192], 128, 3, 0, 0),
    # nearest-x2 + conv3x3 through the kh-fused kernel (four parity 2x2 convs, scattered store)
    ("kf_up2_c128_n64", 1, 40, 128, [128], 64, 3, 2, 0),
    ("kf_up2_c192_n128_ragged", 2, 21, 192, [192], 128, 3, 2, 0),
    ("kf_up2_c256_n192", 1, 16, 96, [256], 192, 3, 2, 0),
    ("kf_up2_c256_n256_w48", 1, 10, 48, [256], 256, 3, 2, 0),
    ("kf_up2_one_row", 1, 1, 128, [128], 64, 3, 2, 0),
    # stride-2 conv3x3 through the kh-fused kernel (even / odd pixel tiles, two-row windows): output widths 128..384,
    # ragged last segment, one output row, accumulator-ring wrap, several units per CTA, two N tiles, dual source
    ("kf_s2_c64_n64_512x768", 1, 512, 768, [64], 64, 3, 1, 0),
    ("kf_s2_c64_n64_ragged_w400", 2, 36, 400, [64], 64, 3, 1, 0),
    ("kf_s2_one_output_row", 1, 2, 256, [64], 64, 3, 1, 0),
    ("kf_s2_long_strips", 6, 80, 512, [64], 64, 3, 1, 0),
    ("kf_s2_units_gt_ctas", 48, 8, 512, [64], 64, 3, 1, 0),
    ("kf_s2_c128_n128_two_tiles", 1, 256, 384, [128], 128, 3, 1, 0),
    ("kf_s2_dual_64+64_n64", 1, 64, 512, [64, 64], 64, 3, 1, 0),
    ("kf_s2_c128_n64", 2, 20, 256, [128], 64, 3, 1, 0),
    ("s2_c192_n192_128x192", 1, 128, 192, [192], 192, 3, 1, 0),  # (general kernel: no kf instantiation for these)
    ("s2_c256_n256_64x96", 2, 64, 96, [256], 256, 3, 1, 0),
]


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv_matches_torch(case):
    name, B, H, W, cins, cout, ks, mode, fbn = case
    srcs = [_mk((B, c, H, W), 10 + i) for i, c in enumerate(cins)]
    K = sum(cins) * ks * ks
    w = _mk((cout, sum(cins), ks, ks), 20, scale=1.0 / np.sqrt(K))
    b = _mk((cout,), 21, scale=0.5)
    o, _ = _run_conv(srcs, w, b, ks, mode, fbn)
    _check(o, _ref_conv(srcs, w, b, ks, mode), name)


def test_conv_up2_refuses_non_3x3():
    """Nearest-x2 convs run on parity weights pre-summed from 3x3 weights: any other kernel size is refused
    (CDC_ERR_SHAPE) before anything launches."""
    L = _lib()
    B, H, W, cin, cout = 1, 16, 16, 64, 64
    src = _nhwc_act(_mk((B, cin, H, W), 1))
    w, b = _mk((cout, cin, 1, 1), 2), _mk((cout,), 3)
    out = torch.zeros(B, 2 * H, 2 * W, cout, device=DEV, dtype=_act_dtype())
    rc = L.cdc_test_conv(0, _ptr(src), cin, C.c_void_p(0), 0, B, H, W, _ptr(w), _ptr(b), cout, 1, 2, 0, C.c_void_p(0),
                         _ptr(out), C.c_void_p(0), C.c_void_p(0))
    assert rc == -1, rc  # CDC_ERR_SHAPE
    assert "weight layout does not match the sources" in L.cdc_last_error(None).decode()
    assert not out.any()


def test_conv_residual_epilogue():
    srcs = [_mk((1, 256, 16, 16), 1)]
    w = _mk((256, 256, 1, 1), 2, scale=1 / 16.0)
    b = _mk((256,), 3)
    r = _mk((1, 256, 16, 16), 4)
    o, _ = _run_conv(srcs, w, b, 1, 0, 0, residual=r)
    _check(o, _ref_conv(srcs, w, b, 1, 0, residual=r), "residual")


@pytest.mark.parametrize("cfg", [(64, 2, 70, 256, 0), (128, 1, 32, 128, 0), (64, 8, 40, 1024, 0), (64, 40, 16, 512, 0), (128, 1, 96, 384, 0, 128),
                                 (64, 1, 50, 640, 0, 128),
                                 # kh-fused variant with N tiles of 32 / 48 channels (weights of wider layers stay resident)
                                 (128, 1, 64, 384, 0, 192), (128, 1, 40, 256, 0, 256), (192, 1, 64, 192, 0, 192),
                                 (256, 1, 32, 96, 0, 256), (256, 2, 16, 48, 0, 256),
                                 # transposed walk (strips along image columns): a 128 x 192 level, a tall narrow image
                                 (192, 1, 128, 192, 0, 192), (128, 2, 256, 40, 0, 128), (64, 1, 64, 128, -1), (64, 1, 64, 128, 0), (128, 2, 32, 64, 0), (128, 1, 16, 16, 64), (192, 1, 32, 32, 0),
                                 (256, 1, 16, 32, 256), (256, 1, 16, 16, 128), (256, 1, 16, 16, 64),
                                 (64, 1, 24, 48, 0)])
def test_conv_groupnorm_partials(cfg):
    cout, B, H, W, fbn = cfg[:5]
    cin = cfg[5] if len(cfg) > 5 else 64
    srcs = [_mk((B, cin, H, W), 5)]
    w = _mk((cout, cin, 3, 3), 6, scale=1 / (3.0 * np.sqrt(cin)))
    b = _mk((cout,), 7)
    o, part = _run_conv(srcs, w, b, 3, 0, fbn, stats=True)
    ref = _ref_conv(srcs, w, b, 3, 0)
    _check(o, ref, "stats-conv output")
    pd = part.double()
    got = torch.stack([pd[..., 0] / 2.0 ** 20, pd[..., 1] / 2.0 ** 20 + pd[..., 2] * 1024.0], dim=-1)  # (sum, sum of squares)
    rg = ref.double().reshape(B, 32, -1)
    want = torch.stack([rg.sum(-1), (rg * rg).sum(-1)], dim=-1)
    rel = (got - want).abs() / want.abs().clamp(min=1.0)
    assert rel.max().item() < 2e-3, f"GN partials off: {rel.max().item()}"
    # bitwise reproducible (integer accumulation is order-independent)
    o2, part2 = _run_conv(srcs, w, b, 3, 0, fbn, stats=True)
    assert torch.equal(part, part2) and torch.equal(o, o2)


