"""The codec at the byte boundary on a real B200 (include/cdc_b200.h cdc_compress_rgb8 / cdc_decompress_rgb8): 8-bit RGB
in, CDC5 bytes out and back, each in one library call -- byte-identical to Codec.compress, pixel-identical to
Codec.decompress_bytes rounded to 8 bits, safe on a y container that starts off a 4-byte boundary, and rejecting
malformed streams before anything runs on them."""
import ctypes as C
import struct

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def codec():
    from tests.test_gpu_codec import _setup
    return _setup()[0]


def _rgb8(B, H, W, index):
    from oracle.weights import synthetic_image
    img = synthetic_image(B, H, W, index=index)
    return (img * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def _reference_bytes(codec, u8):
    return codec.compress(u8.permute(0, 3, 1, 2).float() / 255)[0]


def _reference_image(codec, data, steps, seeds, gamma):
    img = codec.decompress_bytes(data, steps, seeds=seeds, gamma=gamma)
    return (img * 255).round().to(torch.uint8).permute(0, 2, 3, 1).cpu()


def _nz(data):
    return struct.unpack_from("<Q", data, 16)[0]


def _c_decompress(codec, data, out, gamma=0.8):
    buf = bytes(data)
    return codec.L.cdc_decompress_rgb8(codec.ctx, buf, len(buf), gamma, C.c_void_p(out.data_ptr()), codec.dec._stream())


def _bind_for_decode(codec, shape, steps, seeds):
    codec.dec.bind(*shape)
    if codec.dec.steps != steps:
        codec.dec.set_sample_schedule(steps, *codec.dec.sampler)
    codec.dec.set_image_seeds(seeds)


@pytest.mark.parametrize("shape", [(2, 128, 192), (1, 256, 256)])
def test_compress_rgb8_equals_codec_compress(codec, shape):
    u8 = _rgb8(*shape, index=3)
    data = codec.compress_rgb8(u8)
    assert isinstance(data, bytes)
    assert data == _reference_bytes(codec, u8)
    # page-locked caller buffers are copied directly: the same bytes
    L, n = codec.L, C.c_int64(0)
    pin_in = u8.pin_memory()
    pin_out = torch.empty(L.cdc_compress_max_bytes(codec.ctx), dtype=torch.uint8).pin_memory()
    rc = L.cdc_compress_rgb8(codec.ctx, C.c_void_p(pin_in.data_ptr()), C.c_void_p(pin_out.data_ptr()), pin_out.numel(), C.byref(n),
                             codec.dec._stream())
    assert rc == 0 and pin_out[:n.value].numpy().tobytes() == data


@pytest.mark.parametrize("gamma", [0.8, 0.0])
def test_decompress_rgb8_equals_the_python_decode(codec, gamma):
    u8 = _rgb8(2, 128, 192, index=5)
    data = _reference_bytes(codec, u8)
    got = codec.decompress_rgb8(data, 5, seeds=[7, 8], gamma=gamma)
    ref = _reference_image(codec, data, 5, [7, 8], gamma)
    assert got.dtype == torch.uint8 and got.shape == (2, 128, 192, 3)
    assert torch.equal(got, ref)
    # page-locked input and output: the same pixels
    _bind_for_decode(codec, (2, 128, 192), 5, [7, 8])
    pin_data = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
    pin_out = torch.empty(2, 128, 192, 3, dtype=torch.uint8).pin_memory()
    rc = codec.L.cdc_decompress_rgb8(codec.ctx, C.c_void_p(pin_data.data_ptr()), len(data), gamma, C.c_void_p(pin_out.data_ptr()),
                                     codec.dec._stream())
    assert rc == 0 and torch.equal(pin_out, ref)


def test_y_container_off_a_4_byte_boundary_round_trips(codec):
    """nz is a whole number of 16-bit words; when it is 2 mod 4 the y container (and its u32 size table) starts off a
    4-byte boundary inside the stream.  Look for such a stream and check it both ways."""
    found = None
    for shape in [(1, 64, 64), (1, 64, 128), (1, 128, 64), (1, 128, 128), (1, 64, 192), (1, 192, 64), (1, 128, 192),
                  (1, 192, 192), (2, 64, 64), (2, 64, 128)]:
        for index in range(3):
            u8 = _rgb8(*shape, index=index)
            data = codec.compress_rgb8(u8)
            if _nz(data) % 4 == 2:
                found = (shape, u8, data)
                break
        if found:
            break
    assert found, "no synthetic image gave a z container of 2 mod 4 bytes"
    shape, u8, data = found
    print(f"{shape}: nz = {_nz(data)}, {len(data)} bytes")
    assert data == _reference_bytes(codec, u8)
    seeds = list(range(11, 11 + shape[0]))
    assert torch.equal(codec.decompress_rgb8(data, 5, seeds=seeds), _reference_image(codec, data, 5, seeds, 0.8))


def _malformed(data):
    nz, y = _nz(data), 24 + _nz(data)
    patch = lambda off, raw: data[:off] + raw + data[off + len(raw):]
    return {
        **{f"truncated to {n}": data[:n] for n in (0, 3, 23, 24, 24 + nz - 1, len(data) - 2)},
        "bad magic": patch(0, b"XDC5"),
        "header W differs": patch(12, struct.pack("<I", 256)),
        "header B differs": patch(4, struct.pack("<I", 1)),
        "nz > len": patch(16, struct.pack("<Q", len(data) + 8)),
        "z container with the wrong n_chan": patch(24 + 8, struct.pack("<I", 511)),
        "0xFF in the y size table": patch(y + 24, b"\xff" * 8),
    }


def test_malformed_streams_are_rejected_on_the_host(codec):
    from cdc_b200 import _ffi
    shape, seeds = (2, 128, 192), [7, 8]
    u8 = _rgb8(*shape, index=9)
    data = codec.compress_rgb8(u8)
    ref = _reference_image(codec, data, 5, seeds, 0.8)
    out = torch.empty(*shape, 3, dtype=torch.uint8)
    for name, bad in _malformed(data).items():
        with pytest.raises(ValueError):
            codec.decompress_rgb8(bad, 5, seeds=seeds)
        _bind_for_decode(codec, shape, 5, seeds)
        assert _c_decompress(codec, bad, out) in (_ffi.ERR_DATA, _ffi.ERR_SHAPE), name
        if name != "header B differs":  # (a well-formed stream of another shape: the context refuses it, not the parser)
            B, H, W = C.c_int(), C.c_int(), C.c_int()
            assert codec.L.cdc_stream_info(bad, len(bad), C.byref(B), C.byref(H), C.byref(W)) == _ffi.ERR_DATA, name
        assert torch.equal(codec.decompress_rgb8(data, 5, seeds=seeds), ref), f"valid stream after '{name}'"
    # a flipped payload byte passes the host checks; the decoder then either finds it or decodes other symbols
    flip = bytearray(data)
    flip[-1] ^= 0x55
    try:
        assert not torch.equal(codec.decompress_rgb8(bytes(flip), 5, seeds=seeds), ref)
    except ValueError:
        pass
    assert torch.equal(codec.decompress_rgb8(data, 5, seeds=seeds), ref)


def test_misuse_is_refused(codec):
    from cdc_b200 import _ffi
    L, shape = codec.L, (1, 128, 128)
    u8 = _rgb8(*shape, index=2)
    data = codec.compress_rgb8(u8)
    out = torch.empty(*shape, 3, dtype=torch.uint8)
    # no per-image seeds bound
    _bind_for_decode(codec, shape, 5, None)
    assert _c_decompress(codec, data, out) == _ffi.ERR_STATE
    # device pointers where host buffers belong
    _bind_for_decode(codec, shape, 5, [3])
    dev_out = torch.empty(*shape, 3, dtype=torch.uint8, device=DEV)
    assert _c_decompress(codec, data, dev_out) == _ffi.ERR_SHAPE
    dev_in = u8.to(DEV)
    host_out = torch.empty(L.cdc_compress_max_bytes(codec.ctx), dtype=torch.uint8)
    n = C.c_int64(0)
    assert L.cdc_compress_rgb8(codec.ctx, C.c_void_p(dev_in.data_ptr()), C.c_void_p(host_out.data_ptr()), host_out.numel(),
                               C.byref(n), codec.dec._stream()) == _ffi.ERR_SHAPE
    # too small an output buffer: refused, with the size needed reported
    assert L.cdc_compress_rgb8(codec.ctx, C.c_void_p(u8.data_ptr()), C.c_void_p(host_out.data_ptr()), 64, C.byref(n),
                               codec.dec._stream()) == _ffi.ERR_SHAPE
    assert n.value == len(data)
    # python-side argument checks
    for bad in (u8.float(), u8.permute(0, 3, 1, 2), u8[:, :100], u8.to(DEV)):
        with pytest.raises(ValueError):
            codec.compress_rgb8(bad)
    assert torch.equal(codec.decompress_rgb8(data, 5, seeds=[3]), _reference_image(codec, data, 5, [3], 0.8))
