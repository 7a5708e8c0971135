"""cdc_stream_info parses a CDC5 stream on the host alone (no CUDA call), so it runs here without a GPU: what it accepts and
what it rejects, on streams laid out by hand ("CDC5" | u32 B, H, W | u64 nz | z container | y container; each container
"CDCR" | version | n_chan | hw | spc | 0 | u32 size[n_chan * spc] | streams)."""
import ctypes as C
import os
import struct

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "conditional-diffusion-model-for-compression_b200")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    if not os.path.exists(os.path.join(PKG, "libcdc_b200.so")):
        g.build()
    from cdc_b200 import _ffi
    return _ffi.lib()


def _container(n_chan, hw, spc, word_counts=None):
    ns = n_chan * spc
    sizes = [4 + 2 * w for w in (word_counts or [0] * ns)]
    return b"CDCR" + struct.pack("<5I", 1, n_chan, hw, spc, 0) + struct.pack(f"<{ns}I", *sizes) + bytes(sum(sizes))


def _stream(B=2, H=128, W=192, ch=256):
    hw = (H // 16) * (W // 16)
    z = _container(B * ch, hw // 16, 1, [i % 3 for i in range(B * ch)])  # (an odd number of words: nz % 4 == 2)
    y = _container(B * ch, hw, 2, [1] * (B * ch * 2))
    return b"CDC5" + struct.pack("<3IQ", B, H, W, len(z)) + z + y, len(z)


def _info(L, data):
    B, H, W = C.c_int(-1), C.c_int(-1), C.c_int(-1)
    rc = L.cdc_stream_info(data, len(data), C.byref(B), C.byref(H), C.byref(W))
    return rc, (B.value, H.value, W.value)


def _patched(data, off, raw):
    return data[:off] + raw + data[off + len(raw):]


def test_stream_info_reads_the_shape(lib):
    data, nz = _stream()
    assert nz % 4 == 2
    assert _info(lib, data) == (0, (2, 128, 192))
    assert _info(lib, data + b"\0" * 6) == (0, (2, 128, 192))  # bytes past the y container's streams are not read
    from cdc_b200.codec import Codec
    assert Codec.stream_info(data) == (2, 128, 192)


def _malformed(data, nz):
    y = 24 + nz
    return {
        **{f"truncated to {n}": data[:n] for n in (0, 3, 23, 24, 24 + nz - 1, len(data) - 2)},
        "bad magic": _patched(data, 0, b"CDC4"),
        "H not a multiple of 64": _patched(data, 8, struct.pack("<I", 130)),
        "W differs from the containers": _patched(data, 12, struct.pack("<I", 256)),
        "B does not divide the rows": _patched(data, 4, struct.pack("<I", 3)),
        "nz > len": _patched(data, 16, struct.pack("<Q", len(data))),
        "nz leaves no y container": _patched(data, 16, struct.pack("<Q", len(data) - 24)),
        "z container with the wrong n_chan": _patched(data, 24 + 8, struct.pack("<I", 511)),
        "bad z magic": _patched(data, 24, b"CDCX"),
        "y container version 2": _patched(data, y + 4, struct.pack("<I", 2)),
        "y spc 0": _patched(data, y + 16, struct.pack("<I", 0)),
        "y spc 33": _patched(data, y + 16, struct.pack("<I", 33)),
        "0xFF in the y size table": _patched(data, y + 24, b"\xff\xff\xff\xff"),
        "odd stream size": _patched(data, y + 24, struct.pack("<I", 5)),
        "stream size below the state": _patched(data, y + 24, struct.pack("<I", 2)),
    }


def test_stream_info_rejects_malformed_streams(lib):
    from cdc_b200 import _ffi
    from cdc_b200.codec import Codec
    data, nz = _stream()
    for name, bad in _malformed(data, nz).items():
        assert _info(lib, bad)[0] == _ffi.ERR_DATA, name
        with pytest.raises(ValueError):
            Codec.stream_info(bad)
