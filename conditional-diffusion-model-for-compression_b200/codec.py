"""Host-side mirror of the oracle's codec around the decode loop (oracle/codec.py Codec; SURVEY.md section 8 rows f2 / J1):
analysis encoder, hyper-encoder / hyper-decoder, latent rounding and CDF lookup, all on the device through the C ABI.

    codec = Codec(decoder)                  # a Decoder created with the "codec.*" (and "context.*") weights
    enc   = codec.encode(img01)             # dict with the oracle's keys: y, z, qz, z_hat, mu, sigma, q, y_hat, y_sym, z_sym
    img   = codec.decompress(enc["qz"], enc["q"], steps=17)
    data  = codec.compress_rgb8(rgb8)       # uint8 [B,H,W,3] -> CDC5 bytes, one library call (cdc_compress_rgb8)
    rgb8  = codec.decompress_rgb8(data, 17, seeds=[7])   # CDC5 bytes -> uint8 [B,H,W,3] (cdc_decompress_rgb8)

Determinism is the contract that matters for a bitstream: encoder and decoder both derive (mu, sigma) from z_hat with
the same kernels (cdc_hyper_decode), fixed accumulation order, so q / idx / (lo, hi) agree bit for bit between the two
sides.  Against the fp32 CPU oracle, y / mu / sigma agree to the 16-bit storage tolerance (tests/test_gpu_codec.py)."""
import ctypes as C

import torch

from . import _ffi, entropy_tables
from .decoder import Decoder, DeviceTables, _f32c, _seed_values, _stream_ptr, cdf_lookup, quantize_symbols


class Codec:
    def __init__(self, decoder: Decoder, gauss_tables=None, fact_tables=None, median=None):
        """gauss_tables / fact_tables: CDF tables (entropy_tables.Tables layout; the oracle's CDFTables works too).
        Default: built on the host from the scale table and from the prior parameters in the decoder's weights."""
        self.dec = decoder
        self.L, self.ctx, self.device = decoder.L, decoder.ctx, decoder.device
        if not self.L.cdc_has_codec(self.ctx):
            raise RuntimeError("the decoder was created without the codec.* weights")
        self.gauss = DeviceTables(gauss_tables if gauss_tables is not None else entropy_tables.gaussian_tables(), self.device)
        self.fact = DeviceTables(fact_tables, self.device) if fact_tables is not None else None
        c = decoder.cfg.latent_ch
        self.median = (torch.zeros(c) if median is None else median.detach().float()).to(self.device)
        # the same tables in the library, for cdc_compress_rgb8 / cdc_decompress_rgb8
        self._set_tables(0, gauss_tables if gauss_tables is not None else entropy_tables.gaussian_tables())
        if fact_tables is not None:
            self._set_tables(1, fact_tables, self.median.cpu().contiguous())

    def _set_tables(self, which, tables, median=None):
        i32 = [torch.as_tensor(getattr(tables, f)).cpu().to(torch.int32).contiguous() for f in ("cdf", "row_start", "cdf_length", "offset")]
        scale = torch.as_tensor(tables.scale_table).cpu().to(torch.float32).contiguous() if which == 0 else None
        ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)
        cdf, row_start, cdf_length, offset = i32
        self._ck(self.L.cdc_set_entropy_tables(self.ctx, which, ptr(cdf), cdf.numel(), ptr(row_start), ptr(cdf_length), ptr(offset),
                                               row_start.numel(), ptr(scale), ptr(median)), "cdc_set_entropy_tables")

    @staticmethod
    def prior_tables(weights, prefix="codec.prior."):
        """Factorised-prior CDF tables from the prior's parameters in a weight dict (host, float64)."""
        n = 1 + max(int(k[len(prefix) + 5:].split(".")[0]) for k in weights if k.startswith(prefix + "mats."))
        g = lambda name, i: weights[f"{prefix}{name}.{i}"].detach().double().cpu().numpy()
        return entropy_tables.factorized_tables([g("mats", i) for i in range(n)], [g("biases", i) for i in range(n)],
                                                [g("factors", i) for i in range(n - 1)],
                                                weights[prefix + "median"].detach().double().cpu().numpy())

    def _ck(self, rc, what):
        self.dec._ck(rc, what)

    # ---- the three networks ---------------------------------------------------------------------
    @torch.no_grad()
    def analysis(self, img01):
        """y = encoder(2 * img - 1): [B,3,H,W] in [0,1] -> [B,latent_ch,H/16,W/16] fp32 (device)."""
        if img01.dim() != 4 or img01.shape[1] != 3 or img01.shape[2] % 64 or img01.shape[3] % 64:
            raise ValueError(f"img must be [B,3,H,W] with H, W multiples of 64, got {tuple(img01.shape)}")
        B, _, H, W = img01.shape
        with torch.cuda.device(self.device):
            x = _f32c(img01, self.device)
            self.dec.bind(B, H, W)
            y = torch.empty(B, self.dec.cfg.latent_ch, H // 16, W // 16, device=self.device, dtype=torch.float32)
            self._ck(self.L.cdc_encode_analysis(self.ctx, C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()), _stream_ptr()),
                     "cdc_encode_analysis")
        return y

    def _bind_for_latent(self, t, div):
        B, c, h, w = t.shape
        if c != self.dec.cfg.latent_ch:
            raise ValueError(f"expected {self.dec.cfg.latent_ch} channels, got {c}")
        self.dec.bind(B, h * div, w * div)
        return B, h, w

    @torch.no_grad()
    def hyper_encode(self, y):
        with torch.cuda.device(self.device):
            yd = _f32c(y, self.device)
            B, h, w = self._bind_for_latent(yd, 16)
            z = torch.empty(B, yd.shape[1], h // 4, w // 4, device=self.device, dtype=torch.float32)
            self._ck(self.L.cdc_hyper_encode(self.ctx, C.c_void_p(yd.data_ptr()), C.c_void_p(z.data_ptr()), _stream_ptr()),
                     "cdc_hyper_encode")
        return z

    @torch.no_grad()
    def hyper_decode(self, z_hat):
        with torch.cuda.device(self.device):
            zd = _f32c(z_hat, self.device)
            B, h, w = self._bind_for_latent(zd, 64)
            mu = torch.empty(B, zd.shape[1], h * 4, w * 4, device=self.device, dtype=torch.float32)
            sigma = torch.empty_like(mu)
            self._ck(self.L.cdc_hyper_decode(self.ctx, C.c_void_p(zd.data_ptr()), C.c_void_p(mu.data_ptr()),
                                             C.c_void_p(sigma.data_ptr()), _stream_ptr()), "cdc_hyper_decode")
        return mu, sigma

    # ---- oracle Codec.encode ----------------------------------------------------------------------
    @torch.no_grad()
    def encode(self, img01):
        """img in [0,1] -> dict with y, z, mu, sigma, q (int32), y_hat, qz, z_hat and the entropy-coder symbols
        y_sym / z_sym = (idx, v, lo, hi, raw), everything on the device."""
        y = self.analysis(img01)
        z = self.hyper_encode(y)
        qz, z_hat = quantize_symbols(z, self.median, device=self.device, per_channel=True)
        z_sym = cdf_lookup(qz, None, self.fact, device=self.device) if self.fact is not None else None
        mu, sigma = self.hyper_decode(z_hat)
        q, y_hat = quantize_symbols(y, mu, device=self.device)
        y_sym = cdf_lookup(q, sigma, self.gauss, device=self.device)
        return dict(y=y, z=z, mu=mu, sigma=sigma, q=q, y_hat=y_hat, qz=qz, z_hat=z_hat, y_sym=y_sym, z_sym=z_sym)

    # ---- decoder side -----------------------------------------------------------------------------
    @torch.no_grad()
    def latent_from_symbols(self, qz, q):
        """(qz, q) int32 -> (y_hat, mu, sigma): z_hat = qz + median; (mu, sigma) = hyper_dec(z_hat); y_hat = q + mu."""
        z_hat = qz.to(self.device).float() + self.median[None, :, None, None]
        mu, sigma = self.hyper_decode(z_hat)
        return q.to(self.device).float() + mu, mu, sigma

    @torch.no_grad()
    def decompress(self, qz, q, steps, **kw):
        y_hat, _, _ = self.latent_from_symbols(qz, q)
        return self.dec.decode(y_hat, steps, **kw)

    # ---- bitstream (row f3): "CDC5" | u32 B, H, W | u64 len(z stream) | z container | y container ------------------
    @torch.no_grad()
    def compress(self, img01):
        """img in [0,1] -> (bytes, enc): the on-wire representation (two CDCR rANS containers: z, then y) and the encode
        dict.  Needs the factorised-prior tables (fact_tables)."""
        import struct
        from .bitstream import rans_encode
        if self.fact is None:
            raise RuntimeError("compress needs the factorised-prior CDF tables (fact_tables)")
        enc = self.encode(img01)
        B, c, h, w = enc["q"].shape
        zs = rans_encode(enc["z_sym"], self.fact, B * c, (h // 4) * (w // 4), self.device)
        ys = rans_encode(enc["y_sym"], self.gauss, B * c, h * w, self.device)
        head = b"CDC5" + struct.pack("<3IQ", B, h * 16, w * 16, zs.numel())
        return head + zs.cpu().numpy().tobytes() + ys.cpu().numpy().tobytes(), enc

    @torch.no_grad()
    def decode_symbols(self, data: bytes):
        """bytes -> (qz, q) int32 device tensors: the decoder side of the entropy stage.  z is decoded with the
        channel-indexed tables; its hyper-decoder output gives the CDF row of every y symbol."""
        import struct
        from .bitstream import rans_decode
        if data[:4] != b"CDC5":
            raise ValueError("not a CDC5 stream")
        B, H, W, nz = struct.unpack_from("<3IQ", data, 4)
        c, h, w = self.dec.cfg.latent_ch, H // 16, W // 16
        zbytes, ybytes = data[24:24 + nz], data[24 + nz:]
        ch = torch.arange(c, dtype=torch.int32, device=self.device)[None, :, None, None].expand(B, c, h // 4, w // 4)
        qz = rans_decode(zbytes, ch.contiguous(), self.fact, self.device).reshape(B, c, h // 4, w // 4)
        z_hat = qz.float() + self.median[None, :, None, None]
        _, sigma = self.hyper_decode(z_hat)
        idx = cdf_lookup(torch.zeros(B, c, h, w, dtype=torch.int32, device=self.device), sigma, self.gauss, device=self.device)[0]
        q = rans_decode(ybytes, idx, self.gauss, self.device).reshape(B, c, h, w)
        return qz, q

    @torch.no_grad()
    def decompress_bytes(self, data: bytes, steps, **kw):
        qz, q = self.decode_symbols(data)
        return self.decompress(qz, q, steps, **kw)

    # ---- the same two directions in one library call each, 8-bit RGB at the boundary ----------------------------------
    @torch.no_grad()
    def compress_rgb8(self, img):
        """uint8 CPU tensor [B,H,W,3] (interleaved RGB, H and W multiples of 64) -> the CDC5 stream as bytes, equal to
        compress(img.permute(0, 3, 1, 2).float() / 255)[0] (include/cdc_b200.h cdc_compress_rgb8)."""
        if not isinstance(img, torch.Tensor) or img.dtype != torch.uint8 or img.is_cuda or img.dim() != 4 or img.shape[3] != 3 \
                or img.shape[0] < 1 or img.shape[1] < 64 or img.shape[2] < 64 or img.shape[1] % 64 or img.shape[2] % 64:
            raise ValueError("img must be a uint8 CPU tensor [B,H,W,3] with H, W multiples of 64, got "
                             f"{getattr(img, 'dtype', type(img))} {tuple(getattr(img, 'shape', ()))}")
        if self.fact is None:
            raise RuntimeError("compress_rgb8 needs the factorised-prior CDF tables (fact_tables)")
        B, H, W, _ = img.shape
        x = img.contiguous()
        with torch.cuda.device(self.device):
            self.dec.bind(B, H, W)
            cap = self.L.cdc_compress_max_bytes(self.ctx)
            if cap < 0:
                self._ck(cap, "cdc_compress_max_bytes")
            out = torch.empty(cap, dtype=torch.uint8)
            n = C.c_int64(0)
            self._ck(self.L.cdc_compress_rgb8(self.ctx, C.c_void_p(x.data_ptr()), C.c_void_p(out.data_ptr()), cap, C.byref(n),
                                              self.dec._stream()), "cdc_compress_rgb8")
        return out[:n.value].numpy().tobytes()

    @staticmethod
    def stream_info(data):
        """(B, H, W) of a CDC5 stream, from the host alone (cdc_stream_info); ValueError if it is malformed."""
        buf = bytes(data)
        B, H, W = C.c_int(), C.c_int(), C.c_int()
        if _ffi.lib().cdc_stream_info(buf, len(buf), C.byref(B), C.byref(H), C.byref(W)) != 0:
            raise ValueError("not a valid CDC5 stream")
        return B.value, H.value, W.value

    @torch.no_grad()
    def decompress_rgb8(self, data, steps, *, seeds, gamma=0.8):
        """CDC5 bytes -> uint8 CPU tensor [B,H,W,3]: the decode of the stream's latent in `steps` steps with x_T = gamma * z
        from the per-image seeds, round_half_even(255 * image), in one library call (cdc_decompress_rgb8).  Equal to
        (decompress_bytes(data, steps, seeds=seeds, gamma=gamma) * 255).round() in uint8 NHWC.  ValueError if the bytes
        are not a valid stream for this codec."""
        if self.fact is None:
            raise RuntimeError("decompress_rgb8 needs the factorised-prior CDF tables (fact_tables)")
        buf = bytes(data)
        B, H, W = self.stream_info(buf)
        _seed_values(seeds, B)
        with torch.cuda.device(self.device):
            self.dec.bind(B, H, W)
            if steps != self.dec.steps:
                self.dec.set_sample_schedule(steps, *self.dec.sampler)
            self.dec.set_image_seeds(seeds)
            out = torch.empty(B, H, W, 3, dtype=torch.uint8)
            rc = self.L.cdc_decompress_rgb8(self.ctx, buf, len(buf), float(gamma), C.c_void_p(out.data_ptr()), self.dec._stream())
            if rc == _ffi.ERR_DATA:
                raise ValueError(f"corrupt CDC5 stream: {self.L.cdc_last_error(self.ctx).decode()}")
            self._ck(rc, "cdc_decompress_rgb8")
        return out
