"""Host-side mirror of the oracle's decoder interface over the C ABI.

Same surface as oracle/sampler.py OracleDecoder (the reference ships no code, so the oracle
*is* the reference interface for this path; SURVEY.md section 8b):
    set_sample_schedule(steps), predict_x0(x_t, t, cond), denoise_step(x_t, t, cond),
    decode(latent, steps, *, init=None, gamma=0.8, seed=0), quantize_symbols, cdf_lookup.
Tensors at this surface are NCHW fp32 torch tensors; CUDA tensors are used in place, CPU tensors
are staged through pinned memory by the library (cdc_decode_host).
"""
import ctypes as C

import torch

from . import _ffi
from .config import CDCConfig


def _stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t, dev):
    return t.to(device=dev, dtype=torch.float32).contiguous()


class Decoder:
    def __init__(self, cfg: CDCConfig, weights, device="cuda:0", tables=None, variant="product"):
        """weights: dict name -> tensor (oracle UNet.state_dict(); optional 'context.*' entries from
        oracle ContextNet.state_dict()) or a path to a safetensors file holding the same.
        variant: which build of the library to bind ("product"; "bf16" / "tools" exist for tests and tools)."""
        if not torch.cuda.is_available():
            raise RuntimeError("cdc_b200.Decoder needs a CUDA device (sm_100a); there is no CPU fallback")
        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("cdc_b200.Decoder needs a CUDA device (sm_100a); there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.L = _ffi.lib(variant)
        if isinstance(weights, str):
            from safetensors.torch import load_file
            weights = load_file(weights)
        cc = _ffi.CdcConfig(cfg.base, (C.c_int32 * 4)(*cfg.mults), cfg.groups, cfg.heads, cfg.head_dim, cfg.temb,
                            cfg.T, cfg.latent_ch, cfg.gn_eps)
        self.ctx = C.c_void_p()
        rc = self.L.cdc_create(C.byref(cc), self.device.index, C.byref(self.ctx))
        if rc != 0:
            raise RuntimeError(f"cdc_create failed ({rc}): {self.L.cdc_last_error(None).decode()}")
        with torch.cuda.device(self.device):
            for name, t in weights.items():
                d = _f32c(t.detach(), self.device)
                shape = (C.c_int64 * d.dim())(*d.shape)
                self._ck(self.L.cdc_load_weights(self.ctx, name.encode(), C.c_void_p(d.data_ptr()), shape, d.dim()),
                         f"cdc_load_weights({name})")
            self._ck(self.L.cdc_finalize_weights(self.ctx), "cdc_finalize_weights")
        self.has_context_net = bool(self.L.cdc_has_context_net(self.ctx))
        self.tables = tables
        self.steps = 0
        self.sampler = (0.0, "x", 0)
        self.shape = None

    def _ck(self, rc, what):
        _ffi.check(self.ctx, rc, what, self.L)

    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.L.cdc_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    # ---- schedule ------------------------------------------------------------------------------
    def set_sample_schedule(self, steps: int, eta: float = 0.0, pred: str = "x", seed: int = 0):
        """oracle/sampler.py OracleDecoder.set_sample_schedule.  eta > 0: stochastic DDIM; pred = "eps": the network
        predicts the noise (SURVEY.md section 8 row f4)."""
        if pred not in ("x", "eps"):
            raise ValueError("pred must be 'x' or 'eps'")
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_set_sampler(self.ctx, 1 if pred == "eps" else 0, float(eta), int(seed)), "cdc_set_sampler")
            self._ck(self.L.cdc_set_schedule(self.ctx, int(steps)), "cdc_set_schedule")
        self.steps = int(steps)
        self.sampler = (float(eta), pred, int(seed))
        self.idx = [self.L.cdc_schedule_index(self.ctx, k) for k in range(self.steps)]
        return self.idx

    def coeffs(self, k):
        a, b = C.c_float(), C.c_float()
        self._ck(self.L.cdc_schedule_coeffs(self.ctx, k, C.byref(a), C.byref(b)), "cdc_schedule_coeffs")
        return a.value, b.value

    def coeffs5(self, k):
        v = [C.c_float() for _ in range(5)]
        self._ck(self.L.cdc_schedule_coeffs5(self.ctx, k, *[C.byref(x) for x in v]), "cdc_schedule_coeffs5")
        return tuple(x.value for x in v)

    def film_table(self):
        """[steps, film_size] fp32: the (scale | shift) vectors of the 18 ResBlocks for every step of the schedule."""
        if not self.steps:
            raise RuntimeError("call set_sample_schedule first")
        n = self.L.cdc_film_size(self.ctx)
        out = torch.empty(self.steps, n, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_film(self.ctx, C.c_void_p(out.data_ptr()), _stream_ptr()), "cdc_get_film")
        return out

    def _k_of(self, t):
        if not self.steps:
            raise RuntimeError("call set_sample_schedule first")
        if int(t) not in self.idx:
            raise ValueError(f"t={t} is not in the active {self.steps}-step schedule")
        return self.idx.index(int(t))

    # ---- binding -------------------------------------------------------------------------------
    def set_plan_option(self, option: int, value: int):
        """A/B of a planner decision (include/cdc_b200_tools.h cdc_plan_option); re-plans at the next bind."""
        self._ck(self.L.cdc_set_plan_option(self.ctx, int(option), int(value)), "cdc_set_plan_option")
        self.shape = None

    def bind(self, B, H, W):
        if self.shape != (B, H, W):
            with torch.cuda.device(self.device):
                self._ck(self.L.cdc_bind_io(self.ctx, B, H, W), "cdc_bind_io")
            self.shape = (B, H, W)

    def cond_shapes(self, B, H, W):
        return [(B, c, H >> i, W >> i) for i, c in enumerate(self.cfg.channels)]

    def set_cond(self, cond):
        if len(cond) != 4 or cond[0].dim() != 4:
            raise ValueError("cond must be 4 NCHW tensors (c0, c1, c2, c3)")
        B, _, H, W = cond[0].shape
        want = self.cond_shapes(B, H, W)
        for i, t in enumerate(cond):
            if tuple(t.shape) != want[i]:
                raise ValueError(f"cond[{i}] has shape {tuple(t.shape)}, expected {want[i]}")
        with torch.cuda.device(self.device):
            c = [_f32c(t, self.device) for t in cond]
            self.bind(B, H, W)
            self._ck(self.L.cdc_set_cond(self.ctx, *[C.c_void_p(t.data_ptr()) for t in c], _stream_ptr()), "cdc_set_cond")

    def set_latent(self, latent):
        if latent.dim() != 4 or latent.shape[1] != self.cfg.latent_ch:
            raise ValueError(f"latent must be [B, {self.cfg.latent_ch}, H/16, W/16], got {tuple(latent.shape)}")
        B, _, h, w = latent.shape
        with torch.cuda.device(self.device):
            y = _f32c(latent, self.device)
            self.bind(B, h * 16, w * 16)
            self._ck(self.L.cdc_set_latent(self.ctx, C.c_void_p(y.data_ptr()), _stream_ptr()), "cdc_set_latent")

    def get_cond(self):
        """The bound context maps (c0, c1, c2, c3) as NCHW fp32 tensors: what set_latent's context net produced
        (oracle/codec.py ContextNet.forward) or what set_cond stored, after the 16-bit storage rounding."""
        if self.shape is None:
            raise RuntimeError("nothing bound: call set_latent / set_cond first")
        outs = [torch.empty(s, device=self.device, dtype=torch.float32) for s in self.cond_shapes(*self.shape)]
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_cond(self.ctx, *[C.c_void_p(t.data_ptr()) for t in outs], _stream_ptr()), "cdc_get_cond")
        return tuple(outs)

    def _set_x(self, x):
        if self.shape is None:
            raise RuntimeError("nothing bound: call set_latent / set_cond first")
        B, H, W = self.shape
        if tuple(x.shape) != (B, 3, H, W):
            raise ValueError(f"x has shape {tuple(x.shape)}, expected {(B, 3, H, W)} (the bound batch / image size)")
        with torch.cuda.device(self.device):
            xd = _f32c(x, self.device)
            self._ck(self.L.cdc_set_x(self.ctx, C.c_void_p(xd.data_ptr()), _stream_ptr()), "cdc_set_x")

    def _get_x(self, to_image=False):
        B, H, W = self.shape
        out = torch.empty(B, 3, H, W, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_x(self.ctx, C.c_void_p(out.data_ptr()), 1 if to_image else 0, _stream_ptr()), "cdc_get_x")
        return out

    def _get_x0(self):
        B, H, W = self.shape
        out = torch.empty(B, 3, H, W, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_x0(self.ctx, C.c_void_p(out.data_ptr()), _stream_ptr()), "cdc_get_x0")
        return out

    # ---- the hot path --------------------------------------------------------------------------
    @torch.no_grad()
    def denoise_step(self, x_t, t, cond=None):
        """x_prev = c0_k * clamp(x0_hat) + c1_k * x_t (+ sigma_k z), x0_hat from unet(x_t, t, cond).  cond=None reuses the bound cond."""
        k = self._k_of(t)
        with torch.cuda.device(self.device):
            if cond is not None:
                self.set_cond(cond)
            self._set_x(x_t)
            self._ck(self.L.cdc_denoise_step(self.ctx, k, _stream_ptr()), "cdc_denoise_step")
            return self._get_x()

    @torch.no_grad()
    def predict_x0(self, x_t, t, cond=None):
        self.denoise_step(x_t, t, cond)
        return self._get_x0()

    @torch.no_grad()
    def decode(self, latent, steps, *, init=None, gamma=0.8, seed=0, cond=None, out=None):
        """latent y_hat fp32 [B,256,H/16,W/16] -> image fp32 [B,3,H,W] in [0,1] (K steps = one graph launch).
        Host tensors take the cdc_decode_host path (H2D + decode + D2H inside the library); page-locked inputs and a
        page-locked `out` (optional, host path only: fp32 [B,3,H,W], returned) are copied from / to directly."""
        if steps != self.steps:
            self.set_sample_schedule(steps, *self.sampler)
        if latent.dim() != 4 or latent.shape[1] != self.cfg.latent_ch:
            raise ValueError(f"latent must be [B, {self.cfg.latent_ch}, H/16, W/16], got {tuple(latent.shape)}")
        B, _, h, w = latent.shape
        H, W = h * 16, w * 16
        if init is None:
            g = torch.Generator().manual_seed(seed)
            init = gamma * torch.randn(B, 3, H, W, generator=g)
        elif tuple(init.shape) != (B, 3, H, W):
            raise ValueError(f"init has shape {tuple(init.shape)}, expected {(B, 3, H, W)}")
        with torch.cuda.device(self.device):
            self.bind(B, H, W)
            if cond is None and not latent.is_cuda and not init.is_cuda:
                # host buffers: pinned staging + H2D/D2H inside the library
                lat = latent.float().contiguous()
                x0 = init.float().contiguous()
                if out is None:
                    out = torch.empty(B, 3, H, W, dtype=torch.float32)
                elif out.shape != (B, 3, H, W) or out.dtype != torch.float32 or out.is_cuda or not out.is_contiguous():
                    raise ValueError("out must be a contiguous fp32 host tensor of shape [B,3,H,W]")
                self._ck(self.L.cdc_decode_host(self.ctx, C.c_void_p(lat.data_ptr()), C.c_void_p(x0.data_ptr()),
                                                C.c_void_p(out.data_ptr()), _stream_ptr()), "cdc_decode_host")
                return out
            if cond is not None:
                self.set_cond(cond)
            else:
                self.set_latent(latent)
            self._set_x(init)
            self._ck(self.L.cdc_decode(self.ctx, _stream_ptr()), "cdc_decode")
            return self._get_x(to_image=True)

    def decode_resident(self):
        """Replay the K-step graph on whatever x / cond are bound (used by bench.py's device-timed leg)."""
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_decode(self.ctx, _stream_ptr()), "cdc_decode")

    # ---- introspection -------------------------------------------------------------------------
    def launches_per_step(self):
        return self.L.cdc_launches_per_step(self.ctx)

    def flops_per_step(self):
        return self.L.cdc_flops_per_step(self.ctx)

    def saturation_count(self, reset=False):
        """Epilogue passes that stored a value saturated to the fp16 range since creation / the last reset (0 = none)."""
        n = C.c_uint64(0)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_saturation_count(self.ctx, C.byref(n), 1 if reset else 0, _stream_ptr()), "cdc_saturation_count")
        return int(n.value)

    def step_ops(self):
        n = self.L.cdc_num_step_ops(self.ctx)
        return [(self.L.cdc_step_op_name(self.ctx, i).decode(), self.L.cdc_step_op_flops(self.ctx, i),
                 self.L.cdc_step_op_bytes(self.ctx, i)) for i in range(n)]

    def step_op_desc(self, i):
        """_ffi.StepOpDesc of step op i of the bound plan (include/cdc_b200_tools.h cdc_step_op_describe)."""
        d = _ffi.StepOpDesc()
        self._ck(self.L.cdc_step_op_describe(self.ctx, i, C.byref(d)), "cdc_step_op_describe")
        return d

    def run_step_op(self, i, k=0):
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_run_step_op(self.ctx, i, k, _stream_ptr()), "cdc_run_step_op")

    def profile_step(self, k=0, warm=1):
        """In-stream device time (us) of every op of step k (launched back to back, CUDA events in the library)."""
        n = self.L.cdc_num_step_ops(self.ctx)
        buf = (C.c_float * n)()
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_profile_step(self.ctx, k, warm, buf, _stream_ptr()), "cdc_profile_step")
        return list(buf)

    def profile_graph(self, reps=5):
        """In-graph timing of the captured K-step loop: (start_us, dur_us), each [steps][ops] (median over `reps`
        replays), from per-kernel globaltimer stamps (include/cdc_b200_tools.h cdc_profile_graph)."""
        n = self.L.cdc_num_step_ops(self.ctx)
        st = (C.c_float * (n * self.steps))()
        du = (C.c_float * (n * self.steps))()
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_profile_graph(self.ctx, reps, st, du, _stream_ptr()), "cdc_profile_graph")
        rs = [[st[k * n + i] for i in range(n)] for k in range(self.steps)]
        rd = [[du[k * n + i] for i in range(n)] for k in range(self.steps)]
        return rs, rd

    # ---- integer path (same names as the oracle) -----------------------------------------------
    def quantize_symbols(self, y, mu):
        return quantize_symbols(y, mu, device=self.device)

    def cdf_lookup(self, q, sigma):
        return cdf_lookup(q, sigma, self.tables, device=self.device)


def quantize_symbols(y, mu, device="cuda:0", per_channel=False):
    """q = rint(y - mu) int32 (half-to-even), y_hat = q + mu.  per_channel: mu is a [C] vector for NCHW y."""
    L = _ffi.lib()
    dev = torch.device(device)
    yd = _f32c(y, dev)
    md = _f32c(mu, dev)
    q = torch.empty(yd.shape, dtype=torch.int32, device=dev)
    yh = torch.empty_like(yd)
    n = yd.numel()
    inner, mod = 0, 0
    if per_channel:
        mod = yd.shape[1]
        inner = yd[0, 0].numel()
    elif md.numel() != n:
        raise ValueError("mu must match y elementwise (or pass per_channel=True)")
    with torch.cuda.device(dev):
        rc = L.cdc_quantize(C.c_void_p(yd.data_ptr()), C.c_void_p(md.data_ptr()), C.c_void_p(q.data_ptr()),
                            C.c_void_p(yh.data_ptr()), n, inner, mod, _stream_ptr())
    if rc:
        raise RuntimeError(f"cdc_quantize failed ({rc})")
    return q, yh


class DeviceTables:
    """CDF tables (oracle/entropy.py CDFTables layout) resident on the device."""

    def __init__(self, tables, device="cuda:0"):
        dev = torch.device(device)
        self.cdf = torch.as_tensor(tables.cdf, dtype=torch.int32).to(dev)
        self.row_start = torch.as_tensor(tables.row_start, dtype=torch.int32).to(dev)
        self.cdf_length = torch.as_tensor(tables.cdf_length, dtype=torch.int32).to(dev)
        self.offset = torch.as_tensor(tables.offset, dtype=torch.int32).to(dev)
        self.scale_table = torch.as_tensor(tables.scale_table, dtype=torch.float32).to(dev)
        self.rows = int(self.row_start.numel())


def cdf_lookup(q, sigma, tables, device="cuda:0"):
    """(idx, v, lo, hi, raw) int32.  sigma=None: idx = channel of an NCHW q (factorised prior)."""
    L = _ffi.lib()
    dev = torch.device(device)
    if not isinstance(tables, DeviceTables):
        tables = DeviceTables(tables, dev)
    qd = q.to(device=dev, dtype=torch.int32).contiguous()
    n = qd.numel()
    outs = [torch.empty(qd.shape, dtype=torch.int32, device=dev) for _ in range(5)]
    inner = 1
    sp = C.c_void_p(0)
    sd = None
    if sigma is not None:
        sd = _f32c(sigma, dev)
        sp = C.c_void_p(sd.data_ptr())
    else:
        inner = qd[0, 0].numel()
    with torch.cuda.device(dev):
        rc = L.cdc_cdf_lookup(C.c_void_p(qd.data_ptr()), sp, C.c_void_p(tables.cdf.data_ptr()),
                              C.c_void_p(tables.row_start.data_ptr()), C.c_void_p(tables.cdf_length.data_ptr()),
                              C.c_void_p(tables.offset.data_ptr()),
                              C.c_void_p(tables.scale_table.data_ptr()) if sigma is not None else C.c_void_p(0),
                              tables.rows, inner, *[C.c_void_p(o.data_ptr()) for o in outs], n, _stream_ptr())
    if rc:
        raise RuntimeError(f"cdc_cdf_lookup failed ({rc})")
    return tuple(outs)
