"""Host-side mirror of the oracle's decoder interface over the C ABI.

Same surface as oracle/sampler.py OracleDecoder (the reference ships no code, so the oracle
*is* the reference interface for this path; SURVEY.md section 8b):
    set_sample_schedule(steps), predict_x0(x_t, t, cond), denoise_step(x_t, t, cond),
    decode(latent, steps, *, init=None, gamma=0.8, seed=0, trajectory=None), quantize_symbols, cdf_lookup;
plus decode_progressive, a generator of per-step (x_t, x0_hat) previews while the decode runs, and per-image seeds
(decode(..., seeds=[...]) / set_image_seeds): image b's x_T and sampler noise then depend on seeds[b] alone, so an image
decodes to the same result in any batch -- bit for bit with Decoder(..., batch_invariant=True).
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


def _seed_values(seeds, n):
    """seeds (a sequence of ints, or an int64 / uint64 tensor) -> list of n ints in [0, 2^64); ValueError otherwise."""
    if isinstance(seeds, torch.Tensor):
        if seeds.dtype not in (torch.int64, torch.uint64) or seeds.dim() != 1:
            raise ValueError(f"seeds must be a 1-D int64 / uint64 tensor, got {seeds.dtype} of shape {tuple(seeds.shape)}")
        vals = seeds.cpu().tolist()
    else:
        vals = list(seeds)
    if len(vals) != n:
        raise ValueError(f"{len(vals)} seeds for a batch of {n}: give one per image")
    for v in vals:
        if isinstance(v, bool) or not hasattr(v, "__index__"):
            raise ValueError(f"seed {v!r} is not an integer")
        if not 0 <= int(v) < 1 << 64:
            raise ValueError(f"seed {int(v)} is outside [0, 2^64)")
    return [int(v) for v in vals]


class Decoder:
    def __init__(self, cfg: CDCConfig, weights, device="cuda:0", tables=None, variant="product", batch_invariant=False):
        """weights: dict name -> tensor (oracle UNet.state_dict(); optional 'context.*' entries from
        oracle ContextNet.state_dict()) or a path to a safetensors file holding the same.
        variant: which build of the library to bind ("product"; "bf16" / "tools" exist for tests and tools).
        batch_invariant: plan every batch per image as for a batch of 1 (include/cdc_b200.h cdc_set_batch_invariant), so
        that with per-image seeds an image decodes -- and, through a Codec on this decoder, encodes -- to the same bits
        alone, in any batch and in any shard of a multi-GPU run; at batch 1 the plan is the default one."""
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
        self.batch_invariant = bool(batch_invariant)
        self._ck(self.L.cdc_set_batch_invariant(self.ctx, 1 if self.batch_invariant else 0), "cdc_set_batch_invariant")
        self.has_context_net = bool(self.L.cdc_has_context_net(self.ctx))
        self.tables = tables
        self.steps = 0
        self.sampler = (0.0, "x", 0)
        self.shape = None
        self._side = None  # decode_progressive's stream
        self._side_busy = False  # a decode_progressive generator has not ended: its graph may still run on _side

    def _ck(self, rc, what):
        _ffi.check(self.ctx, rc, what, self.L)

    def _stream(self):
        """The stream handle every call of this decoder enqueues on: the current stream, made to wait for the graph of
        an unfinished decode_progressive first (it reads and writes the same workspace)."""
        cur = torch.cuda.current_stream()
        if self._side_busy and cur != self._side:
            cur.wait_stream(self._side)
        return C.c_void_p(cur.cuda_stream)

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
            self._ck(self.L.cdc_get_film(self.ctx, C.c_void_p(out.data_ptr()), self._stream()), "cdc_get_film")
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
            self.shape = None  # (a refused bind leaves nothing bound)
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
            self._ck(self.L.cdc_set_cond(self.ctx, *[C.c_void_p(t.data_ptr()) for t in c], self._stream()), "cdc_set_cond")

    def set_latent(self, latent):
        if latent.dim() != 4 or latent.shape[1] != self.cfg.latent_ch:
            raise ValueError(f"latent must be [B, {self.cfg.latent_ch}, H/16, W/16], got {tuple(latent.shape)}")
        B, _, h, w = latent.shape
        with torch.cuda.device(self.device):
            y = _f32c(latent, self.device)
            self.bind(B, h * 16, w * 16)
            self._ck(self.L.cdc_set_latent(self.ctx, C.c_void_p(y.data_ptr()), self._stream()), "cdc_set_latent")

    def get_cond(self):
        """The bound context maps (c0, c1, c2, c3) as NCHW fp32 tensors: what set_latent's context net produced
        (oracle/codec.py ContextNet.forward) or what set_cond stored, after the 16-bit storage rounding."""
        if self.shape is None:
            raise RuntimeError("nothing bound: call set_latent / set_cond first")
        outs = [torch.empty(s, device=self.device, dtype=torch.float32) for s in self.cond_shapes(*self.shape)]
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_cond(self.ctx, *[C.c_void_p(t.data_ptr()) for t in outs], self._stream()), "cdc_get_cond")
        return tuple(outs)

    def _set_x(self, x):
        if self.shape is None:
            raise RuntimeError("nothing bound: call set_latent / set_cond first")
        B, H, W = self.shape
        if tuple(x.shape) != (B, 3, H, W):
            raise ValueError(f"x has shape {tuple(x.shape)}, expected {(B, 3, H, W)} (the bound batch / image size)")
        with torch.cuda.device(self.device):
            xd = _f32c(x, self.device)
            self._ck(self.L.cdc_set_x(self.ctx, C.c_void_p(xd.data_ptr()), self._stream()), "cdc_set_x")

    def _get_x(self, to_image=False):
        B, H, W = self.shape
        out = torch.empty(B, 3, H, W, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_x(self.ctx, C.c_void_p(out.data_ptr()), 1 if to_image else 0, self._stream()), "cdc_get_x")
        return out

    def _get_x0(self):
        B, H, W = self.shape
        out = torch.empty(B, 3, H, W, device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_get_x0(self.ctx, C.c_void_p(out.data_ptr()), self._stream()), "cdc_get_x0")
        return out

    def set_image_seeds(self, seeds):
        """Per-image noise for the bound batch (include/cdc_b200.h cdc_set_image_seeds): seeds[b] keys image b's x_T
        (init_noise) and its sampler noise at eta > 0, at the pixel's index within the image.  None turns the mode off:
        the batch-wide seed of set_sample_schedule applies again.  denoise_step / predict_x0 / decode_resident use
        whatever is bound; a bind to another shape turns the mode off."""
        if self.shape is None:
            raise RuntimeError("nothing bound: call set_latent / set_cond first")
        vals = [] if seeds is None else _seed_values(seeds, self.shape[0])
        arr = (C.c_uint64 * max(len(vals), 1))(*vals)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_set_image_seeds(self.ctx, arr, len(vals), self._stream()), "cdc_set_image_seeds")

    def init_noise(self, gamma=0.8):
        """x_T = gamma * z from the bound per-image seeds, written into the sampler state on the device."""
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_init_noise(self.ctx, float(gamma), self._stream()), "cdc_init_noise")

    # ---- the hot path --------------------------------------------------------------------------
    @torch.no_grad()
    def denoise_step(self, x_t, t, cond=None):
        """x_prev = c0_k * clamp(x0_hat) + c1_k * x_t (+ sigma_k z), x0_hat from unet(x_t, t, cond).  cond=None reuses the bound cond."""
        k = self._k_of(t)
        with torch.cuda.device(self.device):
            if cond is not None:
                self.set_cond(cond)
            self._set_x(x_t)
            self._ck(self.L.cdc_denoise_step(self.ctx, k, self._stream()), "cdc_denoise_step")
            return self._get_x()

    @torch.no_grad()
    def predict_x0(self, x_t, t, cond=None):
        self.denoise_step(x_t, t, cond)
        return self._get_x0()

    def _decode_inputs(self, latent, steps, init, gamma, seed, seeds=None):
        """Schedule, shape checks and the default x_T shared by decode and decode_progressive.  With per-image seeds
        x_T is drawn on the device later (init stays None); the seeds are checked here, before anything is bound."""
        if steps != self.steps:
            self.set_sample_schedule(steps, *self.sampler)
        if latent.dim() != 4 or latent.shape[1] != self.cfg.latent_ch:
            raise ValueError(f"latent must be [B, {self.cfg.latent_ch}, H/16, W/16], got {tuple(latent.shape)}")
        B, _, h, w = latent.shape
        H, W = h * 16, w * 16
        if seeds is not None:
            if init is not None:
                raise ValueError("give init or seeds, not both")
            _seed_values(seeds, B)
        elif init is None:
            g = torch.Generator().manual_seed(seed)
            init = gamma * torch.randn(B, 3, H, W, generator=g)
        elif tuple(init.shape) != (B, 3, H, W):
            raise ValueError(f"init has shape {tuple(init.shape)}, expected {(B, 3, H, W)}")
        return init, (B, H, W)

    @staticmethod
    def _check_host_out(out, B, H, W):
        if out is None:
            return torch.empty(B, 3, H, W, dtype=torch.float32)
        if out.shape != (B, 3, H, W) or out.dtype != torch.float32 or out.is_cuda or not out.is_contiguous():
            raise ValueError("out must be a contiguous fp32 host tensor of shape [B,3,H,W]")
        return out

    def _bind_x(self, init, seeds, gamma):
        """x_T into the sampler state: init copied in, or drawn on the device from the per-image seeds."""
        if seeds is None:
            self._set_x(init)
        else:
            self.init_noise(gamma)

    @torch.no_grad()
    def decode(self, latent, steps, *, init=None, gamma=0.8, seed=0, seeds=None, cond=None, out=None, trajectory=None,
               x0_trajectory=None):
        """latent y_hat fp32 [B,256,H/16,W/16] -> image fp32 [B,3,H,W] in [0,1] (K steps = one graph launch).
        Host tensors take the cdc_decode_host path (H2D + decode + D2H inside the library); page-locked inputs and a
        page-locked `out` (optional, host path only: fp32 [B,3,H,W], returned) are copied from / to directly.
        trajectory / x0_trajectory (lists, as oracle/sampler.py OracleDecoder.decode(trajectory=...)): K device tensors
        [B,3,H,W] are appended to each given list, x_t entering step k and the raw x0_hat of step k (views of one
        allocation, recorded inside the graph by cdc_decode_trajectory).  The image is the same bits either way.
        seeds (one int in [0, 2^64) per image: a sequence, or an int64 / uint64 tensor; not with init): x_T = gamma * z and
        the eta > 0 sampler noise of image b are keyed by seeds[b] alone (set_image_seeds), so image b decodes the same in
        any batch.  Without seeds the batch-wide seed applies (x_T from torch.randn with `seed`, as before)."""
        init, (B, H, W) = self._decode_inputs(latent, steps, init, gamma, seed, seeds)
        record = trajectory is not None or x0_trajectory is not None
        host = cond is None and not latent.is_cuda and (init is None or not init.is_cuda)
        with torch.cuda.device(self.device):
            self.bind(B, H, W)
            self.set_image_seeds(seeds)
            if host and not record and seeds is not None:
                # host buffers, x_T drawn on the device: no x_T transfer
                lat = latent.float().contiguous()
                out = self._check_host_out(out, B, H, W)
                self._ck(self.L.cdc_decode_host_seeded(self.ctx, C.c_void_p(lat.data_ptr()), float(gamma),
                                                       C.c_void_p(out.data_ptr()), self._stream()), "cdc_decode_host_seeded")
                return out
            if host and not record:
                # host buffers: pinned staging + H2D/D2H inside the library
                lat = latent.float().contiguous()
                x0 = init.float().contiguous()
                out = self._check_host_out(out, B, H, W)
                self._ck(self.L.cdc_decode_host(self.ctx, C.c_void_p(lat.data_ptr()), C.c_void_p(x0.data_ptr()),
                                                C.c_void_p(out.data_ptr()), self._stream()), "cdc_decode_host")
                return out
            if host:
                out = self._check_host_out(out, B, H, W)
            if cond is not None:
                self.set_cond(cond)
            else:
                self.set_latent(latent)
            self._bind_x(init, seeds, gamma)
            if not record:
                self._ck(self.L.cdc_decode(self.ctx, self._stream()), "cdc_decode")
                return self._get_x(to_image=True)
            xt, x0 = self._traj_buffers(trajectory is not None, x0_trajectory is not None, 1)
            self.decode_trajectory(xt, x0)
            for lst, buf in ((trajectory, xt), (x0_trajectory, x0)):
                if lst is not None:
                    lst.extend(buf.unbind(0))
            img = self._get_x(to_image=True)
            return out.copy_(img) if host else img

    def decode_resident(self):
        """Replay the K-step graph on whatever x / cond are bound (used by bench.py's device-timed leg)."""
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_decode(self.ctx, self._stream()), "cdc_decode")

    def trajectory_slots(self, every=1):
        """Slots a trajectory decode with this `every` records: ceil(K / every), slot j = step j * every."""
        return (self.steps + every - 1) // every

    def _traj_buffers(self, want_x, want_x0, every):
        B, H, W = self.shape
        n = self.trajectory_slots(every)
        buf = torch.empty((int(want_x) + int(want_x0)) * n, B, 3, H, W, device=self.device, dtype=torch.float32)
        xt = buf[:n] if want_x else None
        x0 = buf[n * int(want_x):] if want_x0 else None
        return xt, x0

    def decode_trajectory(self, x_traj=None, x0_traj=None, every=1):
        """Replay the K-step loop on whatever x / cond are bound (like decode_resident) and record slot j = step
        j * every into x_traj[j] (x_t entering the step) and x0_traj[j] (its raw x0_hat): contiguous fp32 device
        tensors [ceil(K / every), B, 3, H, W], either may be None.  Enqueued on the current stream; the image is then
        what decode_resident leaves (include/cdc_b200.h cdc_decode_trajectory)."""
        if self.shape is None or not self.steps:
            raise RuntimeError("bind a shape (set_latent / set_cond) and set a schedule first")
        if int(every) < 1:
            raise ValueError(f"every must be >= 1, got {every}")
        if x_traj is None and x0_traj is None:
            raise ValueError("give x_traj, x0_traj or both")
        want = (self.trajectory_slots(int(every)), *self.shape[:1], 3, *self.shape[1:])
        for name, t in (("x_traj", x_traj), ("x0_traj", x0_traj)):
            if t is not None and (tuple(t.shape) != want or t.dtype != torch.float32 or t.device != self.device
                                  or not t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous fp32 tensor {want} on {self.device}, got "
                                 f"{tuple(t.shape)} {t.dtype} on {t.device}")
        ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_decode_trajectory(self.ctx, ptr(x_traj), ptr(x0_traj), int(every), self._stream()),
                     "cdc_decode_trajectory")

    @torch.no_grad()
    def decode_progressive(self, latent, steps, *, every=1, init=None, gamma=0.8, seed=0, seeds=None, cond=None):
        """Generator: decode as `decode` does and yield (k, x_t, x0_hat) for k = 0, every, 2 * every, ... as soon as
        the graph has written step k: x_t [B,3,H,W] entering step k and the network's raw x0_hat of that step, device
        fp32.  (x0_hat.clamp(-1, 1) + 1) / 2 is the preview image.  The graph runs on a stream of its own, so the
        caller's stream can copy or display a slot while later steps run; stepping the last x_t once more gives decode()'s
        image.  The buffers live until the graph has passed them, so stopping early is safe.  While the generator is
        suspended, any call of this decoder first makes the current stream wait for the graph; once it ends (exhausted
        or closed), the caller's stream waits for the graph.  seeds: as in decode."""
        if int(every) < 1:
            raise ValueError(f"every must be >= 1, got {every}")
        init, (B, H, W) = self._decode_inputs(latent, steps, init, gamma, seed, seeds)
        with torch.cuda.device(self.device):
            self.bind(B, H, W)
            self.set_image_seeds(seeds)
            if cond is not None:
                self.set_cond(cond)
            else:
                self.set_latent(latent)
            self._bind_x(init, seeds, gamma)
            xt, x0 = self._traj_buffers(True, True, every)
            cur = torch.cuda.current_stream()
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.device)
            side = self._side
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                self.decode_trajectory(xt, x0, every)
            xt.record_stream(side)  # (one allocation: the caching allocator keeps it until the graph has passed)
            self._side_busy = True
        try:
            for j in range(xt.shape[0]):
                self._ck(self.L.cdc_trajectory_wait(self.ctx, j), "cdc_trajectory_wait")
                yield j * every, xt[j], x0[j]
        finally:
            cur.wait_stream(side)
            self._side_busy = False

    # ---- introspection -------------------------------------------------------------------------
    def launches_per_step(self):
        return self.L.cdc_launches_per_step(self.ctx)

    def flops_per_step(self):
        return self.L.cdc_flops_per_step(self.ctx)

    def saturation_count(self, reset=False):
        """Epilogue passes that stored a value saturated to the fp16 range since creation / the last reset (0 = none)."""
        n = C.c_uint64(0)
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_saturation_count(self.ctx, C.byref(n), 1 if reset else 0, self._stream()), "cdc_saturation_count")
        return int(n.value)

    def step_ops(self, seq=0):
        """[(name, flops, bytes)] of the ops of sequence seq of the bound plan (_ffi.SEQ_*: the denoise step, the context
        net, the analysis encoder, the hyper-encoder, the hyper-decoder; include/cdc_b200_tools.h cdc_seq)."""
        n = self.L.cdc_seq_num_ops(self.ctx, seq)
        if n < 0:
            self._ck(n, "cdc_seq_num_ops")
        return [(self.L.cdc_seq_op_name(self.ctx, seq, i).decode(), self.L.cdc_seq_op_flops(self.ctx, seq, i),
                 self.L.cdc_seq_op_bytes(self.ctx, seq, i)) for i in range(n)]

    def step_op_desc(self, i, seq=0):
        """_ffi.StepOpDesc of op i of sequence seq of the bound plan (include/cdc_b200_tools.h cdc_seq_op_describe)."""
        d = _ffi.StepOpDesc()
        self._ck(self.L.cdc_seq_op_describe(self.ctx, seq, i, C.byref(d)), "cdc_seq_op_describe")
        return d

    def run_step_op(self, i, k=0, seq=0):
        """Op i of sequence seq alone, on the current stream (k: the sampler step; the codec sequences ignore it)."""
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_run_seq_op(self.ctx, seq, i, k, self._stream()), "cdc_run_seq_op")

    def profile_step(self, k=0, warm=1):
        """In-stream device time (us) of every op of step k (launched back to back, CUDA events in the library)."""
        n = self.L.cdc_num_step_ops(self.ctx)
        buf = (C.c_float * n)()
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_profile_step(self.ctx, k, warm, buf, self._stream()), "cdc_profile_step")
        return list(buf)

    def profile_graph(self, reps=5):
        """In-graph timing of the captured K-step loop: (start_us, dur_us), each [steps][ops] (median over `reps`
        replays), from per-kernel globaltimer stamps (include/cdc_b200_tools.h cdc_profile_graph)."""
        n = self.L.cdc_num_step_ops(self.ctx)
        st = (C.c_float * (n * self.steps))()
        du = (C.c_float * (n * self.steps))()
        with torch.cuda.device(self.device):
            self._ck(self.L.cdc_profile_graph(self.ctx, reps, st, du, self._stream()), "cdc_profile_graph")
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
