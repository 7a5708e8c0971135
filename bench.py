#!/usr/bin/env python
"""bench.py -- decoded images/s for BASELINE.json configs[1]: full decode of one 768x512
synthetic image, 17-step DDIM, bf16, batch 1 per GPU (CUDA-graphed step loop).

    python bench.py --gpus N --steps K --warmup W            # product (libcdc_b200.so)
    python bench.py --impl reference --gpus N --steps K ...  # CPU oracle on the host cores
    python bench.py ... --dump-outputs DIR                   # also save the images of the last timed step (.npy)

One "step" = one full decode of one image per GPU (context net + 17 DDIM steps).
  value : images/s, inputs (latent, x_T) resident in HBM, timed with CUDA events, max over ranks
  e2e   : same metric through the public API with HOST tensors (pinned staging, H2D + D2H inside
          the timed region)
  roofline : tcgen05 conv kernels, algorithmic FLOPs of their launches in one step / their summed in-graph
          durations (globaltimer stamps written by the kernels themselves), against MEASURED_PEAKS.json bf16_tflops
  roofline_int : the integer kernels (latent rounding, CDF lookup) at the cfg5 symbol count, GB/s against hbm_gbs
  cpu_baseline : the oracle (oracle/, "port": the reference ships no code) on the host cores, bounded sample
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, K_DDIM = 512, 768, 17
METRIC = "decoded images/sec (768x512, 17-step DDIM)"
WORKLOAD = "configs[1]: full decode of one 768x512 synthetic image, 17-step DDIM, 16-bit operands / fp32 accumulate, batch 1 per GPU, CUDA-graphed step loop"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, burst)"
    return 1590.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        """Summarise the samples taken inside the host-time window [t0, t1] (the timed region); nvidia-smi is started
        before the warm-up so that it is already polling when the window opens."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [l for (t, l) in self.samples if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.12)]
        if not inside:  # window shorter than the polling period: the nearest samples
            inside = [l for (_, l) in self.samples[-2:]]
        for s in inside:
            f = [x.strip() for x in s.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_sample(n_steps=2, threads=None):
    """Time the oracle on the host: 1 context-net pass + n_steps of the 17 DDIM steps of one 768x512 decode."""
    import torch
    from oracle.config import CDCConfig
    from oracle.sampler import OracleDecoder
    from oracle.weights import build_codec, build_unet, synthetic_init, synthetic_latent
    cores = threads or os.cpu_count()
    torch.set_num_threads(cores)
    cfg = CDCConfig()
    net = build_unet(cfg).to(memory_format=torch.channels_last)
    codec = build_codec(cfg)
    orc = OracleDecoder(cfg, net, context_net=codec.context)
    orc.set_sample_schedule(K_DDIM)
    lat, x = synthetic_latent(1, H, W), synthetic_init(1, H, W)
    with torch.no_grad():
        t0 = time.perf_counter()
        cond = orc.context_net(lat)
        t_ctx = time.perf_counter() - t0
        ts = []
        for k in range(n_steps):
            t0 = time.perf_counter()
            x = orc.denoise_step(x, orc.sched.idx[k], cond)
            ts.append(time.perf_counter() - t0)
    t_step = min(ts)
    sec_per_image = t_ctx + (sum(ts) if n_steps == K_DDIM else K_DDIM * t_step)  # a full decode is not extrapolated
    return 1.0 / sec_per_image, cores, t_ctx, t_step


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference ships no
    code, so this is the oracle port on all host threads; each bench step = one bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # a CPU sample needs no more than one warm-up (it only pages in weights and the thread pool);
    # keeps `--steps K --warmup W` within minutes whatever W the driver passes
    warm = min(args.warmup, 1)
    vals = []
    for i in range(warm + args.steps):
        v, cores, t_ctx, t_step = cpu_oracle_sample(n_steps=4)
        if i >= warm:
            vals.append(v)
    v = statistics.mean(vals)
    sample = (f"1 context-net pass + 4 of {K_DDIM} DDIM steps of one 768x512 decode per bench step, extrapolated to a full "
              f"decode; {len(vals)} of {args.steps} steps sampled")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def int_roofline(dev, peak_gbs, n=4194304, reps=9):
    """Achieved HBM GB/s of the integer kernels (rows a8 / a9) at the cfg5 symbol count (2048^2 / 256 * 256 = 4 194 304),
    algorithmic bytes (SURVEY.md 8d: 16 B and 28 B per symbol) / CUDA-event time, L2 flushed before every launch."""
    import torch
    from cdc_b200 import cdf_lookup, quantize_symbols
    from cdc_b200.decoder import DeviceTables
    from cdc_b200.synthetic import entropy_inputs, gaussian_tables
    y, mu, sigma = (t.to(dev) for t in entropy_inputs(n))
    tb = DeviceTables(gaussian_tables(), dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    q, _ = quantize_symbols(y, mu, device=dev)

    def timed(fn):
        ts = []
        for i in range(reps + 2):
            flush.fill_(i)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(s.elapsed_time(e))
        return statistics.median(ts)

    # (the Python wrappers allocate their outputs: time the raw ABI calls on preallocated buffers)
    import ctypes as C
    from cdc_b200 import _ffi
    L = _ffi.lib()
    qo = torch.empty(n, dtype=torch.int32, device=dev)
    yh = torch.empty(n, dtype=torch.float32, device=dev)
    outs = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(5)]
    P = lambda t: C.c_void_p(t.data_ptr())
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ms_q = timed(lambda: L.cdc_quantize(P(y), P(mu), P(qo), P(yh), n, 0, 0, st))
    ms_c = timed(lambda: L.cdc_cdf_lookup(P(q), P(sigma), P(tb.cdf), P(tb.row_start), P(tb.cdf_length), P(tb.offset),
                                          P(tb.scale_table), tb.rows, 1, *[P(o) for o in outs], n, st))
    assert torch.equal(qo, q)
    ms_floor = timed(lambda: L.cdc_quantize(P(y), P(mu), P(qo), P(yh), 4, 0, 0, st))  # same call on 4 symbols: launch + event floor
    gq, gc = 16.0 * n / (ms_q * 1e-3) / 1e9, 28.0 * n / (ms_c * 1e-3) / 1e9
    return {"symbols": n, "bound": "hbm", "unit": "GB/s", "peak": peak_gbs,
            "quantize_kernel": {"achieved": gq, "frac": gq / peak_gbs, "us": ms_q * 1e3, "bytes_per_symbol": 16},
            "cdf_lookup_kernel": {"achieved": gc, "frac": gc / peak_gbs, "us": ms_c * 1e3, "bytes_per_symbol": 28},
            "launch_floor_us": ms_floor * 1e3,
            "how": "cdc_quantize / cdc_cdf_lookup on device buffers, CUDA events around ONE launch, median of %d, 256 MiB L2 flush (a write: "
                   "the L2 is full of dirty lines the kernel has to evict) before every launch; launch_floor_us = the same call on 4 symbols" % reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cdc_b200")
    ap.add_argument("--ops-out", default=None, help="write the per-kernel in-graph table of one denoise step (CSV)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--plan-opt", action="append", default=[], metavar="ID=VALUE",
                    help="A/B a planner decision (include/cdc_b200_tools.h cdc_plan_option ids), e.g. 5=0")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the images the last timed step decoded (rank 0) as DIR/image.npy (device-resident leg) and "
                         "DIR/image_e2e.npy (host-tensor leg), fp32 [1, 3, 512, 768]; inputs depend only on the arguments, "
                         "so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the cdc_b200 decode, not to the reference arm's partial decodes")
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))

    # the product arm never touches oracle/: weights and inputs come from the package's own generators
    from cdc_b200 import CDCConfig, Decoder, dp
    from cdc_b200.synthetic import init_noise as synthetic_init, latent as synthetic_latent, random_weights
    dec = Decoder(CDCConfig(), random_weights(CDCConfig(), seed=0, with_context=True), device=dev)
    for po in args.plan_opt:
        dec.set_plan_option(*[int(v) for v in po.split("=")])
    dec.set_sample_schedule(K_DDIM)
    # The job is a list of world * (warmup + steps) images; rank r decodes {i : i mod world == r} (cdc_b200.dp, SURVEY 8e):
    # per-GPU work is fixed as N grows (weak scaling), no collective on the data path.
    n_img = args.warmup + args.steps
    n_job = world * n_img
    mine = dp.shard_indices(n_job, rank, world)
    assert len(mine) == n_img
    lat_h = {i: synthetic_latent(1, H, W, index=i).pin_memory() for i in mine}
    x_h = {i: synthetic_init(1, H, W, index=i).pin_memory() for i in mine}
    lat_d = {i: t.to(dev) for i, t in lat_h.items()}
    x_d = {i: t.to(dev) for i, t in x_h.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    n_warm_job = world * args.warmup  # the first `warmup` images of every rank are untimed

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        sampler = ClockSampler(local)
        sampler.start()  # before the warm-up: nvidia-smi needs ~0.1-0.5 s to deliver its first sample
        dp.decode_sharded(fn, n_warm_job, rank, world)
        barrier()
        t_begin = time.perf_counter()
        evs = []

        def one(i):
            flush.fill_(i & 0xFF)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(i)
            e.record()
            evs.append((s, e))
            return out

        n_done, _ = dp.decode_sharded(lambda j: one(n_warm_job + j), n_job - n_warm_job, rank, world)
        barrier()
        clocks = sampler.stop(t_begin, time.perf_counter())
        ms = sum(s.elapsed_time(e) for s, e in evs)
        # one gather of (images, device seconds) per rank AFTER the timed region; whole-job rate = images / slowest rank
        table = dp.gather_metrics([n_done, ms / 1e3], device=dev)
        return dp.aggregate_throughput(table), float(table[:, 1].max()) * 1e3, clocks

    # device-resident leg: latent and x_T already in HBM; context net + K-step graph + image conversion
    out_keep = []

    def dev_step(i):
        out_keep[:] = [dec.decode(lat_d[i], K_DDIM, init=x_d[i])]
        return out_keep[0]

    value, ms_dev, clocks = timed(dev_step)
    dumps = {"image": out_keep[0].cpu()}

    out_h = torch.empty(1, 3, H, W, dtype=torch.float32).pin_memory()  # the caller's page-locked result buffer

    def host_step(i):
        out_keep[:] = [dec.decode(lat_h[i], K_DDIM, init=x_h[i], out=out_h)]  # cdc_decode_host: H2D + decode + D2H + sync
        return out_keep[0]

    e2e, ms_e2e, _ = timed(host_step)
    assert torch.isfinite(out_keep[0]).all()
    dumps["image_e2e"] = out_keep[0].clone()
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.float().numpy())
    launches = args.steps * (dec.L.cdc_launches_context(dec.ctx) + 2 + K_DDIM * dec.launches_per_step())

    out = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp16" if dec.L.cdc_act_dtype() == 1 else "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "image": [H, W], "ddim_steps": K_DDIM, "batch_per_gpu": 1,
                   "parallelism": f"image-sharded dp{world} (cdc_b200.dp: rank r decodes images i = r mod {world}), no data-path collective",
                   "l2": "flushed between timed iterations (256 MiB write, outside the event brackets)",
                   "precision": "fp16 storage + tcgen05 kind::f16 operands, fp32 accumulate/statistics/sampler state "
                                "(ratified in BASELINE.md: bf16 operands measure 0.02-0.04 against the 1e-2 per-step tolerance; "
                                "tests/test_gpu_parity_r2.py runs the bf16 build)"},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(lat_h[mine[0]].numel() * 4 + x_h[mine[0]].numel() * 4),
                "d2h_bytes_per_step": int(x_h[mine[0]].numel() * 4), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "saturation_events": dec.saturation_count(),
    }

    if rank == 0:
        # ---- roofline of the dominant kernel class (the tcgen05 convs), measured live INSIDE the captured graph ----
        # cdc_profile_graph replays the same 17-step graph with every kernel stamping (earliest CTA start, latest CTA end)
        # in globaltimer ns: per-kernel durations and start-to-start slots without event overhead and with the caches
        # exactly as in the timed decode (replaces round 1's replay-time differencing, VERDICT r1 #6).
        ops = dec.step_ops()
        i0 = mine[0]
        dec.decode(lat_d[i0], K_DDIM, init=x_d[i0])
        torch.cuda.synchronize()
        start, dur = dec.profile_graph(reps=7)
        nops = len(ops)
        kidx = [i for i in range(nops) if ops[i][0] != "gn.clear"]
        # slot of a kernel = time until the next kernel of the graph starts (its duration + the gap behind it)
        flat = [(k, i) for k in range(K_DDIM) for i in kidx]
        slot = {}
        for a, b in zip(flat[:-1], flat[1:]):
            slot[a] = start[b[0]][b[1]] - start[a[0]][a[1]]
        slot[flat[-1]] = dur[flat[-1][0]][flat[-1][1]]
        med = lambda v: statistics.median(v)
        d_us = [med([dur[k][i] for k in range(K_DDIM)]) for i in range(nops)]
        s_us = [med([slot[(k, i)] for k in range(K_DDIM)]) if i in kidx else 0.0 for i in range(nops)]
        graph_us = start[K_DDIM - 1][kidx[-1]] + dur[K_DDIM - 1][kidx[-1]]
        is_conv = [f > 0 and "sdpa" not in n for (n, f, b) in ops]
        conv_fl = sum(f for (n, f, b), c in zip(ops, is_conv) if c)
        conv_us = sum(sum(dur[k][i] for i in range(nops) if is_conv[i]) for k in range(K_DDIM)) / K_DDIM
        conv_slot_us = sum(sum(slot[(k, i)] for i in kidx if is_conv[i]) for k in range(K_DDIM)) / K_DDIM
        ew = [i for i in kidx if ops[i][1] == 0]
        ew_us = sum(sum(dur[k][i] for i in ew) for k in range(K_DDIM)) / K_DDIM
        ew_bytes = sum(ops[i][2] for i in ew)
        n_conv = sum(is_conv)
        n_gn_in = sum(1 for (n, f, b), c in zip(ops, is_conv) if c and "+gn_in" in n)
        peak_tf, peak_gbs, which = peaks()
        conv_us, conv_slot_us, graph_us = max(conv_us, 1e-6), max(conv_slot_us, 1e-6), max(graph_us, 1e-6)  # (a build without stamps reports 0)
        ach = conv_fl / (conv_us * 1e-6) / 1e12
        ach_slot = conv_fl / (conv_slot_us * 1e-6) / 1e12
        traffic, traffic_of = None, None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # dram bytes / launch of the top kernel (ncu --set full)
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic, traffic_of = tj.get("dram_bytes_per_launch"), tj.get("kernel")
        out["roofline"] = {
            "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
            "traffic": traffic, "traffic_of": traffic_of,
            "kernel": f"conv_kf_kernel + conv_tc_kernel: the {n_conv} tcgen05 conv launches of one denoise step "
                      f"({conv_fl / 1e9:.1f} GFLOP algorithmic)"
                      + (f"; {n_gn_in} of them also apply GroupNorm+FiLM+SiLU to their input rows in shared memory, "
                         "replacing elementwise passes" if n_gn_in else ""),
            "peak_source": which,
            "how": "sum over the conv launches of (latest CTA end - earliest CTA start), globaltimer stamps written by the kernels inside the "
                   "captured 17-step graph (cdc_profile_graph, median of 7 replays), averaged over the 17 steps",
            "conv_us_per_step": conv_us,
            "achieved_incl_gaps": ach_slot, "frac_incl_gaps": ach_slot / peak_tf, "conv_slot_us_per_step": conv_slot_us,
            "incl_gaps_how": "same FLOPs / start-to-next-kernel-start slots (kernel + the launch gap behind it): comparable with round 1's "
                             "replay-time differencing (0.499)",
            "graph_ms": graph_us / 1e3, "step_us": graph_us / K_DDIM,
            "step_tflops": dec.flops_per_step() / (graph_us / K_DDIM * 1e-6) / 1e12,
            "elementwise_us_per_step": ew_us, "elementwise_launches": len(ew),
            "elementwise_gbs": ew_bytes / (ew_us * 1e-6) / 1e9 if ew_us > 0 else None,
            "elementwise_frac_of_hbm_peak": ew_bytes / (ew_us * 1e-6) / 1e9 / peak_gbs if ew_us > 0 else None,
        }
        try:
            out["roofline_int"] = int_roofline(dev, peak_gbs)
        except Exception as ex:  # never lose the headline line to the secondary measurement
            out["roofline_int"] = {"error": repr(ex)}
        if args.ops_out:
            with open(args.ops_out, "w") as f:
                f.write("op,gflop,mbytes,us_in_graph,slot_us,tflops,gbs\n")
                for i in kidx:
                    n, fl, b = ops[i]
                    t = max(d_us[i], 1e-3)
                    f.write(f"{n},{fl / 1e9:.3f},{b / 1e6:.3f},{d_us[i]:.2f},{s_us[i]:.2f},{fl / (t * 1e-6) / 1e12:.1f},{b / (t * 1e-6) / 1e9:.0f}\n")
        if not args.no_cpu and world == 1:  # the CPU baseline is an N=1 figure (contract); torchrun also pins OMP threads
            v, cores, t_ctx, t_step = cpu_oracle_sample(n_steps=K_DDIM)
            out["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                                   "sample": f"oracle (fp32 torch eager, channels_last): one full 768x512 decode = 1 context-net pass ({t_ctx:.2f} s) "
                                             f"+ all {K_DDIM} DDIM steps (fastest {t_step:.2f} s/step)"}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
