#!/usr/bin/env python
"""What drawing x_T costs per image, host vs device (DESIGN.md section 3.11).

    python tools/seeded_init_cost.py [--reps N] [--sizes 768x512,2048x2048]

For each size (batch 1, K = 17, synthetic weights and latents), four arms, alternated image by image (the first rotates):
  host_randn   decode(latent_host, K, seed=i): torch.randn x_T on the host, cdc_decode_host (H2D of latent + x_T)
  host_seeded  decode(latent_host, K, seeds=[i]): cdc_decode_host_seeded (no x_T on the host or on the bus)
  dev_init     decode(latent_dev, K, init=x_T_dev): x_T already in HBM (cdc_set_x)
  dev_seeded   decode(latent_dev, K, seeds=[i]): x_T drawn by init_noise_kernel
Each arm's time is the host clock from the call to a device synchronise, median over the reps, in ms per image.  Also
timed on their own: torch.randn of one x_T on the host, Decoder.set_image_seeds of one seed (host clock to a device
synchronise), and init_noise_kernel (CUDA events over 200 launches)."""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # (the numbers still stand; the card line says why it is missing)
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=12)
    ap.add_argument("--sizes", default="768x512,2048x2048", help="WxH list")
    ap.add_argument("--steps", type=int, default=17)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("seeded_init_cost.py measures on the GPU; no CUDA device found")
    from cdc_b200 import CDCConfig, Decoder
    from cdc_b200.synthetic import init_noise, latent, random_weights
    dev = "cuda:0"
    K = args.steps
    dec = Decoder(CDCConfig(), random_weights(CDCConfig(), seed=0, with_context=True), device=dev)
    dec.set_sample_schedule(K)
    print(f"card: {card()}; torch {torch.__version__}; host CPUs: {os.cpu_count()}; K = {K}, batch 1")

    for size in args.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        lat_h = latent(1, H, W, index=0)
        lat_d = lat_h.to(dev)
        x_d = init_noise(1, H, W, index=0).to(dev)
        arms = {
            "host_randn": lambda i: dec.decode(lat_h, K, seed=i),
            "host_seeded": lambda i: dec.decode(lat_h, K, seeds=[i]),
            "dev_init": lambda i: dec.decode(lat_d, K, init=x_d),
            "dev_seeded": lambda i: dec.decode(lat_d, K, seeds=[i]),
        }
        times = {n: [] for n in arms}
        for i in range(args.reps + 2):  # the first two rounds warm up (graph capture, pinned staging, allocator)
            names = list(arms)
            for n in names[i % 4:] + names[:i % 4]:  # the arm that goes first rotates
                fn = arms[n]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(i)
                torch.cuda.synchronize()
                if i >= 2:
                    times[n].append((time.perf_counter() - t0) * 1e3)
        # the two pieces on their own
        rt = []
        for i in range(args.reps):
            t0 = time.perf_counter()
            g = torch.Generator().manual_seed(i)
            _ = 0.8 * torch.randn(1, 3, H, W, generator=g)
            rt.append((time.perf_counter() - t0) * 1e3)
        st = []  # binding one image's seed: host call to device synchronise
        for i in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dec.set_image_seeds([i])
            torch.cuda.synchronize()
            st.append((time.perf_counter() - t0) * 1e3)
        dec.set_image_seeds([1])
        for _ in range(10):
            dec.init_noise(0.8)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(200):
            dec.init_noise(0.8)
        e.record()
        torch.cuda.synchronize()
        k_us = s.elapsed_time(e) / 200 * 1e3
        dec.set_image_seeds(None)
        gbs = H * W * (3 * 4 + 16 * 2) / (k_us * 1e-6) / 1e9
        print(f"{W}x{H}: " + ", ".join(f"{n} {statistics.median(v):.2f} ms" for n, v in times.items())
              + f" (median of {args.reps}; spread {min(times['dev_init']):.2f}-{max(times['dev_init']):.2f} ms on dev_init)")
        print(f"{W}x{H}: host randn of x_T alone {statistics.median(rt):.2f} ms; set_image_seeds {statistics.median(st) * 1e3:.0f} us; "
              f"init_noise_kernel {k_us:.1f} us ({gbs:.0f} GB/s of stores)")


if __name__ == "__main__":
    main()
