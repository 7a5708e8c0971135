#!/usr/bin/env python
"""What one library call per direction costs against the Python codec path, per image (DESIGN.md section 3.12).

    python tools/codec_rgb8_cost.py [--reps N] [--sizes 768x512,2048x2048] [--steps K]

For each size (batch 1, synthetic weights and images), two arms per direction, alternated image by image (the first
rotates):
  compress    C: Codec.compress_rgb8(u8)              (cdc_compress_rgb8: u8 in, bytes out)
              py: Codec.compress(u8 -> fp32 NCHW / 255) (torch conversion, then the per-stage calls and host glue)
  decompress  C: Codec.decompress_rgb8(data, K, seeds)  (cdc_decompress_rgb8: bytes in, u8 out)
              py: Codec.decompress_bytes(data, K, seeds) -> * 255 -> round -> uint8 NHWC on the host
Each time is the host clock from the call to a device synchronise, median over the reps, in ms per image; the two arms'
outputs are checked equal."""
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
    ap.add_argument("--reps", type=int, default=16)
    ap.add_argument("--sizes", default="768x512,2048x2048", help="WxH list")
    ap.add_argument("--steps", type=int, default=17)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("codec_rgb8_cost.py measures on the GPU; no CUDA device found")
    from cdc_b200 import CDCConfig, Codec, Decoder
    from cdc_b200.synthetic import image, random_weights
    dev = "cuda:0"
    K = args.steps
    w = random_weights(CDCConfig(), seed=0, with_context=True, with_codec=True)
    codec = Codec(Decoder(CDCConfig(), w, device=dev), fact_tables=Codec.prior_tables(w))
    print(f"card: {card()}; torch {torch.__version__}; host CPUs: {os.cpu_count()}; K = {K}, batch 1")

    def to_u8(img01):
        return (img01 * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()

    for size in args.sizes.split(","):
        W, H = (int(v) for v in size.split("x"))
        imgs = [to_u8(image(1, H, W, index=i)) for i in range(4)]
        streams = [codec.compress_rgb8(u8) for u8 in imgs]
        arms = {
            "compress C": lambda i: codec.compress_rgb8(imgs[i % 4]),
            "compress py": lambda i: codec.compress(imgs[i % 4].permute(0, 3, 1, 2).float() / 255)[0],
            "decompress C": lambda i: codec.decompress_rgb8(streams[i % 4], K, seeds=[i]),
            "decompress py": lambda i: (codec.decompress_bytes(streams[i % 4], K, seeds=[i]) * 255).round().to(torch.uint8)
                                       .permute(0, 2, 3, 1).cpu(),
        }
        times = {n: [] for n in arms}
        for i in range(args.reps + 2):  # the first two rounds warm up (plans, graph capture, work buffers, allocator)
            names = list(arms)
            outs = {}
            for n in names[i % 4:] + names[:i % 4]:  # the arm that goes first rotates
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                outs[n] = arms[n](i)
                torch.cuda.synchronize()
                if i >= 2:
                    times[n].append((time.perf_counter() - t0) * 1e3)
            assert outs["compress C"] == outs["compress py"], "compress: the two paths wrote different bytes"
            assert torch.equal(outs["decompress C"], outs["decompress py"]), "decompress: the two paths gave different pixels"
        print(f"{W}x{H}: " + ", ".join(f"{n} {statistics.median(v):.2f} ms" for n, v in times.items())
              + f" (median of {args.reps}; {len(streams[0])} bytes for image 0)")


if __name__ == "__main__":
    main()
