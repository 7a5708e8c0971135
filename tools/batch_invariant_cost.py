#!/usr/bin/env python
"""What batch-invariant plans cost (DESIGN.md section 3.13): replay time of the K-step decode graph of a default decoder
against a batch-invariant one (Decoder(..., batch_invariant=True)), at batches 1, 2, 4, 8 and 16.  One process, both
decoders bound to the same batch; per round each arm replays its graph for at least --window seconds, timed with CUDA
events, the arms alternating and the first arm rotating from round to round; the result is the median round.

    python tools/batch_invariant_cost.py            # 512 x 768, K = 17, B = 1 2 4 8 16, 16 rounds

Prints one line per batch (ms per image and images/s of each arm, their ratio, the spread over the rounds), the card,
its power limit and maximum SM clock, then ONE JSON line with the same numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cdc_b200 import CDCConfig, Decoder  # noqa: E402
from cdc_b200.synthetic import latent, random_weights  # noqa: E402


def card_line():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=768)
    ap.add_argument("--steps", type=int, default=17)
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 2, 4, 8, 16])
    ap.add_argument("--rounds", type=int, default=16)
    ap.add_argument("--window", type=float, default=0.25, help="timed seconds per arm and round (at least)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_invariant_cost.py measures on the GPU; no CUDA device found")
    H, W, K = a.height, a.width, a.steps
    weights = random_weights(CDCConfig(), seed=0, with_context=True)
    decs = {"default": Decoder(CDCConfig(), weights, device="cuda:0"),
            "invariant": Decoder(CDCConfig(), weights, device="cuda:0", batch_invariant=True)}
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"shape": [H, W], "steps": K, "rounds": a.rounds, "card": card_line(), "batches": {}}
    print(f"{res['card']}; {H}x{W}, K = {K}, {a.rounds} rounds per batch")
    for B in a.batches:
        for d in decs.values():
            d.set_sample_schedule(K)
            d.set_latent(latent(B, H, W, index=0).cuda())
            d.set_image_seeds(list(range(1, B + 1)))
            d.init_noise(0.8)
            for _ in range(3):  # capture the graph, warm up
                d.decode_resident()
        torch.cuda.synchronize()
        s.record()
        decs["default"].decode_resident()
        e.record()
        torch.cuda.synchronize()
        reps = max(1, int(a.window * 1e3 / s.elapsed_time(e)) + 1)
        per = {n: [] for n in decs}
        names = list(decs)
        for r in range(a.rounds):
            for name in (names if r % 2 == 0 else names[::-1]):
                d = decs[name]
                torch.cuda.synchronize()
                s.record()
                for _ in range(reps):
                    d.decode_resident()
                e.record()
                torch.cuda.synchronize()
                per[name].append(s.elapsed_time(e) / reps / B)
        med = {n: sorted(v)[len(v) // 2] for n, v in per.items()}
        ratio = med["invariant"] / med["default"]
        res["batches"][str(B)] = {
            n: {"ms_per_image": round(med[n], 4), "images_per_s": round(1e3 / med[n], 2),
                "spread_ms_per_image": [round(min(per[n]), 4), round(max(per[n]), 4)]} for n in decs}
        res["batches"][str(B)]["reps_per_round"] = reps
        res["batches"][str(B)]["invariant_over_default"] = round(ratio, 4)
        print(f"B = {B:2d}: default {med['default']:7.3f} ms/image ({1e3 / med['default']:6.2f} images/s)  "
              f"invariant {med['invariant']:7.3f} ms/image ({1e3 / med['invariant']:6.2f} images/s)  "
              f"ratio {ratio:.4f}  spread default [{min(per['default']):.3f}, {max(per['default']):.3f}] "
              f"invariant [{min(per['invariant']):.3f}, {max(per['invariant']):.3f}]  ({reps} replays per window)", flush=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
