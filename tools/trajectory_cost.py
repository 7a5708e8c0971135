#!/usr/bin/env python
"""What recording the trajectory costs (DESIGN.md section 3.10): replay time of the plain K-step graph (cdc_decode, as
bench.py's device-timed leg runs it) against the trajectory graph (cdc_decode_trajectory) recording every step and every
4th step, x_t and x0_hat both.  One process, one decoder, the arms alternated round by round and timed with CUDA events
over at least --seconds per arm; the result is the median round.

    python tools/trajectory_cost.py            # 1 x 512 x 768, K = 17

Prints one line per arm (ms per image, overhead against the plain graph, and that overhead per recorded step as a share
of one denoise step), the card and its power limit, then ONE JSON line with the same numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cdc_b200 import CDCConfig, Decoder  # noqa: E402
from cdc_b200.synthetic import init_noise, latent, random_weights  # noqa: E402


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=768)
    ap.add_argument("--steps", type=int, default=17)
    ap.add_argument("--seconds", type=float, default=2.5, help="timed seconds per arm (at least)")
    ap.add_argument("--rounds", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("trajectory_cost.py measures on the GPU; no CUDA device found")
    B, H, W, K = 1, a.height, a.width, a.steps
    dec = Decoder(CDCConfig(), random_weights(CDCConfig(), seed=0, with_context=True), device="cuda:0")
    dec.set_sample_schedule(K)
    dec.set_latent(latent(B, H, W, index=0).cuda())
    dec._set_x(init_noise(B, H, W, index=0).cuda())
    bufs = {e: dec._traj_buffers(True, True, e) for e in (1, 4)}
    arms = {"plain": dec.decode_resident,
            "every=1": lambda: dec.decode_trajectory(*bufs[1], every=1),
            "every=4": lambda: dec.decode_trajectory(*bufs[4], every=4)}
    for run in arms.values():  # capture every graph and warm up
        for _ in range(3):
            run()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    dec.decode_resident()
    e.record()
    torch.cuda.synchronize()
    reps = max(1, int(a.seconds * 1e3 / s.elapsed_time(e) / a.rounds) + 1)
    per = {n: [] for n in arms}
    for _ in range(a.rounds):
        for name, run in arms.items():
            # the context keeps one trajectory graph: switching `every` re-captures it, on the host.  One untimed replay
            # and a synchronise keep that (and the previous arm's tail) out of the timed window.
            run()
            torch.cuda.synchronize()
            s.record()
            for _ in range(reps):
                run()
            e.record()
            torch.cuda.synchronize()
            per[name].append(s.elapsed_time(e) / reps)
    med = {n: sorted(v)[len(v) // 2] for n, v in per.items()}
    base = med["plain"]
    step_us = base / K * 1e3
    card, plimit = torch.cuda.get_device_name(), power_limit()
    res = {"shape": [B, H, W], "steps": K, "reps_per_round": reps, "rounds": a.rounds, "card": card, "power_limit": plimit,
           "step_us": round(step_us, 1), "arms": {}}
    print(f"{card}, power limit {plimit}; {B}x{H}x{W}, K = {K}, {a.rounds} rounds x {reps} replays per arm")
    for name, ms in med.items():
        slots = {"plain": 0, "every=1": dec.trajectory_slots(1), "every=4": dec.trajectory_slots(4)}[name]
        over = (ms - base) / base * 100
        per_slot = (ms - base) * 1e3 / slots if slots else 0.0
        res["arms"][name] = {"ms_per_image": round(ms, 4), "overhead_pct": round(over, 3), "slots": slots,
                             "us_per_recorded_step": round(per_slot, 2),
                             "pct_of_step_per_recorded_step": round(per_slot / step_us * 100, 3),
                             "spread_ms": [round(min(per[name]), 4), round(max(per[name]), 4)]}
        print(f"{name:8s} {ms:8.3f} ms/image  overhead {over:+6.2f} %" +
              (f"  {per_slot:6.2f} us per recorded step ({per_slot / step_us * 100:+.2f} % of a {step_us:.0f} us step)"
               if slots else ""))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
