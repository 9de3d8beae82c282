"""Quality sweeps (v5ela_analyze_sweep) against one call per quality, on one GPU. The two arms of each case alternate rep by rep in
the same run, and their outputs are compared byte for byte first.

  1. node scale: three 257x301 crops from host memory at 10 qualities (50, 55, ..., 95) — one analyze_sweep_host call against
     10 analyze_ragged_host calls; host wall clock per call sequence (every call synchronises).
  2. device scale: 64 x 1080p at {75, 85, 90, 95} — one v5ela.analyze_sweep call against four v5ela.analyze_batch calls (those take
     the FAST instantiation, the sweep the general one); CUDA events around the whole sequence (host enqueue included).
  3. ghost-map cost: case 2's sweep with and without the maps; CUDA events.
Prints the card name and power limit first. usage: python profiles/sweep_perf.py [--out result.json] [--reps N]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "fake-video-detection-engine_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import v5ela  # noqa: E402
from v5ela import host  # noqa: E402
from v5ela.synth import gen_batch_torch, gen_frame  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def alternate(arms, reps, timer):
    """Times each arm once per rep, arms interleaved; -> {name: (median ms, min ms)}."""
    times = {name: [] for name in arms}
    for _ in range(reps):
        for name, fn in arms.items():
            times[name].append(timer(fn))
    return {name: (float(np.median(t)), float(np.min(t))) for name, t in times.items()}


def wall_ms(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def node_case(reps):
    crops = [gen_frame(k, 257, 301, 7) for k in range(3)]
    qualities = list(range(50, 100, 5))
    sweep = host.analyze_sweep_host(crops, qualities)[0]
    loop = np.stack([host.analyze_ragged_host(crops, quality=q)[0] for q in qualities])
    same = sweep.tobytes() == loop.tobytes()
    arms = {"sweep_host": lambda: host.analyze_sweep_host(crops, qualities),
            "ten_ragged_host": lambda: [host.analyze_ragged_host(crops, quality=q) for q in qualities]}
    alternate(arms, 20, wall_ms)                                 # warm-up
    t = alternate(arms, reps, wall_ms)
    return {"case": "node: 3 x 257x301 host crops at 10 qualities", "identical": same,
            **{f"{k}_ms_median": v[0] for k, v in t.items()}, **{f"{k}_ms_min": v[1] for k, v in t.items()}}


def device_cases(reps):
    frames = gen_batch_torch(0, 64, 1080, 1920, seed=64)
    qualities = [75, 85, 90, 95]
    sweep = v5ela.analyze_sweep(frames, qualities, want_ghost=True)
    loop = [v5ela.analyze_batch(frames, quality=q)["records"] for q in qualities]
    plain = v5ela.analyze_sweep(frames, qualities)
    torch.cuda.synchronize()
    same = all(torch.equal(sweep["records"][k], loop[k]) for k in range(4))
    same_plain = torch.equal(plain["records"], sweep["records"])
    arms = {"sweep": lambda: v5ela.analyze_sweep(frames, qualities),
            "four_analyze_batch": lambda: [v5ela.analyze_batch(frames, quality=q) for q in qualities],
            "sweep_with_ghost": lambda: v5ela.analyze_sweep(frames, qualities, want_ghost=True)}
    alternate(arms, 3, event_ms)                                 # warm-up
    t = alternate(arms, reps, event_ms)
    px = 64 * 1080 * 1920 * len(qualities)
    device = {"case": "device: 64 x 1080p at {75, 85, 90, 95}", "identical": same,
              "sweep_ms_median": t["sweep"][0], "sweep_ms_min": t["sweep"][1],
              "four_analyze_batch_ms_median": t["four_analyze_batch"][0], "four_analyze_batch_ms_min": t["four_analyze_batch"][1],
              "sweep_gpix_per_s": px / (t["sweep"][0] * 1e6), "four_analyze_batch_gpix_per_s": px / (t["four_analyze_batch"][0] * 1e6)}
    ghost = {"case": "ghost-map cost: the device-scale sweep with and without d_ghost", "identical": same_plain,
             "without_ms_median": t["sweep"][0], "with_ms_median": t["sweep_with_ghost"][0], "with_ms_min": t["sweep_with_ghost"][1],
             "overhead_pct": 100.0 * (t["sweep_with_ghost"][0] / t["sweep"][0] - 1.0)}
    return [device, ghost]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result as JSON to this path")
    ap.add_argument("--reps", type=int, default=10, help="timed repetitions of the device cases (the node case takes 20x as many)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    res = {"card": card(), "cases": [node_case(20 * args.reps), *device_cases(args.reps)]}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not all(c["identical"] for c in res["cases"]):
        sys.exit("sweep outputs differ from the per-quality calls")


if __name__ == "__main__":
    main()
