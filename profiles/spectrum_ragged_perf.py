"""Ragged spectrum calls against what a caller does without them, on one GPU, with the outputs compared byte for byte in the same run.

  1. node case: the reference node's three face crops (257x301, 211x173, 127x255) from host memory — one
     spectrum_ragged_host call against three spectrum_host calls; median wall clock per call (each call synchronises).
  2. 512 device-resident crops of seeded random sizes, 64..400 pixels a side — one v5ela.spectrum_ragged call against a loop of
     one v5ela.spectrum_batch call per crop; CUDA events around the whole call (host enqueue included).
  3. 64 x 1080p — one ragged call against one uniform v5ela.spectrum_batch call; CUDA events.
Prints the card name and power limit first. usage: python profiles/spectrum_ragged_perf.py [--out result.json]"""
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def event_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), float(np.min(times))


def node_case(reps):
    rng = np.random.default_rng(0)
    crops = [rng.integers(0, 256, hw, dtype=np.uint8) for hw in ((257, 301), (211, 173), (127, 255))]
    rag = host.spectrum_ragged_host(crops)
    loop = [host.spectrum_host(c) for c in crops]
    same = all(np.array_equal(a, b) for a, b in zip(rag, loop))
    res = {}
    for name, fn in (("ragged_host", lambda: host.spectrum_ragged_host(crops)), ("three_spectrum_host", lambda: [host.spectrum_host(c) for c in crops])):
        for _ in range(20):
            fn()
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            t.append((time.perf_counter() - t0) * 1e3)
        res[name + "_ms_median"] = float(np.median(t))
    return {"case": "node 3 crops, host arrays", "identical": same, **res}


def mixed_crops(reps):
    rng = np.random.default_rng(512)
    sizes = rng.integers(64, 401, (512, 2))
    crops = [torch.from_numpy(rng.integers(0, 256, (int(h), int(w)), dtype=np.uint8)).cuda() for h, w in sizes]
    rag = v5ela.spectrum_ragged(crops)
    loop = [v5ela.spectrum_batch(c[None])[0] for c in crops]
    torch.cuda.synchronize()
    same = all(torch.equal(a, b) for a, b in zip(rag, loop))
    ragged_ms = event_ms(lambda: v5ela.spectrum_ragged(crops), reps)
    loop_ms = event_ms(lambda: [v5ela.spectrum_batch(c[None]) for c in crops], reps)
    smooth = sum(1 for h, w in sizes if all(_smooth(int(v)) for v in (h, w)))
    return {"case": "512 device crops, 64..400 px a side", "identical": same, "fft_path_crops": smooth, "ragged_ms_median": ragged_ms[0],
            "ragged_ms_min": ragged_ms[1], "per_crop_loop_ms_median": loop_ms[0], "per_crop_loop_ms_min": loop_ms[1]}


def hd_batch(reps):
    g = torch.randint(0, 256, (64, 1080, 1920), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(64))
    views = [g[i] for i in range(64)]
    rag = v5ela.spectrum_ragged(views)
    uni = v5ela.spectrum_batch(g)
    torch.cuda.synchronize()
    same = all(torch.equal(rag[i], uni[i]) for i in range(64))
    ragged_ms = event_ms(lambda: v5ela.spectrum_ragged(views), reps)
    uniform_ms = event_ms(lambda: v5ela.spectrum_batch(g), reps)
    return {"case": "64 x 1080p", "identical": same, "ragged_ms_median": ragged_ms[0], "ragged_ms_min": ragged_ms[1],
            "uniform_ms_median": uniform_ms[0], "uniform_ms_min": uniform_ms[1]}


def _smooth(n):
    for p in (2, 3, 5):
        while n % p == 0:
            n //= p
    return n == 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result as JSON to this path")
    ap.add_argument("--reps", type=int, default=10, help="timed repetitions of cases 2 and 3 (case 1 takes 20x as many)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    res = {"card": card(), "cases": [node_case(20 * args.reps), mixed_crops(args.reps), hd_batch(args.reps)]}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not all(c["identical"] for c in res["cases"]):
        sys.exit("ragged outputs differ from the per-image calls")


if __name__ == "__main__":
    main()
