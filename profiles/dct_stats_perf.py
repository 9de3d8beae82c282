"""DCT statistics (v5ela_jpeg_dct_stats) against decoding the same files (v5ela_jpeg_decode), on one GPU: 256 x 1080p 4:2:0 files
at quality 90, pageable host bytes, one call per arm. Arms: jpeg.decode_batch (RGB), jpeg.dct_stats without and with the map. The
arms alternate rep by rep; CUDA events around each whole call (header parsing and staging on the calling thread included).
Outputs are checked first: the histograms and maps of the first and last file against NumPy over the oracle decoder's
coefficients, and the first file's pixels against the oracle decoder.
Prints the card name and power limit first. usage: python profiles/dct_stats_perf.py [--out result.json] [--reps N]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "fake-video-detection-engine_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from v5ela import jpeg, records  # noqa: E402
from v5ela.synth import gen_batch_torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def make_files(n):
    files = []
    for k in range(0, n, 32):
        frames = gen_batch_torch(k, min(32, n - k), 1080, 1920, seed=90)
        out, sizes = jpeg.encode_batch(frames, 90)
        torch.cuda.synchronize()
        o, s = out.cpu().numpy(), sizes.cpu().numpy()
        files += [o[i, :s[i]].tobytes() for i in range(len(s))]
    return files


def check(files):
    from dct_helpers import luma_grid, np_hist
    from oracle import c_oracle

    stats = jpeg.dct_stats(files, want_map=True)
    dec = jpeg.decode_batch(files[:1])
    torch.cuda.synchronize()
    ok = bool((stats["status"] == 0).all())
    hist = stats["hist"].cpu().numpy().view(np.uint32)
    worst = 0.0
    for i in (0, len(files) - 1):
        ok = ok and np.array_equal(hist[i], np_hist(files[i]))
        ref = records.dq_map(hist[i], luma_grid(files[i]))
        worst = max(worst, float(np.abs(stats["map"][i].cpu().numpy().astype(np.float64) - ref).max()))
    ok = ok and worst <= 1e-6 and np.array_equal(dec["rgb"][0].cpu().numpy(), c_oracle.jpeg_decode(files[0])["rgb"])
    return ok, worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result as JSON to this path")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--files", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    files = make_files(args.files)
    ok, worst = check(files)
    arms = {"decode_rgb": lambda: jpeg.decode_batch(files),
            "dct_stats": lambda: jpeg.dct_stats(files),
            "dct_stats_map": lambda: jpeg.dct_stats(files, want_map=True)}
    for fn in arms.values():                                      # warm-up
        event_ms(fn)
    times = {k: [] for k in arms}
    for _ in range(args.reps):
        for k, fn in arms.items():
            times[k].append(event_ms(fn))
    res = {"card": card(), "case": f"{args.files} x 1080p 4:2:0 q90 files, pageable host bytes, one call per arm",
           "outputs_checked": ok, "map_max_abs_diff_vs_numpy": worst, "mean_file_bytes": float(np.mean([len(f) for f in files])),
           **{f"{k}_ms_median": float(np.median(v)) for k, v in times.items()},
           **{f"{k}_ms_min": float(np.min(v)) for k, v in times.items()}, "reps": args.reps}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not ok:
        sys.exit("outputs differ from the references")


if __name__ == "__main__":
    main()
