"""Randomised parity soak on one B200 (development aid; the pytest -m gpu suite is the gate): random sizes, qualities and
content through every C-ABI path, against the live libraries (Pillow / OpenCV) and the C oracle.
Usage: python profiles/soak_parity.py [cases] [seed]  -> one summary line per path."""
import io
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "fake-video-detection-engine_b200")]
import cv2  # noqa: E402
from PIL import Image  # noqa: E402

import v5ela  # noqa: E402
from oracle import c_oracle  # noqa: E402
from v5ela import host as v5host, jpeg  # noqa: E402


def content(rng, kind, h, w):
    if kind == 0:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:
        return v5ela.gen_frame(int(rng.integers(1 << 20)), h, w, int(rng.integers(100)))
    if kind == 2:
        return np.full((h, w, 3), rng.integers(0, 256, 3), dtype=np.uint8)
    if kind == 3:
        return (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    a = v5ela.gen_frame(int(rng.integers(1 << 20)), h, w, 7).astype(np.int16)
    return np.clip(a + rng.integers(-40, 41, a.shape), 0, 255).astype(np.uint8)


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 600
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 2026
    rng = np.random.default_rng(seed)
    bad = {"encode_rgb": 0, "encode_gray": 0, "decode_rgb": 0, "decode_gray": 0, "analyze_records": 0, "analyze_residual": 0,
           "records_only_fast": 0, "ragged_records": 0, "ragged_residual": 0}
    counts = {"records_only_fast": 0, "ragged_frames": 0}
    t0 = time.time()
    pending, crops = [], []
    hd = v5host.get_handle(0)
    for it in range(cases):
        hd.block_stage = "mma" if it % 2 else "smem"                      # both builds of the block stage, alternating
        big = it % 20 == 0
        h = int(rng.integers(1, 900 if big else 200))
        w = int(rng.integers(1, 1300 if big else 260))
        if it % 3 == 0:
            w = 16 * max(1, w // 16)                                       # a third of the widths: multiples of 16 (FAST instantiation)
        q = int(rng.integers(1, 101))
        img = content(rng, it % 5, h, w)
        buf = io.BytesIO()
        Image.fromarray(img, "RGB").save(buf, "JPEG", quality=q)
        ref_file = buf.getvalue()
        gray = np.ascontiguousarray(img[..., it % 3])
        ok, enc = cv2.imencode(".jpg", gray, [cv2.IMWRITE_JPEG_QUALITY, q])
        ref_gray_file = enc.tobytes()
        bad["encode_rgb"] += jpeg.encode_host(img[None], q)[0] != ref_file
        bad["encode_gray"] += jpeg.encode_host(gray[None], q)[0] != ref_gray_file
        pending.append((ref_file, ref_gray_file))
        recs, resid, _ = v5host.analyze_frames_host(img[None], quality=q, want_residual=True)
        orec, oresid = c_oracle.analyze(img[None], q, want_residual=True)
        bad["analyze_records"] += recs.tobytes() != orec.tobytes()
        bad["analyze_residual"] += not np.array_equal(resid, oresid)
        if w % 16 == 0:                                                    # records-only call: the benchmarked instantiation
            recs2, _, _ = v5host.analyze_frames_host(img[None], quality=q)
            bad["records_only_fast"] += recs2.tobytes() != orec.tobytes() or hd.last_instantiation != "fast"
            counts["records_only_fast"] += 1
        crops.append(img)
        if len(crops) == 7 or it == cases - 1:                             # ragged batch: different sizes in one launch
            rrecs, rres, _ = v5host.analyze_ragged_host(crops, quality=q, want_residual=True)
            for j, c in enumerate(crops):
                o = c_oracle.analyze_frame(c, q)
                bad["ragged_records"] += rrecs[j].tobytes() != o["record"].tobytes()
                bad["ragged_residual"] += not np.array_equal(rres[j], o["residual"])
            counts["ragged_frames"] += len(crops)
            crops = []
        if len(pending) == 16 or it == cases - 1:                          # mixed-size decode batches
            files = [f for pair in pending for f in pair]
            outs = jpeg.decode_host(files, want_rgb=True, want_gray=True)
            for f, o in zip(files, outs):
                bad["decode_rgb"] += not np.array_equal(o["rgb"], np.asarray(Image.open(io.BytesIO(f)).convert("RGB")))
                bad["decode_gray"] += not np.array_equal(o["gray"], cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_GRAYSCALE))
            pending = []
    print(f"soak: {cases} random cases (seed {seed}), sizes 1..899 x 1..1299, quality 1..100, 5 content kinds, {time.time() - t0:.0f} s")
    for k, v in bad.items():
        print(f"  {k:18s} mismatches: {int(v)}")
    print(f"  (records-only FAST calls: {counts['records_only_fast']}, frames through ragged batches: {counts['ragged_frames']}; block stage alternating smem / mma)")
    return 1 if any(bad.values()) else 0


if __name__ == "__main__":
    sys.exit(main())
