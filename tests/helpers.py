"""Shared helpers for the test-suite (test infrastructure; may import oracle/)."""
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def sha(a) -> str:
    if isinstance(a, np.ndarray):
        a = np.ascontiguousarray(a).tobytes()
    return hashlib.sha256(a).hexdigest()[:16]


def load_json(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def golden_frame(case) -> np.ndarray:
    """Rebuild the input frame of a frames_golden.json case (same code as tests/golden/make_golden.py)."""
    from v5ela.synth import gen_frame

    spec, h, w = case["spec"], case["h"], case["w"]
    if spec[0] == "gen":
        return gen_frame(spec[1], h, w, spec[2])
    rng = np.random.default_rng(spec[1])
    kind = spec[0]
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "binary":
        return (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    if kind == "checker":
        yy, xx = np.mgrid[0:h, 0:w]
        return np.repeat((((yy + xx) & 1) * 255).astype(np.uint8)[..., None], 3, axis=2)
    if kind == "flat":
        return np.full((h, w, 3), [200, 30, 90], dtype=np.uint8)
    if kind == "saturated":
        a = np.zeros((h, w, 3), np.uint8)
        a[..., 0] = 255 * ((np.arange(w)[None, :] // 3) & 1)
        a[..., 2] = 255 * ((np.arange(h)[:, None] // 5) & 1)
        return a
    raise ValueError(kind)


def record_matches_golden(rec, case) -> list:
    """List of field names where a structured record differs from a golden case (empty = match)."""
    bad = []
    for k in ("ela_max", "ela_sum", "ela_sumsq"):
        if [int(v) for v in rec[k]] != case[k]:
            bad.append(k)
    for k in ("tex_sumabs", "tex_sumsq", "tex_maxabs"):
        if int(rec[k]) != case[k]:
            bad.append(k)
    if sha(rec["ela_hist"]) != case["ela_hist_sha"]:
        bad.append("ela_hist")
    if sha(rec.tobytes()) != case["record_sha"]:
        bad.append("record_bytes")
    return bad


def layout_golden_files():
    """[(case, label, file bytes, golden entry)] of tests/golden/layouts_golden.json: the files are written again with the
    generator's own code (tests/golden/make_layouts_golden.py) and must hash to what it recorded."""
    import hashlib
    import importlib.util

    spec = importlib.util.spec_from_file_location("make_layouts_golden", os.path.join(GOLDEN, "make_layouts_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    out = []
    for case in load_json("layouts_golden.json")["cases"]:
        rgb = golden_frame(case)
        assert sha(rgb) == case["in_sha"]
        written = dict(gen.layout_files(rgb, case["q"]))
        for entry in case["files"]:
            data = written[entry["label"]]
            assert (len(data), hashlib.sha256(data).hexdigest()[:16]) == (entry["file_len"], entry["file_sha"]), (case["spec"], entry["label"])
            out.append((case, entry["label"], data, entry))
    return out


def check_layout_goldens(decode):
    """decode(list of file bytes) -> list of dict(rgb, gray); every file of layouts_golden.json must decode to the recorded pixels."""
    items = layout_golden_files()
    outs = decode([data for _, _, data, _ in items])
    assert len(outs) == len(items) == 100
    for (case, label, _, entry), o in zip(items, outs):
        assert sha(o["rgb"]) == entry["dec_rgb_sha"], (case["spec"], case["h"], case["w"], label)
        assert sha(o["gray"]) == entry["dec_y_sha"], (case["spec"], case["h"], case["w"], label)


def adversarial_blocks_frame(rng=None):
    """A frame whose 8x8 blocks drive the intermediates of the round trip to their extremes: for every pair (u, v) the sign
    pattern of the 2-D basis function (u, v) at full swing (0 / 255) and its negative — these maximise the forward row / column
    outputs and, at coarse tables, the quantisation error that the inverse column pass amplifies — plus the rounded cosine itself,
    single-pixel impulses, and all of it again per channel in saturated colours (chroma blocks see the same patterns)."""
    import math

    blocks = []
    for u in range(8):
        for v in range(8):
            cu = [math.cos((2 * x + 1) * u * math.pi / 16) for x in range(8)]
            cv = [math.cos((2 * y + 1) * v * math.pi / 16) for y in range(8)]
            sign = np.array([[255 if cu[x] * cv[y] >= 0 else 0 for x in range(8)] for y in range(8)], np.uint8)
            cosb = np.array([[int(round(127.5 + 127.5 * cu[x] * cv[y])) for x in range(8)] for y in range(8)], np.uint8)
            blocks += [sign, 255 - sign, cosb, 255 - cosb]
    for k in range(8):
        imp = np.zeros((8, 8), np.uint8)
        imp[k, 7 - k] = 255
        blocks += [imp, 255 - imp]
    n = len(blocks)                                       # 272 luma blocks -> 17 x 16 blocks
    cols = 16
    rows = (n + cols - 1) // cols
    plane = np.zeros((8 * rows, 8 * cols), np.uint8)
    for i, b in enumerate(blocks):
        plane[8 * (i // cols):8 * (i // cols) + 8, 8 * (i % cols):8 * (i % cols) + 8] = b
    gray = np.repeat(plane[..., None], 3, axis=2)
    # chroma sees 2x2-averaged planes: upscale the patterns by two so that the chroma blocks get the same extremes
    big = np.kron(plane, np.ones((2, 2), np.uint8))
    col = np.zeros(big.shape + (3,), np.uint8)
    col[..., 0] = big                                     # red swings: Cr (and Cb) at full range
    col[..., 2] = 255 - big
    return gray, col
