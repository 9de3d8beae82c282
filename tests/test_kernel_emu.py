"""CPU: the CUDA kernel's device code (csrc/*.cuh), compiled by g++ with threads emulated per barrier phase
(tests/emu/v5ela_emu.cpp), against the oracle. Debug aid for band/halo/edge indexing in a container without a GPU;
the GPU parity tests (-m gpu) are the real gate."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import HERE, golden_frame, load_json, record_matches_golden, sha
from oracle import c_oracle
from oracle.pil_oracle import RECORD_DTYPE
from v5ela.synth import gen_frame

ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module", params=["2cta", "3cta", "2cta_rows_split", "2cta_mma", "2cta_mma_np2", "3cta_mma", "2cta_rev", "2cta_mma_rev", "2cta_fuse2", "2cta_fuse2_rev"])
def emu(request):
    """The default layout (2 CTAs/SM, double-buffered RGB), the -DV5_MIN_CTAS=3 single-buffer layout, and the default layout
    with the two compile-time variants of the width-multiple-of-16 instantiation flipped (one row per residual unit instead
    of two, split barrier on); "_mma": the tensor-core block stage (csrc/v5ela_dctmma.cuh, the library's second build of the
    kernel) with the m16n8k16 fragment layout emulated lane by lane, one or two pairs of blocks in flight per warp; "_rev": the
    emulated threads of every barrier-delimited phase run last to first (a read-after-overwrite inside a phase shows up in one of the two
    orders); "_fuse2": the two-phase band loop (-DV5_FUSE2=1, a compile-time variant: the residual stage of one band and the conversion
    of the next in the same phase), in both orders."""
    variant = request.param
    so = os.path.join(HERE, "emu", f"libv5ela_emu_{variant}.so")
    src = os.path.join(HERE, "emu", "v5ela_emu.cpp")
    csrc = os.path.join(ROOT, "fake-video-detection-engine_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("v5ela_device.cuh", "v5ela_dctmma.cuh", "v5ela_workitem.cuh", "v5ela_host.h")]
    deps.append(__file__)
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        extra = ["-DV5_PAIR_ROWS=0", "-DV5_SPLIT_BARRIER=1"] if variant.endswith("rows_split") else []
        if "_fuse2" in variant:
            extra += ["-DV5_FUSE2=1"]
        if variant.endswith("_rev"):
            extra += ["-DV5_EMU_REVERSE=1"]
        if "_mma" in variant:
            extra += ["-DV5_MMA_BLOCKS=1", "-DV5_MMA_NP=2" if "np2" in variant else "-DV5_MMA_NP=1"]
        tmp = f"{so}.{os.getpid()}.so"          # written aside, then renamed: parallel test processes never load a half-written file
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", f"-DV5_MIN_CTAS={variant[0]}", *extra,
                               "-I", os.path.join(ROOT, "include"), "-I", csrc, src, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    u8p = ctypes.POINTER(ctypes.c_uint8)
    lib.v5emu_analyze.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                  ctypes.c_int, ctypes.c_void_p, u8p, ctypes.c_int, ctypes.c_void_p]

    def run(frames, q, seg=0, want_residual=True, tex_hist=None):
        frames = np.ascontiguousarray(frames)
        n, h, w, _ = frames.shape
        recs = np.zeros(n, RECORD_DTYPE)
        res = np.zeros((n, h, w, 3), np.uint8) if want_residual else None
        rc = lib.v5emu_analyze(frames.ctypes.data_as(u8p), n, h, w, h * w * 3, w * 3, q,
                               recs.ctypes.data_as(ctypes.c_void_p), res.ctypes.data_as(u8p) if want_residual else None, seg,
                               tex_hist.ctypes.data_as(ctypes.c_void_p) if tex_hist is not None else None)
        assert rc == 0
        return recs, res

    run.lib = lib
    return run


def test_exact_division_constants(emu):
    assert emu.lib.v5emu_quant_selftest() == 0          # every table entry 1..255 x every coefficient -8192..8192


@pytest.mark.parametrize("hw", [(1, 1), (2, 3), (9, 1), (16, 16), (17, 33), (31, 9), (33, 497), (100, 1000), (272, 496)])
@pytest.mark.parametrize("seg", [0, 1, 3])
def test_emulated_kernel_vs_oracle(emu, hw, seg):
    h, w = hw
    rng = np.random.default_rng(h * 7 + w)
    for q in (90, 25):
        for frame in (gen_frame(3, h, w, 1), rng.integers(0, 256, (h, w, 3), dtype=np.uint8)):
            o = c_oracle.analyze_frame(frame, q)
            recs, res = emu(frame[None], q, seg)
            assert np.array_equal(res[0], o["residual"])
            assert recs[0].tobytes() == o["record"].tobytes()


@pytest.mark.parametrize("hw", [(1, 16), (2, 16), (15, 32), (16, 16), (17, 32), (31, 16), (32, 48), (33, 496), (40, 48), (100, 1008),
                                (272, 512), (9, 976)])
@pytest.mark.parametrize("seg", [0, 1, 2])
def test_emulated_fast_instantiation_vs_oracle(emu, hw, seg):
    """Statistics-only calls on widths that are a multiple of 16 take the kernel instantiation without the horizontal edge
    predicates (csrc/v5ela_host.h fast_path_ok); same records as the oracle and as the general instantiation."""
    h, w = hw
    rng = np.random.default_rng(h * 11 + w)
    for q in (90, 40):
        for frame in (gen_frame(5, h, w, 2), rng.integers(0, 256, (h, w, 3), dtype=np.uint8)):
            o = c_oracle.analyze_frame(frame, q)
            recs, _ = emu(frame[None], q, seg, want_residual=False)
            assert recs[0].tobytes() == o["record"].tobytes()
            general, _ = emu(frame[None], q, seg)
            assert general[0].tobytes() == recs[0].tobytes()


@pytest.mark.parametrize("hw", [(1, 1), (1, 7), (9, 1), (16, 16), (17, 33), (40, 48), (33, 497), (100, 1000)])
def test_emulated_texture_histogram(emu, hw):
    """The optional tex_hist[256] output (SURVEY.md §8a) against OpenCV's Laplacian of Pillow's luma; the record and the
    residual map of the same call stay what they are without it."""
    from oracle import pil_oracle

    h, w = hw
    rng = np.random.default_rng(h * 13 + w)
    for frame in (gen_frame(2, h, w, 3), rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
                  np.where(rng.integers(0, 2, (h, w, 1)) > 0, 255, 0).astype(np.uint8).repeat(3, axis=2)):   # saturates the last bin
        for want_residual in (False, True):
            th = np.full((1, 256), 0xA5A5A5A5, np.uint32)
            recs, res = emu(frame[None], 90, 0, want_residual=want_residual, tex_hist=th)
            assert np.array_equal(th[0], pil_oracle.texture_hist(frame))
            assert int(th[0].sum()) == h * w
            o = c_oracle.analyze_frame(frame, 90)
            assert recs[0].tobytes() == o["record"].tobytes()
            if want_residual:
                assert np.array_equal(res[0], o["residual"])


def test_emulated_texture_histogram_goldens(emu):
    """tests/golden/layouts_golden.json: tex_hist recorded from OpenCV's Laplacian of Pillow's luma."""
    for case in load_json("layouts_golden.json")["cases"]:
        th = np.zeros((1, 256), np.uint32)
        emu(golden_frame(case)[None], 90, 0, want_residual=False, tex_hist=th)
        assert sha(th[0]) == case["tex_hist_sha"] and [int(v) for v in th[0][:8]] == case["tex_hist_head"]
        assert int(th[0][255]) == case["tex_hist_last"]


def test_emulated_kernel_vs_reference_goldens(emu):
    cases = [c for c in load_json("frames_golden.json")["cases"] if c["h"] * c["w"] <= 64 * 96]
    assert len(cases) > 20
    for case in cases:
        recs, res = emu(golden_frame(case)[None], case["q"])
        assert sha(res[0]) == case["resid_sha"]
        assert record_matches_golden(recs[0], case) == []


@pytest.mark.parametrize("seg", [0, 2])
def test_emulated_ragged_instantiation_vs_oracle(emu, seg):
    """v5ela_analyze_ragged's kernel instantiation: frames of different sizes share one work-item space (binary search over the
    frame table per work item); every frame against the oracle."""
    import ctypes

    sizes = [(1, 1), (17, 33), (16, 16), (40, 48), (33, 497), (9, 976), (100, 1000), (2, 3)]
    rng = np.random.default_rng(7)
    frames = [gen_frame(i, h, w, 2) if i % 2 == 0 else rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for i, (h, w) in enumerate(sizes)]
    blob = np.concatenate([f.reshape(-1) for f in frames])
    hw = np.array(sizes, np.int32).reshape(-1)
    recs = np.zeros(len(sizes), RECORD_DTYPE)
    res = np.zeros_like(blob)
    u8p = ctypes.POINTER(ctypes.c_uint8)
    rc = emu.lib.v5emu_analyze_ragged(blob.ctypes.data_as(u8p), hw.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), len(sizes), 90,
                                      recs.ctypes.data_as(ctypes.c_void_p), res.ctypes.data_as(u8p), seg)
    assert rc == 0
    off = 0
    for i, f in enumerate(frames):
        o = c_oracle.analyze_frame(f, 90)
        assert recs[i].tobytes() == o["record"].tobytes(), sizes[i]
        assert np.array_equal(res[off:off + f.size].reshape(f.shape), o["residual"]), sizes[i]
        off += f.size


@pytest.mark.parametrize("hw", [(257, 301), (40, 1000), (64, 96), (300, 48)])
def test_emulated_small_batch_decomposition(emu, hw):
    """Batches that cannot fill the GPU get short segments and narrow strips (csrc/v5ela_host.h fill_params / widen_strips: down to
    4 MCU rows x 4 MCU columns per work item); same records and residual map as the default decomposition and the oracle."""
    h, w = hw
    frame = gen_frame(1, h, w, 7)
    o = c_oracle.analyze_frame(frame, 90)
    try:
        emu.lib.v5emu_set_target_items(592)                  # 2 x 148 SMs x 2 CTAs
        for want_residual in (True, False):
            recs, res = emu(frame[None], 90, 0, want_residual=want_residual)
            assert recs[0].tobytes() == o["record"].tobytes()
            if want_residual:
                assert np.array_equal(res[0], o["residual"])
    finally:
        emu.lib.v5emu_set_target_items(0)


def test_emulated_two_regime_decomposition(emu):
    """A batch with plenty of work is cut into long segments (whole-height strips) except for its last frames, which get short
    segments so that the launch's tail is short (csrc/v5ela_host.h fill_params: split_frame / n_segs_b): every frame of both
    regimes against the oracle."""
    frames = np.stack([gen_frame(i, 300, 32, 3) for i in range(40)])          # 19 MCU rows: long = 1 segment of 19, short = 3 segments of <= 8
    orecs, oresid = c_oracle.analyze(frames, 90, want_residual=True)
    try:
        emu.lib.v5emu_set_target_items(16)                   # 8 "CTAs": 40 columns >= 3 x 8 -> long segments; the last 4 frames short
        for want_residual in (True, False):
            recs, res = emu(frames, 90, 0, want_residual=want_residual)
            assert recs.tobytes() == orecs.tobytes()
            if want_residual:
                assert np.array_equal(res, oresid)
            assert emu.lib.v5emu_last_split_frame() == 36 and emu.lib.v5emu_last_segments(0) == 1 and emu.lib.v5emu_last_segments(1) == 3
    finally:
        emu.lib.v5emu_set_target_items(0)


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


@pytest.mark.parametrize("q", [1, 2, 25, 50, 90, 100])
def test_adversarial_ranges_of_the_int16_hand_offs(emu, q):
    """The block stage hands 16-bit intermediates from pass to pass (shared-memory int16 pairs in one build, 8-bit limb pairs in
    the tensor-core build): |forward row output| <= 4096, |coefficient| <= 8192 (the exact division's domain), |inverse column
    output| <= 21047 (DESIGN.md 4.1) must hold for blocks built to maximise them, at the coarsest (q=1, T=255) and the finest
    (q=100, T=1) tables — a silent wrap would be a parity bug. The tensor-core emulation counts every violation; both builds
    must reproduce Pillow bit for bit."""
    from oracle import pil_oracle

    for frame in adversarial_blocks_frame():
        rec, resid = pil_oracle.record(frame, q, with_residual=True)
        recs, res = emu(frame[None], q, 0)
        assert np.array_equal(res[0], resid)
        assert recs[0].tobytes() == rec.tobytes()
        if frame.shape[1] % 16 == 0:
            fast, _ = emu(frame[None], q, 0, want_residual=False)
            assert fast[0].tobytes() == rec.tobytes()
    emu.lib.v5emu_range_violations.restype = __import__("ctypes").c_longlong
    assert emu.lib.v5emu_range_violations() == 0


def test_no_range_violations_after_the_whole_module(emu):
    """Runs last: everything this module pushed through the tensor-core emulation stayed inside the limb ranges."""
    import ctypes

    emu.lib.v5emu_range_violations.restype = ctypes.c_longlong
    assert emu.lib.v5emu_range_violations() == 0
