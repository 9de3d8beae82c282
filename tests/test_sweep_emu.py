"""CPU: quality sweeps (v5ela_analyze_sweep, include/v5ela.h) — the host plan (csrc/v5ela_host.h plan_sweep) and the sweep kernel's
work items (process_work_item's SWEEP: per-entry quantisation tables, JPEG-ghost cells), both block-stage builds compiled by g++ with
threads emulated per barrier phase (tests/emu/v5ela_sweep_emu.cpp), against the C oracle. The GPU side is tests/test_gpu_sweep.py."""
import ctypes
import io
import os
import subprocess

import numpy as np
import pytest

from helpers import HERE
from oracle import c_oracle
from oracle.pil_oracle import RECORD_DTYPE
from v5ela._abi import FrameDesc
from v5ela.records import ghost_curve
from v5ela.synth import gen_frame

ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "fake-video-detection-engine_b200", "csrc")
u8p, i32p, u32p, i64p = (ctypes.POINTER(t) for t in (ctypes.c_uint8, ctypes.c_int, ctypes.c_uint32, ctypes.c_int64))


def build_emu(variant):
    so = os.path.join(HERE, "emu", f"libv5ela_sweep_emu_{variant}.so")
    src = os.path.join(HERE, "emu", "v5ela_sweep_emu.cpp")
    deps = [src, __file__] + [os.path.join(CSRC, f) for f in ("v5ela_device.cuh", "v5ela_dctmma.cuh", "v5ela_workitem.cuh", "v5ela_host.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        extra = ["-DV5_MMA_BLOCKS=1", "-DV5_MMA_NP=1"] if variant == "mma" else []
        tmp = f"{so}.{os.getpid()}.so"          # written aside, then renamed: parallel test processes never load a half-written file
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-DV5_MIN_CTAS=2", *extra,
                               "-I", os.path.join(ROOT, "include"), "-I", CSRC, src, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    lib.v5emu_analyze_sweep.argtypes = [u8p, i32p, ctypes.c_int, i32p, ctypes.c_int, ctypes.c_void_p, u32p, ctypes.c_int]
    lib.v5emu_plan_sweep.argtypes = [ctypes.POINTER(FrameDesc), ctypes.c_int, i32p, ctypes.c_int, u32p, ctypes.c_int, ctypes.c_int, i64p,
                                     i32p, i32p, ctypes.POINTER(ctypes.c_longlong), i32p, i32p]
    lib.v5emu_plan_ragged.argtypes = [i32p, ctypes.c_int, ctypes.c_int, ctypes.c_int, i32p, ctypes.POINTER(ctypes.c_longlong)]
    return lib


@pytest.fixture(scope="module", params=["smem", "mma"])
def emu(request):
    """Both builds of the block stage: shared-memory transposes and the tensor-core form (m16n8k16 fragments emulated lane by lane)."""
    return build_emu(request.param)


@pytest.fixture(scope="module")
def planner():
    return build_emu("smem")


def ghost_of(residual):
    """NumPy: per 16 x 16 MCU the sum over its image pixels of sum_c residual_c^2 (partial edge MCUs included)."""
    h, w, _ = residual.shape
    mh, mw = -(-h // 16), -(-w // 16)
    sq = np.zeros((16 * mh, 16 * mw), np.int64)
    sq[:h, :w] = (residual.astype(np.int64) ** 2).sum(axis=2)
    return sq.reshape(mh, 16, mw, 16).sum(axis=(1, 3))


def descs_of(sizes, ptr=lambda i: 4096 * (i + 1)):
    """Descriptors of frames `sizes` with made-up pixel pointers (the plan reads no pixel)."""
    d = (FrameDesc * max(len(sizes), 1))()
    for i, (h, w) in enumerate(sizes):
        d[i].rgb, d[i].height, d[i].width, d[i].row_stride_bytes = ptr(i), h, w, 3 * w
    return d


def plan_sweep(lib, descs, n, qualities, ghost=None, seg=0, target=0, nq=None):
    """-> (status, bad_frame, bad_quality, plan rows (n*nq, 6), slot qualities, total). qualities=None: a null array of nq."""
    nq = len(qualities) if nq is None else nq
    qs = np.array(qualities if qualities is not None else [90], np.int32)
    m = max(n * nq, 1)
    plan = np.zeros((m, 6), np.int64)
    slots = np.zeros(101, np.int32)
    n_slots, bad_f, bad_q, total = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0), ctypes.c_longlong(-1)
    rc = lib.v5emu_plan_sweep(descs, n, qs.ctypes.data_as(i32p) if qualities is not None else None, nq,
                              ctypes.cast(ghost, u32p) if ghost else None, seg, target, plan.ctypes.data_as(i64p), slots.ctypes.data_as(i32p),
                              ctypes.byref(n_slots), ctypes.byref(total), ctypes.byref(bad_f), ctypes.byref(bad_q))
    return rc, bad_f.value, bad_q.value, plan, list(slots[:n_slots.value]), total.value


def ragged_plan(lib, sizes, seg, target):
    hw = np.array(sizes, np.int32).reshape(-1)
    plan = np.zeros(3 * len(sizes), np.int32)
    total = ctypes.c_longlong(-1)
    assert lib.v5emu_plan_ragged(hw.ctypes.data_as(i32p), len(sizes), seg, target, plan.ctypes.data_as(i32p), ctypes.byref(total)) == 0
    return plan.reshape(-1, 3), total.value


SIZES = [(1, 1), (17, 33), (257, 301), (40, 1000), (1080, 1920), (9, 976)]


@pytest.mark.parametrize("seg,target", [(0, 0), (2, 0), (0, 592), (0, 20000)])
def test_plan_is_the_ragged_plan_of_the_expanded_list(planner, seg, target):
    """Work items, strips, segments and first items of every entry equal plan_ragged over the quality-major expanded list."""
    qualities = [90, 75, 90, 50]
    n = len(SIZES)
    rc, _, _, plan, _, total = plan_sweep(planner, descs_of(SIZES), n, qualities, seg=seg, target=target)
    assert rc == 0
    want, want_total = ragged_plan(planner, SIZES * len(qualities), seg, target)
    assert total == want_total
    assert np.array_equal(plan[:, 2:5], want)


def test_plan_entries_frames_slots_and_ghost_maps(planner):
    qualities = [75, 90, 75, 1, 100, 90]
    n = len(SIZES)
    base = 1 << 20
    rc, _, _, plan, slots, _ = plan_sweep(planner, descs_of(SIZES), n, qualities, ghost=base, target=592)
    assert rc == 0
    assert slots == [75, 90, 1, 100]                            # distinct qualities, in order of first appearance, share slots
    m = [(-(-h // 16)) * (-(-w // 16)) for h, w in SIZES]
    M = sum(m)
    for q, qual in enumerate(qualities):
        for i in range(n):
            row = plan[q * n + i]
            assert row[0] == 4096 * (i + 1)                     # frame i's pixels
            assert row[1] == slots.index(qual)
            assert row[5] == base + 4 * (q * M + sum(m[:i]))    # map (q, i) at element q * M + sum_{j<i} m_j
    _, _, _, plan, _, _ = plan_sweep(planner, descs_of(SIZES), n, qualities)
    assert not plan[:, 5].any()                                 # no ghost maps asked for


def test_plan_refusals(planner):
    ok = descs_of([(17, 33), (40, 48)])
    assert plan_sweep(planner, ok, 2, [90])[0] == 0
    assert plan_sweep(planner, ok, 0, [90])[0] == 0             # n == 0 is an empty call
    assert plan_sweep(planner, None, 2, [90])[:3] == (-1, -1, -1)
    assert plan_sweep(planner, ok, 2, None, nq=1)[:3] == (-1, -1, -1)
    assert plan_sweep(planner, ok, -1, [90])[:3] == (-1, -1, -1)
    assert plan_sweep(planner, ok, 2, [])[:3] == (-1, -1, -1)   # nq = 0
    assert plan_sweep(planner, ok, 2, [90] * 101)[:3] == (-1, -1, -1)
    assert plan_sweep(planner, ok, 2, [90] * 100)[0] == 0
    assert plan_sweep(planner, ok, 2, [90, 0, 75])[:3] == (-1, -1, 1)
    assert plan_sweep(planner, ok, 2, [90, 75, 101])[:3] == (-1, -1, 2)
    bad = [("rgb", 0), ("height", 0), ("width", 0), ("width", 65537), ("row_stride_bytes", 3 * 48 - 1)]
    for field, value in bad:
        d = descs_of([(17, 33), (40, 48)])
        setattr(d[1], field, value)
        assert plan_sweep(planner, d, 2, [90, 75])[:3] == (-1, 1, -1), field
    d = descs_of([(65536, 32768)])                              # 2^31 pixels: the per-frame counters are 32-bit
    d[0].row_stride_bytes = 3 * 32768
    assert plan_sweep(planner, d, 1, [90])[:3] == (-1, 0, -1)
    for field in ("residual", "enhanced"):
        d = descs_of([(17, 33), (40, 48)])
        setattr(d[0], field, 1 << 20)
        assert plan_sweep(planner, d, 2, [90])[:3] == (-1, 0, -1), field
    big = [(65536, 32767)] * 80                                 # 69 strips x 4096 one-row segments per entry, x 80 frames x 100 qualities
    assert plan_sweep(planner, descs_of(big), len(big), [90] * 100, seg=1)[:3] == (-1, -1, -1)
    assert plan_sweep(planner, descs_of(big), len(big), [90] * 10, seg=1)[0] == 0


EMU_SIZES = [(1, 1), (17, 33), (45, 61), (24, 520), (300, 40)]   # edge units (61), several strips (520), several segments (300)
EMU_QUALITIES = [1, 50, 75, 90, 100, 75]


def emu_frames():
    rng = np.random.default_rng(11)
    return [gen_frame(i, h, w, 4) if i % 2 == 0 else rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for i, (h, w) in enumerate(EMU_SIZES)]


@pytest.mark.parametrize("seg,target", [(0, 0), (2, 592)], ids=["0", "2-592"])
def test_emulated_sweep_vs_oracle(emu, seg, target):
    """Every record equals the oracle's analysis of that frame at that quality byte for byte, and every ghost map the NumPy block sums
    of the oracle's squared residual."""
    frames = emu_frames()
    n, nq = len(frames), len(EMU_QUALITIES)
    blob = np.concatenate([f.reshape(-1) for f in frames])
    hw = np.array(EMU_SIZES, np.int32).reshape(-1)
    qs = np.array(EMU_QUALITIES, np.int32)
    m = [(-(-h // 16)) * (-(-w // 16)) for h, w in EMU_SIZES]
    recs = np.zeros(n * nq, RECORD_DTYPE)
    ghost = np.full(nq * sum(m), 0xA5A5A5A5, np.uint32)
    try:
        emu.v5emu_set_target_items(target)
        rc = emu.v5emu_analyze_sweep(blob.ctypes.data_as(u8p), hw.ctypes.data_as(i32p), n, qs.ctypes.data_as(i32p), nq,
                                     recs.ctypes.data_as(ctypes.c_void_p), ghost.ctypes.data_as(u32p), seg)
    finally:
        emu.v5emu_set_target_items(0)
    assert rc == 0
    off = 0
    for q, qual in enumerate(EMU_QUALITIES):
        for i, f in enumerate(frames):
            o = c_oracle.analyze_frame(f, qual)
            assert recs[q * n + i].tobytes() == o["record"].tobytes(), (qual, f.shape)
            h, w, _ = f.shape
            assert np.array_equal(ghost[off:off + m[i]].reshape(-(-h // 16), -(-w // 16)), ghost_of(o["residual"])), (qual, f.shape)
            off += m[i]
    # without maps: the same records
    recs2 = np.zeros(n * nq, RECORD_DTYPE)
    assert emu.v5emu_analyze_sweep(blob.ctypes.data_as(u8p), hw.ctypes.data_as(i32p), n, qs.ctypes.data_as(i32p), nq,
                                   recs2.ctypes.data_as(ctypes.c_void_p), None, seg) == 0
    assert recs2.tobytes() == recs.tobytes()


def test_ghost_curve_is_the_mean_squared_residual():
    frames = [gen_frame(0, 40, 56, 1), gen_frame(1, 17, 33, 1)]
    recs = np.zeros((2, 2), RECORD_DTYPE)
    for q, qual in enumerate((60, 90)):
        for i, f in enumerate(frames):
            recs[q, i] = c_oracle.analyze_frame(f, qual)["record"]
    curve = ghost_curve(recs, [40 * 56, 17 * 33])
    assert curve.shape == (2, 2) and curve.dtype == np.float64
    for q, qual in enumerate((60, 90)):
        for i, f in enumerate(frames):
            r = c_oracle.analyze_frame(f, qual)["residual"].astype(np.float64)
            assert curve[q, i] == pytest.approx((r ** 2).mean(), rel=1e-12)


@pytest.mark.parametrize("q0", [60, 70, 85])
def test_ghost_minimum_at_the_earlier_quality(q0):
    """The JPEG-ghost premise on the oracle: frames decoded from Pillow files saved at q0 have their smallest mean squared residual at q0
    over q = 50, 55, ..., 95."""
    from PIL import Image

    grid = list(range(50, 100, 5))
    for seed in range(3):
        buf = io.BytesIO()
        Image.fromarray(gen_frame(0, 288, 352, seed)).save(buf, "JPEG", quality=q0)
        decoded = np.asarray(Image.open(io.BytesIO(buf.getvalue())).convert("RGB"))
        recs = np.zeros(len(grid), RECORD_DTYPE)
        for k, q in enumerate(grid):
            recs[k] = c_oracle.analyze_frame(decoded, q)["record"]
        curve = ghost_curve(recs, 288 * 352)
        assert grid[int(np.argmin(curve))] == q0, (seed, curve)
