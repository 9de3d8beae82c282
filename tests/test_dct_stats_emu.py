"""CPU: the DCT-statistics kernels' host/device-shared logic (csrc/v5jpeg_dct.cuh), compiled by g++ with the CTAs, warps and lanes
emulated (tests/emu/v5jpeg_dct_emu.cpp), over the oracle decoder's coefficients, against NumPy: histograms and periods identical,
maps within 1e-6. Also jpeg.ijg_quality (host only). The -m gpu tests (test_gpu_dct_stats.py) run the kernels themselves."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from dct_helpers import layout_files, luma_grid, np_hist, odd_size_files, pil_bytes, qtab_of
from helpers import HERE
from v5ela import records

ROOT = os.path.dirname(HERE)
CASES = layout_files()
ODD = odd_size_files(np.random.default_rng(2026), 40)


@pytest.fixture(scope="module")
def emu():
    so = os.path.join(HERE, "emu", "libv5jpeg_dct_emu.so")
    src = os.path.join(HERE, "emu", "v5jpeg_dct_emu.cpp")
    csrc = os.path.join(ROOT, "fake-video-detection-engine_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("v5jpeg_dct.cuh", "v5jpeg_dec.cuh", "v5jpeg_common.h", "v5ela_device.cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = f"{so}.{os.getpid()}.so"          # written aside, then renamed: parallel test processes never load a half-written file
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-I",
                               os.path.join(ROOT, "include"), "-I", csrc, src, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    vp = ctypes.c_void_p
    lib.v5jdct_emu_stats.argtypes = [vp, ctypes.c_int64, vp, vp, vp, vp, vp, vp]
    lib.v5jdct_emu_period.argtypes = [vp, vp]
    lib.v5jdct_emu_twiddles.argtypes = [vp, vp]
    return lib


def emu_stats(emu, data):
    from dct_helpers import oracle_blocks

    coef, h, w, *_ = oracle_blocks(data)
    coef = np.ascontiguousarray(coef)
    buf = np.frombuffer(data, np.uint8)
    hist = np.zeros((3, 64, 129), np.uint32)
    qtab = np.zeros((3, 64), np.uint16)
    period = np.zeros(15, np.int32)
    lut = np.zeros((15, 130))
    m = np.zeros(((h + 7) // 8, (w + 7) // 8), np.float32)
    rc = emu.v5jdct_emu_stats(buf.ctypes.data, len(data), coef.ctypes.data, hist.ctypes.data, qtab.ctypes.data, period.ctypes.data,
                              lut.ctypes.data, m.ctypes.data)
    assert rc == 0
    return hist, qtab, period, m


def check_file(emu, data):
    hist, qtab, period, m = emu_stats(emu, data)
    want = np_hist(data)
    assert np.array_equal(hist, want)
    assert np.array_equal(qtab, qtab_of(data))
    assert np.array_equal(period, records.dq_periods(want))
    ref = records.dq_map(want, luma_grid(data))
    assert m.shape == ref.shape and np.abs(m.astype(np.float64) - ref).max() <= 1e-6
    return period


@pytest.mark.parametrize("label,data", CASES, ids=[c[0] for c in CASES])
def test_layouts_against_numpy(emu, label, data):
    check_file(emu, data)


@pytest.mark.parametrize("label,data", ODD, ids=[c[0] for c in ODD])
def test_odd_sizes_against_numpy(emu, label, data):
    check_file(emu, data)


def test_multi_chunk_file_against_numpy(emu):
    """A file of more blocks than one dct_hist_kernel CTA takes (DQ_CHUNK = 4096): 720p 4:2:0 has 21600."""
    from v5ela.synth import gen_frame

    data = pil_bytes(gen_frame(3, 720, 1280, 0), 85)
    period = check_file(emu, data)
    assert period.shape == (15,)


def test_twiddle_tables_match(emu):
    """The GPU multiplies the same doubles as records.dq_periods, and they are cos / sin (2 pi j / p)."""
    c, s = np.zeros(77), np.zeros(77)
    emu.v5jdct_emu_twiddles(c.ctypes.data, s.ctypes.data)
    assert c.tobytes() == np.array(records.DQ_COS).tobytes() and s.tobytes() == np.array(records.DQ_SIN).tobytes()
    i = 0
    for p in range(2, 13):
        j = np.arange(p)
        assert np.allclose(c[i:i + p], np.cos(2 * np.pi * j / p), atol=1e-15, rtol=0)
        assert np.allclose(s[i:i + p], np.sin(2 * np.pi * j / p), atol=1e-15, rtol=0)
        i += p


def test_period_rule_on_synthetic_histograms(emu):
    """The per-warp period decision against NumPy on histograms with planted periods, noise, ties and too few values."""
    rng = np.random.default_rng(7)
    hists = []
    v = np.arange(-64, 65)
    for p in range(2, 13):
        base = np.exp(-np.abs(v) / 6.0) * 5000
        h = base * (np.mod(v, p) == 0) + rng.poisson(3, v.size)
        hists.append(h)
    hists += [rng.poisson(40, v.size), np.zeros(129), np.full(129, 7), (np.exp(-np.abs(v) / 3.0) * 900)]
    hists += [np.where(np.abs(v) == 3, 20, 0), np.where(np.abs(v) <= 1, 10 ** 6, 0)]
    for _ in range(200):
        q = int(rng.integers(1, 13))
        h = np.exp(-np.abs(v) / rng.uniform(1, 20)) * rng.uniform(10, 1e5)
        h = np.where(np.mod(v, q) == 0, h, h * rng.uniform(0, 1))
        hists.append(rng.poisson(h))
    found = set()
    for h in hists:
        h = np.ascontiguousarray(np.asarray(h).astype(np.uint32))
        row = np.zeros(130)
        p = emu.v5jdct_emu_period(h.ctypes.data, row.ctypes.data)
        assert p == records._dq_period(h)
        ref = records._dq_lut(h, p)
        assert np.array_equal(np.isinf(row), np.isinf(ref))
        fin = np.isfinite(ref)
        assert np.abs(row[fin] - ref[fin]).max() <= 1e-12
        found.add(p)
    assert {1, 2, 3, 4, 5, 12} <= found, found       # (a comb of period 8 also scores fully at 4: the smaller p wins)


def test_ijg_quality_round_trips_pillow_files():
    from v5ela import jpeg

    rgb = np.random.default_rng(3).integers(0, 256, (24, 40, 3), dtype=np.uint8)
    for q in range(1, 101):
        assert jpeg.ijg_quality(qtab_of(pil_bytes(rgb, q))) == q
        assert jpeg.ijg_quality(qtab_of(pil_bytes(np.ascontiguousarray(rgb[..., 0]), q))) == q       # one component: luma only
    custom = qtab_of(pil_bytes(rgb, 75))
    custom[0, 5] += 1
    assert jpeg.ijg_quality(custom) is None
    tabs = qtab_of(pil_bytes(rgb, 60))
    assert jpeg.ijg_quality(tabs[:2]) == 60 and jpeg.ijg_quality(tabs[0]) == 60
    tabs[2, 0] += 1
    assert jpeg.ijg_quality(tabs) is None                           # Cb and Cr tables differ: not an IJG pair
