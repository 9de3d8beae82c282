"""CPU: the host plan of ragged spectrum calls (csrc/v5ela_spec_plan.h, compiled by g++ behind tests/emu/v5ela_spec_emu.cpp):
the per-image choice between the Stockham FFT and the exact-size DFT, the CTA lookup of every ragged launch, workspace ranges,
twiddle-table de-duplication, chunking and refusals. The -m gpu tests (test_gpu_spectrum_ragged.py) check the images."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from helpers import HERE

ROOT = os.path.dirname(HERE)
L_FFT_ROWS, L_FFT_COLS, L_DFT_ROWS, L_DFT_COLS, L_IMAGE = range(5)
CAP = 1 << 30


class GrayDesc(ctypes.Structure):
    _fields_ = [("gray", ctypes.c_void_p), ("height", ctypes.c_int32), ("width", ctypes.c_int32), ("row_stride_bytes", ctypes.c_int64),
                ("out", ctypes.c_void_p)]


@pytest.fixture(scope="module")
def lib():
    so = os.path.join(HERE, "emu", "libv5ela_spec_emu.so")
    src = os.path.join(HERE, "emu", "v5ela_spec_emu.cpp")
    csrc = os.path.join(ROOT, "fake-video-detection-engine_b200", "csrc")
    deps = [src, os.path.join(csrc, "v5ela_spec_plan.h"), os.path.join(ROOT, "include", "v5ela.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = f"{so}.{os.getpid()}.so"          # written aside, then renamed: parallel test processes never load a half-written file
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", csrc, src, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    i64p, i32p, ip = ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int)
    lib.v5semu_fft_path.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ip]
    lib.v5semu_plan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ip]
    lib.v5semu_error.restype = ctypes.c_char_p
    lib.v5semu_counts.argtypes = [i64p]
    lib.v5semu_frame.argtypes = [ctypes.c_int, i64p]
    lib.v5semu_size.argtypes = [ctypes.c_int, i64p]
    lib.v5semu_chunk.argtypes = [ctypes.c_int, i64p]
    lib.v5semu_walk.argtypes = [ctypes.c_int, ctypes.c_int, i32p, i32p]
    return lib


def smooth(n):
    for p in (2, 3, 5):
        while n % p == 0:
            n //= p
    return n == 1


def uniform_rule(h, w, fft_on=True):
    """v5ela_spectrum's choice, restated: both sides made of 2, 3 and 5, and both FFT passes within 200 KB of shared memory."""
    cc = (96 << 10) // (32 * h)
    cc = 4 if cc >= 4 else (2 if cc >= 2 else cc)
    return fft_on and smooth(w) and smooth(h) and cc >= 1 and 32 * w <= 200 << 10 and 32 * cc * h <= 200 << 10, cc


def ceil(a, b):
    return (a + b - 1) // b


def descs_of(sizes, stride_pad=0):
    d = (GrayDesc * len(sizes))()
    for i, (h, w) in enumerate(sizes):
        d[i].gray, d[i].out = 0x1000 + i, 0x100000 + i          # never dereferenced by the plan
        d[i].height, d[i].width, d[i].row_stride_bytes = h, w, w + stride_pad
    return d


class Plan:
    def __init__(self, lib, sizes, fft_on=True, cap=CAP):
        self.lib, self.sizes = lib, sizes
        bad = ctypes.c_int(0)
        self.status = lib.v5semu_plan(descs_of(sizes), len(sizes), 1 if fft_on else 0, cap, ctypes.byref(bad))
        self.bad = bad.value
        if self.status:
            return
        c = np.zeros(5, np.int64)
        lib.v5semu_counts(c.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
        self.n_frames, self.n_sizes, self.n_chunks, self.launches, self.tw_elems = (int(v) for v in c)
        self.frames = [self._get(lib.v5semu_frame, i, 12, "h w wh cc g_off ms_off sw sh mm gx bx by") for i in range(self.n_frames)]
        self.tsizes = [self._get(lib.v5semu_size, k, 3, "n tw fft") for k in range(self.n_sizes)]
        self.chunks = [self._get(lib.v5semu_chunk, k, 12, "f0 n g_elems ms_elems c0 c1 c2 c3 c4 rows_smem cols_smem launches")
                       for k in range(self.n_chunks)]

    @staticmethod
    def _get(fn, i, k, names):
        a = np.zeros(k, np.int64)
        fn(i, a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
        return dict(zip(names.split(), (int(v) for v in a)))

    def walk(self, c, kind):
        n = self.chunks[c][f"c{kind}"] if kind >= 0 else sum(ceil(s["n"], 256) for s in self.tsizes)
        fr, lo = np.zeros(n, np.int32), np.zeros(n, np.int32)
        self.lib.v5semu_walk(c, kind, fr.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), lo.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
        return list(zip(fr.tolist(), lo.tolist()))


RULE_SIZES = [(1, 1), (2, 3), (1, 9), (9, 1), (45, 2), (257, 301), (211, 173), (486, 250), (360, 640), (1080, 1920), (2160, 3840)]


@pytest.mark.parametrize("fft_on", [True, False])
def test_path_choice_is_the_uniform_rule(lib, fft_on):
    p = Plan(lib, RULE_SIZES, fft_on=fft_on)
    assert p.status == 0
    for (h, w), f in zip(RULE_SIZES, p.frames):
        fast, cc = uniform_rule(h, w, fft_on)
        got_cc = ctypes.c_int(0)
        assert lib.v5semu_fft_path(1 if fft_on else 0, h, w, ctypes.byref(got_cc)) == int(fast), (h, w)
        assert f["cc"] == (cc if fast else 0), (h, w)
    if not fft_on:
        assert all(f["cc"] == 0 for f in p.frames)
    else:
        assert [f["cc"] > 0 for f in p.frames] == [True, True, True, True, True, False, False, True, True, True, True]


MIXED = [(1, 1), (1, 300), (300, 1), (2, 3), (257, 301), (211, 173), (45, 2), (360, 640), (127, 255), (97, 89), (1, 9), (9, 1), (64, 400),
         (400, 64), (2, 2), (125, 243)]


def expected_ctas(f, kind):
    fast = f["cc"] > 0
    if kind == L_FFT_ROWS:
        return ceil(f["h"], 2) if fast else 0
    if kind == L_FFT_COLS:
        return ceil(f["wh"], f["cc"]) if fast else 0
    if kind in (L_DFT_ROWS, L_DFT_COLS):
        return 0 if fast else ceil(f["wh"], 32) * ceil(f["h"], 32)
    return ceil(f["w"], 256) * min(ceil(f["h"], 16), 65535)


@pytest.mark.parametrize("fft_on", [True, False])
@pytest.mark.parametrize("cap", [CAP, 1 << 20])
def test_cta_lookup_covers_every_unit_once(lib, fft_on, cap):
    p = Plan(lib, MIXED, fft_on=fft_on, cap=cap)
    assert p.status == 0
    for c, C in enumerate(p.chunks):
        frames = p.frames[C["f0"]:C["f0"] + C["n"]]
        for kind in range(5):
            visited = p.walk(c, kind)
            want = [(j, loc) for j, f in enumerate(frames) for loc in range(expected_ctas(f, kind))]
            assert sorted(visited) == want, (c, kind)           # every unit, each exactly once, in frame order
            assert visited == want
    # the twiddle launch: ceil(n / 256) CTAs per distinct side
    tw = p.walk(0, -1)
    assert tw == [(k, loc) for k, s in enumerate(p.tsizes) for loc in range(ceil(s["n"], 256))]


@pytest.mark.parametrize("cap", [CAP, 1 << 20, 64 << 10])
def test_workspace_ranges_are_disjoint_and_aligned(lib, cap):
    p = Plan(lib, MIXED + [(1080, 1920)], cap=cap)
    assert p.status == 0
    for C in p.chunks:
        frames = p.frames[C["f0"]:C["f0"] + C["n"]]
        assert [f["mm"] for f in frames] == list(range(C["n"]))
        for key, unit, total in (("g_off", 16, "g_elems"), ("ms_off", 8, "ms_elems")):
            spans = sorted((f[key], f[key] + f["h"] * f["wh"]) for f in frames)
            for a, b in spans:
                assert (a * unit) % 256 == 0 and b <= C[total]
            for (a0, b0), (a1, _) in zip(spans, spans[1:]):
                assert b0 <= a1


def test_twiddle_tables_are_shared_between_equal_sides(lib):
    sizes = [(257, 301), (301, 257), (257, 257), (100, 301), (7, 7), (1, 100)]
    p = Plan(lib, sizes)
    assert p.status == 0
    ns = [s["n"] for s in p.tsizes]
    assert sorted(ns) == sorted({v for hw in sizes for v in hw}) and len(ns) == len(set(ns))
    for (h, w), f in zip(sizes, p.frames):
        assert p.tsizes[f["sw"]]["n"] == w and p.tsizes[f["sh"]]["n"] == h
    tw = sorted((s["tw"], s["n"]) for s in p.tsizes)
    assert tw[0][0] == 0 and all(a + n == b for (a, n), (b, _) in zip(tw, tw[1:])) and p.tw_elems == sum(ns)
    assert [s["fft"] for s in p.tsizes] == [int(smooth(n)) for n in ns]


def frame_bytes(h, w):
    s = h * (w // 2 + 1)
    return 16 * ceil(s, 16) * 16 + 8 * ceil(s, 32) * 32


def test_chunks_keep_frame_order_under_the_cap(lib):
    sizes = [(64, 64)] * 5 + [(400, 400)] + [(32, 48)] * 7 + [(300, 200), (10, 10)]
    cap = 3 * frame_bytes(64, 64)
    assert frame_bytes(400, 400) > cap
    p = Plan(lib, sizes, cap=cap)
    assert p.status == 0
    assert [C["f0"] for C in p.chunks] == [sum(C["n"] for C in p.chunks[:k]) for k in range(p.n_chunks)]
    assert sum(C["n"] for C in p.chunks) == len(sizes)
    for k, C in enumerate(p.chunks):
        used = sum(frame_bytes(*sizes[i]) for i in range(C["f0"], C["f0"] + C["n"]))
        assert used <= cap or C["n"] == 1
        if k + 1 < p.n_chunks:                                  # a chunk ends only where the next frame would not fit
            assert used + frame_bytes(*sizes[C["f0"] + C["n"]]) > cap
    big = [C for C in p.chunks if C["f0"] == 5]
    assert len(big) == 1 and big[0]["n"] == 1                   # the oversize frame is alone
    assert Plan(lib, sizes).n_chunks == 1


def test_launch_counts(lib):
    node = [(257, 301), (211, 173), (127, 255)]                 # no side made of 2, 3 and 5 only: DFT for all
    assert Plan(lib, node).launches == 4
    for n in (2, 5, 40):
        mixed = [(360, 640), (257, 301)] * (n // 2) + [(97, 89)] * (n % 2)
        assert Plan(lib, mixed).launches == 6, n
    assert Plan(lib, [(360, 640), (120, 160)]).launches == 4
    assert Plan(lib, [(360, 640), (257, 301)], fft_on=False).launches == 4
    p = Plan(lib, MIXED, cap=1 << 20)
    assert p.n_chunks > 1 and p.launches == 1 + sum(C["launches"] for C in p.chunks)


def test_refusals_name_the_frame(lib):
    good = [(20, 30), (5, 7), (9, 9)]
    bad = ctypes.c_int(0)

    def plan(descs, n):
        return lib.v5semu_plan(descs, n, 1, CAP, ctypes.byref(bad)), bad.value, lib.v5semu_error().decode()

    assert plan(None, 3)[0] == -1
    d = descs_of(good)
    assert plan(d, -1)[0] == -1
    assert plan(d, 0)[0] == 0 and plan(d, 3)[0] == 0
    cases = [("gray", 0, "null pointer"), ("out", 0, "null pointer"), ("height", 0, "non-positive size"), ("width", -4, "non-positive size"),
             ("height", 65537, "side over 65536"), ("width", 70000, "side over 65536"), ("row_stride_bytes", 8, "row stride smaller than the width")]
    for idx in range(3):
        for field, value, why in cases:
            d = descs_of(good)
            if field == "row_stride_bytes":
                d[idx].width = 9
            setattr(d[idx], field, value)
            assert plan(d, 3) == (-1, idx, why), (idx, field)
    d = descs_of(good)
    d[1].width, d[1].row_stride_bytes = 65536, 65536           # the largest side is accepted
    assert plan(d, 3)[0] == 0
