"""GPU: ragged spectrum calls (v5ela_spectrum_ragged / _host, include/v5ela.h) — images of different sizes in one launch sequence.
Every image must be byte-identical to v5ela_spectrum of that image alone, on both paths (FFT / DFT) and across chunks, and within
one grey level of NumPy (oracle/pil_oracle.fft_spectrum)."""
import ctypes

import numpy as np
import pytest

from oracle import pil_oracle
from v5ela.synth import gen_frame

pytestmark = pytest.mark.gpu

# the path-choice sizes of tests/test_spectrum_plan.py, primes, and node-like crops (V1's padded face boxes)
SIZES = [(1, 1), (2, 3), (1, 9), (9, 1), (45, 2), (257, 301), (211, 173), (486, 250), (360, 640), (1080, 1920), (2160, 3840),
         (97, 89), (127, 255), (199, 151), (1, 331)]


def images(sizes, seed=0):
    rng = np.random.default_rng(seed)
    out = []
    for k, (h, w) in enumerate(sizes):
        if k % 2:
            out.append(rng.integers(0, 256, (h, w), dtype=np.uint8))
        else:
            out.append(pil_oracle.luma(gen_frame(k, h, w, seed)))
    return out


def uniform(t):
    import v5ela

    return v5ela.spectrum_batch(t[None])[0]


def ragged(ts):
    import v5ela

    return v5ela.spectrum_ragged(ts)


@pytest.fixture
def env(monkeypatch):
    return monkeypatch


@pytest.mark.parametrize("mode", ["default", "dft", "chunks"])
def test_byte_identical_to_the_uniform_call(env, mode):
    import torch

    if mode == "dft":
        env.setenv("V5ELA_FFT", "0")
    if mode == "chunks":
        env.setenv("V5ELA_SPEC_CHUNK_MB", "1")                  # the larger images need more: several chunks, some of one image
    ts = [torch.from_numpy(a).cuda() for a in images(SIZES, seed=len(mode))]
    outs = ragged(ts)
    want = [uniform(t) for t in ts]
    torch.cuda.synchronize()
    assert len(outs) == len(ts)
    for (h, w), o, u in zip(SIZES, outs, want):
        assert o.shape == (h, w) and o.dtype == torch.uint8
        assert torch.equal(o, u), (mode, h, w)


def test_within_one_level_of_numpy():
    import torch

    sizes = [hw for hw in SIZES if hw[0] * hw[1] <= 1080 * 1920]
    arrs = images(sizes, seed=7)
    outs = ragged([torch.from_numpy(a).cuda() for a in arrs])
    for a, o in zip(arrs, outs):
        ref = pil_oracle.fft_spectrum(a)
        d = np.abs(o.cpu().numpy().astype(np.int16) - ref.astype(np.int16))
        assert int(d.max()) <= 1, a.shape
        if a.size > 1000:
            assert float((d == 0).mean()) >= 0.999, a.shape


def test_strided_views_and_odd_row_strides():
    import torch

    plane = torch.from_numpy(pil_oracle.luma(gen_frame(4, 720, 1280, 1))).cuda()
    boxes = [(0, 0, 720, 1280), (13, 7, 300, 411), (400, 1000, 720, 1280), (100, 100, 101, 101), (5, 640, 250, 1279), (719, 0, 720, 1280),
             (0, 1279, 720, 1280), (333, 222, 590, 523)]
    views = [plane[y1:y2, x1:x2] for (y1, x1, y2, x2) in boxes]
    rng = np.random.default_rng(3)
    for h, w in ((61, 77), (120, 160), (33, 1)):
        wide = torch.from_numpy(rng.integers(0, 256, (h, w + 3), dtype=np.uint8)).cuda()
        views.append(wide[:, 1:1 + w])                          # row stride w + 3 (odd for even w), unaligned start
    outs = ragged(views)
    for v, o in zip(views, outs):
        assert torch.equal(o, uniform(v.contiguous())), tuple(v.shape)


def test_host_entry_point_gives_the_device_bytes():
    import torch
    from v5ela import host

    arrs = images(SIZES[:10] + SIZES[11:], seed=2)
    arrs.append(np.ascontiguousarray(images([(90, 130)], seed=4)[0])[5:80, 3:101])   # strided host view
    got = host.spectrum_ragged_host(arrs)
    dev = ragged([torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs])
    for a, g, d in zip(arrs, got, dev):
        assert g.shape == a.shape and np.array_equal(g, d.cpu().numpy()), a.shape
    assert host.spectrum_ragged_host([]) == []


def _handle():
    import torch
    from v5ela.batch import get_handle

    return get_handle(torch.cuda.current_device())


def test_launch_counts():
    import torch

    hd = _handle()
    node = [torch.from_numpy(a).cuda() for a in images([(257, 301), (211, 173), (127, 255)])]
    c0 = hd.launch_count
    ragged(node)
    assert hd.launch_count - c0 == 4                            # twiddles, DFT rows, DFT columns, image
    for n in (2, 6, 24):
        mixed = [torch.from_numpy(a).cuda() for a in images([(360, 640), (257, 301)] * (n // 2))]
        c0 = hd.launch_count
        outs = ragged(mixed)
        assert hd.launch_count - c0 == 6, n                      # + FFT rows, FFT columns
        assert torch.equal(outs[0], uniform(mixed[0])) and torch.equal(outs[-1], uniform(mixed[-1]))


def test_uniform_twiddle_cache_survives_a_ragged_call():
    import torch

    a = torch.from_numpy(images([(211, 173)], seed=9)[0]).cuda()
    first = uniform(a).clone()
    ragged([torch.from_numpy(x).cuda() for x in images([(97, 89), (173, 211), (360, 640), (1, 211)], seed=1)])
    again = uniform(a)
    torch.cuda.synchronize()
    assert torch.equal(first, again)


def test_bad_descriptors_are_refused_before_any_launch():
    import torch
    from v5ela import _abi

    hd = _handle()
    src = torch.zeros((40, 50), dtype=torch.uint8, device="cuda")
    dst = torch.empty((40, 50), dtype=torch.uint8, device="cuda")

    def descs(n=3):
        d = (_abi.GrayDesc * n)()
        for i in range(n):
            d[i].gray, d[i].out = src.data_ptr(), dst.data_ptr()
            d[i].height, d[i].width, d[i].row_stride_bytes = 40, 50, 50
        return d

    stream = torch.cuda.current_stream().cuda_stream
    cases = [("gray", None), ("out", None), ("height", 0), ("width", -1), ("height", 65537), ("width", 65537), ("row_stride_bytes", 49)]
    for idx in (0, 2):
        for field, value in cases:
            d = descs()
            setattr(d[idx], field, value)
            c0 = hd.launch_count
            with pytest.raises(_abi.V5ElaError) as ei:
                hd.spectrum_ragged(d, 3, stream)
            assert ei.value.status == -1 and f"frame {idx}:" in str(ei.value), (idx, field)
            assert hd.launch_count == c0
            with pytest.raises(_abi.V5ElaError) as ei:
                hd.spectrum_ragged_host(d, 3)                   # host pointers expected, but refused before any copy
            assert ei.value.status == -1 and f"frame {idx}:" in str(ei.value), (idx, field)
            assert hd.launch_count == c0
    lib = _abi.load()
    assert lib.v5ela_spectrum_ragged(hd._h, None, 2, None) == -1
    assert lib.v5ela_spectrum_ragged(hd._h, descs(), -1, None) == -1
    assert lib.v5ela_spectrum_ragged(hd._h, None, 0, None) == 0
    assert lib.v5ela_spectrum_ragged_host(hd._h, ctypes.cast(None, ctypes.POINTER(_abi.GrayDesc)), 1) == -1
    assert hd.launch_count == c0
