"""GPU: v5ela_jpeg_dct_stats / _host (include/v5ela.h) against NumPy over the oracle decoder's coefficients — histograms identical,
quantisation tables equal to the DQT, maps within 1e-6 of records.dq_map on the GPU's own histograms — across every layout, a mixed
call of 40 random sizes and qualities, both Huffman paths, pinned and pageable files; refusals, truncated files, and the decoder
left as it was."""
import io

import numpy as np
import pytest
from PIL import Image

from dct_helpers import layout_files, luma_grid, np_hist, odd_size_files, pil_bytes, qtab_of

pytestmark = pytest.mark.gpu

CASES = layout_files()
MIXED = odd_size_files(np.random.default_rng(40), 40, max_side=300)


def _check(files, out, maps=True):
    hist = out["hist"].cpu().numpy().view(np.uint32) if hasattr(out["hist"], "cpu") else out["hist"]
    qtab = out["qtab"].cpu().numpy() if hasattr(out["qtab"], "cpu") else out["qtab"]
    from v5ela import records

    for i, data in enumerate(files):
        assert np.array_equal(hist[i], np_hist(data)), i
        assert np.array_equal(qtab[i], qtab_of(data)), i
        if maps:
            m = out["map"][i]
            m = m.cpu().numpy() if hasattr(m, "cpu") else m
            ref = records.dq_map(hist[i], luma_grid(data))
            assert m.shape == ref.shape and np.abs(m.astype(np.float64) - ref).max() <= 1e-6, i


@pytest.mark.parametrize("path", ["one", "three"])
def test_every_layout_in_one_call(monkeypatch, path):
    import torch
    from v5ela import jpeg

    monkeypatch.setenv("V5ELA_HUFF_PATH", path)
    files = [d for _, d in CASES]
    out = jpeg.dct_stats(files, want_map=True)
    torch.cuda.synchronize()
    assert (out["status"].cpu().numpy() == 0).all()
    _check(files, out)


@pytest.mark.parametrize("path", ["one", "three"])
def test_forty_random_sizes_and_qualities_in_one_call(monkeypatch, path):
    import torch
    from v5ela import jpeg

    monkeypatch.setenv("V5ELA_HUFF_PATH", path)
    files = [d for _, d in MIXED]
    out = jpeg.dct_stats(files, want_map=True)
    torch.cuda.synchronize()
    _check(files, out)
    host = jpeg.dct_stats_host(files, want_map=True)
    assert np.array_equal(host["hist"], out["hist"].cpu().numpy().view(np.uint32))
    assert np.array_equal(host["qtab"], out["qtab"].cpu().numpy())
    for a, b in zip(host["map"], out["map"]):
        assert np.array_equal(a, b.cpu().numpy())


def test_pinned_and_pageable_files_agree():
    import torch
    from v5ela import jpeg

    files = [d for _, d in MIXED[:12]]
    sizes = [len(f) for f in files]
    arena = torch.empty(sum(sizes) + 64 * len(files), dtype=torch.uint8).pin_memory()
    views, off = [], 0
    for f in files:
        a = arena[off:off + len(f)].numpy()
        a[:] = np.frombuffer(f, np.uint8)
        views.append(a)
        off += len(f) + 64
    pinned = jpeg.dct_stats(views, want_map=True)
    pageable = jpeg.dct_stats(files, want_map=True)
    torch.cuda.synchronize()
    assert torch.equal(pinned["hist"], pageable["hist"]) and torch.equal(pinned["qtab"], pageable["qtab"])
    for a, b in zip(pinned["map"], pageable["map"]):
        assert torch.equal(a, b)
    del arena


def test_map_offsets_and_no_optional_outputs():
    import ctypes

    import torch
    from v5ela import _abi, jpeg

    files = [d for _, d in MIXED[:5]]
    keep, ptrs, lens = jpeg._file_table(files)
    dims = jpeg.info_batch(files)
    cnt = [((int(h) + 7) // 8) * ((int(w) + 7) // 8) for h, w, _ in dims]
    offs, total = np.zeros(5, np.int64), 0
    for i in reversed(range(5)):                                             # maps in reverse file order, gaps between them
        offs[i] = total
        total += cnt[i] + 17
    arena = torch.full((total,), -7.0, dtype=torch.float32, device="cuda")
    hist = torch.zeros((5, 3, 64, 129), dtype=torch.int32, device="cuda")
    hd = _abi.get_handle(0)
    hd.jpeg_dct_stats(ptrs, lens, 5, hist.data_ptr(), None, arena.data_ptr(), offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), None,
                      torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    packed = jpeg.dct_stats(files, want_qtab=False, want_map=True)
    torch.cuda.synchronize()
    assert "qtab" not in packed and torch.equal(packed["hist"], hist)
    a = arena.cpu().numpy()
    used = np.zeros(total, bool)
    for i in range(5):
        got = a[offs[i]:offs[i] + cnt[i]]
        assert np.array_equal(got, packed["map"][i].cpu().numpy().ravel())
        used[offs[i]:offs[i] + cnt[i]] = True
    assert (a[~used] == -7.0).all()                                          # nothing outside the maps is written
    del keep


def test_refusals_truncation_and_empty_calls():
    import ctypes

    import torch
    from v5ela import _abi, jpeg

    rgb = np.random.default_rng(1).integers(0, 256, (40, 48, 3), dtype=np.uint8)
    good = pil_bytes(rgb, 80)
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, "JPEG", quality=80, progressive=True)
    with pytest.raises(_abi.V5ElaError) as ei:
        jpeg.dct_stats([good, buf.getvalue()])
    assert ei.value.status == -5 and "file 1" in str(ei.value)
    with pytest.raises(_abi.V5ElaError) as ei:
        jpeg.dct_stats_host([good, good, buf.getvalue()])
    assert ei.value.status == -5 and "file 2" in str(ei.value)
    # a truncated entropy-coded segment: status -1 from the device call, V5ELA_ERR_INVALID from the host call
    cut = good[:len(good) // 2] + b"\xff\xd9"
    out = jpeg.dct_stats([good, cut])
    torch.cuda.synchronize()
    assert out["status"].cpu().tolist() == [0, -1]
    with pytest.raises(_abi.V5ElaError) as ei:
        jpeg.dct_stats_host([good, cut])
    assert ei.value.status == -1 and "file 1" in str(ei.value)
    # a negative map offset is refused before anything is launched
    hd = _abi.get_handle(0)
    keep, ptrs, lens = jpeg._file_table([good, good])
    offs = np.array([0, -1], np.int64)
    before = hd.launch_count
    with pytest.raises(_abi.V5ElaError) as ei:
        hd.jpeg_dct_stats(ptrs, lens, 2, out["hist"].data_ptr(), None, out["hist"].data_ptr(),
                          offs.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), None, None)
    assert ei.value.status == -1 and "file 1" in str(ei.value) and hd.launch_count == before
    # n == 0 is OK
    lib = _abi.load()
    assert lib.v5ela_jpeg_dct_stats(hd._h, None, None, 0, None, None, None, None, None, None) == 0
    assert lib.v5ela_jpeg_dct_stats_host(hd._h, None, None, 0, None, None, None, None) == 0
    assert jpeg.dct_stats([])["hist"].shape == (0, 3, 64, 129)
    del keep


def test_launch_counts(monkeypatch):
    import torch
    from v5ela import _abi, jpeg

    hd = _abi.get_handle(0)
    files = [d for _, d in MIXED[:6]]
    for path, want in (("one", 3), ("three", 5)):                           # unstuff, Huffman (1 or 3 launches), dc
        monkeypatch.setenv("V5ELA_HUFF_PATH", path)
        before = hd.launch_count
        jpeg.dct_stats(files)
        assert hd.launch_count - before == want + 1
        before = hd.launch_count
        jpeg.dct_stats(files, want_map=True)
        assert hd.launch_count - before == want + 3
        before = hd.launch_count
        jpeg.decode_host(files)
        assert hd.launch_count - before == want + 2                         # the decoder's count is unchanged
    torch.cuda.synchronize()


def test_decode_on_the_same_handle_is_unchanged():
    import torch
    from v5ela import jpeg

    files = [d for _, d in MIXED[:10]]
    before = jpeg.decode_host(files, want_rgb=True, want_gray=True)
    jpeg.dct_stats(files, want_map=True)
    jpeg.dct_stats_host(files, want_map=True)
    torch.cuda.synchronize()
    after = jpeg.decode_host(files, want_rgb=True, want_gray=True)
    for a, b in zip(before, after):
        assert np.array_equal(a["rgb"], b["rgb"]) and np.array_equal(a["gray"], b["gray"])


def test_ijg_quality_of_the_gpu_tables():
    import torch
    from v5ela import jpeg

    rgb = np.random.default_rng(5).integers(0, 256, (30, 50, 3), dtype=np.uint8)
    qs = [1, 37, 60, 90, 100]
    out = jpeg.dct_stats([pil_bytes(rgb, q) for q in qs] + [pil_bytes(np.ascontiguousarray(rgb[..., 0]), 77)])
    torch.cuda.synchronize()
    assert [jpeg.ijg_quality(t) for t in out["qtab"]] == qs + [77]


def test_pasted_single_compressed_region_stands_out():
    """A 512x512 synthetic frame saved at quality 60, decoded, an 8-aligned 128x128 block of the never-compressed frame pasted in,
    saved at 90: the map is higher over the pasted blocks than over the rest (DESIGN.md §4.8 records the margin)."""
    import torch
    from v5ela import jpeg, records
    from v5ela.synth import gen_frame

    frame = gen_frame(0, 512, 512, 0)
    once = np.asarray(Image.open(io.BytesIO(pil_bytes(frame, 60))).convert("RGB")).copy()
    y0, x0 = 192, 256
    once[y0:y0 + 128, x0:x0 + 128] = frame[y0:y0 + 128, x0:x0 + 128]
    data = pil_bytes(once, 90)
    out = jpeg.dct_stats([data], want_map=True)
    torch.cuda.synchronize()
    m = out["map"][0].cpu().numpy()
    mask = np.zeros(m.shape, bool)
    mask[y0 // 8:(y0 + 128) // 8, x0 // 8:(x0 + 128) // 8] = True
    margin = float(m[mask].mean() - m[~mask].mean())
    print(f"pasted {m[mask].mean():.4f} rest {m[~mask].mean():.4f} margin {margin:.4f} periods {records.dq_periods(out['hist'][0].cpu().numpy().view(np.uint32)).tolist()}")
    assert margin > 0.3
