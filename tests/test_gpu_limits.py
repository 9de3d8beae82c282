"""GPU: every entry point at the size limits include/v5ela.h promises — frames of up to 2^31 - 65536 pixels and sides of 65536,
strides and batch offsets past 2^32 bytes, spectra and JPEG files with 65535-pixel sides, JPEG entropy streams past 2^32 bits,
and calls of more than 65535 frames — and the refusals just past those limits.

Giant frames repeat a 16 x 16 tile and are checked against tests/periodic_ref.py (the C oracle on small frames, exact; proven by
tests/test_periodic_reference.py). Inputs are built on the device and freed after each test; every descriptor, refused ones
included, points at a real allocation of the size it claims."""
import gc
import hashlib
import io

import numpy as np
import pytest

from oracle import c_oracle, pil_oracle
from periodic_ref import band_index, expected_ghost, expected_record, expected_residual_bands, expected_tex_hist, ghost_of, tile_of
from v5ela.records import RECORD_DTYPE, as_records, combine

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_UNSUPPORTED = -1, -5


def handle():
    import torch
    from v5ela.batch import get_handle

    return get_handle(torch.cuda.current_device())


@pytest.fixture(autouse=True)
def free_device_memory():
    import torch

    yield
    gc.collect()
    torch.cuda.empty_cache()


def dev_tiled(tile, h, w, out=None):
    """tiled(tile, h, w) written on the device into `out` (an (h, w, 3) uint8 view, any row stride) or a new tensor."""
    import torch

    t = torch.from_numpy(np.ascontiguousarray(tile)).cuda()
    band = t.repeat(1, w // 16 + 1, 1)[:, :w]                           # 16 x w x 3
    if out is None:
        out = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    m = h // 16
    if m:
        out[:16 * m].unflatten(0, (m, 16)).copy_(band.expand(m, 16, w, 3))
    out[16 * m:].copy_(band[:h - 16 * m])
    return out


def records_of(t):
    return as_records(t.reshape(-1, 3144).cpu().numpy())


def compare_residual(res, tile, h, w, q, slab_rows=4096):
    """The device residual map (h, w, 3) against the band reference, one device-built slab of expected rows at a time."""
    import torch

    small, _ = expected_residual_bands(tile, h, w, q)
    small_t = torch.from_numpy(small).cuda()
    rows, cols = torch.from_numpy(band_index(h)).cuda(), torch.from_numpy(band_index(w)).cuda()
    for y0 in range(0, h, slab_rows):
        y1 = min(h, y0 + slab_rows)
        want = small_t.index_select(0, rows[y0:y1]).index_select(1, cols)
        assert torch.equal(res[y0:y1], want), (h, w, q, y0)


# ------------------------------------------------------------------------------------------- 1. largest admissible frames
@pytest.mark.usefixtures("block_stage")
def test_largest_frame_general_with_residual_and_tex_hist():
    """65536 x 32767 = 2^31 - 65536 px (6.4 GB) through analyze_ex with the residual map and tex_hist: the GENERAL / TEXHIST code."""
    import torch

    h, w, q = 65536, 32767, 90
    tile = tile_of("noise", seed=11)
    hd = handle()
    hd.set_quality(q)
    frame = dev_tiled(tile, h, w)
    rec = torch.empty(3144, dtype=torch.uint8, device="cuda")
    res = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    th = torch.empty(256, dtype=torch.int32, device="cuda")
    hd.analyze(frame.data_ptr(), 1, h, w, h * w * 3, w * 3, rec.data_ptr(), res.data_ptr(), torch.cuda.current_stream().cuda_stream,
               th.data_ptr())
    assert hd.last_instantiation == "texhist"
    del frame
    assert records_of(rec)[0].tobytes() == expected_record(tile, h, w, q).tobytes()
    assert np.array_equal(th.cpu().numpy().view(np.uint32), expected_tex_hist(tile, h, w))
    compare_residual(res, tile, h, w, q)


@pytest.mark.usefixtures("block_stage")
@pytest.mark.parametrize("kind", ["noise", "flat"])
def test_largest_frame_fast_records_only(kind):
    """32768 x 65520 records only: the FAST instantiation. The flat tile puts ~2^31 counts into one histogram bin per channel."""
    import torch

    h, w, q = 32768, 65520, 75
    tile = tile_of(kind, seed=12)
    hd = handle()
    hd.set_quality(q)
    frame = dev_tiled(tile, h, w)
    rec = torch.empty(3144, dtype=torch.uint8, device="cuda")
    hd.analyze(frame.data_ptr(), 1, h, w, h * w * 3, w * 3, rec.data_ptr(), None, torch.cuda.current_stream().cuda_stream)
    assert hd.last_instantiation == "fast"
    got = records_of(rec)[0]
    assert got.tobytes() == expected_record(tile, h, w, q).tobytes()
    if kind == "flat":
        assert int(got["ela_hist"].max()) == h * w


# ----------------------------------------------------------------------------- 2. batch and stride offsets past 2^32 bytes
@pytest.mark.usefixtures("block_stage")
def test_batch_offsets_past_4gib():
    """Three 24000 x 32000 frames (6.9 GB), each its own tile, as views into one wider buffer with padded rows: y * row_stride and
    the frame offsets pass 2^31 and 2^32. Uniform call, one ragged call, and a two-quality sweep with ghost maps."""
    import torch
    import v5ela

    h, w, n, q = 24000, 32000, 3, 90
    row = 3 * w + 64
    fstride = h * row + 4096
    assert (h - 1) * row > 2 ** 31 and (n - 1) * fstride > 2 ** 32
    buf = torch.empty(n * fstride, dtype=torch.uint8, device="cuda")
    frames = buf.as_strided((n, h, w, 3), (fstride, row, 3, 1))
    tiles = [tile_of(k, seed=20 + i) for i, k in enumerate(["noise", "smooth", "saturated"])]
    for i in range(n):
        dev_tiled(tiles[i], h, w, out=frames[i])
    want = {qq: [expected_record(tiles[i], h, w, qq).tobytes() for i in range(n)] for qq in (q, 40)}

    uni = v5ela.analyze_batch(frames, quality=q)["records"]
    rag = v5ela.analyze_ragged([frames[i] for i in range(n)], quality=q)["records"]
    sw = v5ela.analyze_sweep(frames, [q, 40], want_ghost=True)
    torch.cuda.synchronize()
    assert [r.tobytes() for r in records_of(uni)] == want[q]
    assert [r.tobytes() for r in records_of(rag)] == want[q]
    srec = records_of(sw["records"]).reshape(2, n)
    for k, qq in enumerate((q, 40)):
        assert [r.tobytes() for r in srec[k]] == want[qq], qq
        for i in range(n):
            _, gslab = expected_ghost(tiles[i], h, w, qq)
            assert np.array_equal(sw["ghost"][k, i].cpu().numpy(), gslab(0, -(-h // 16))), (qq, i)


# ------------------------------------------------------------------------- 3. extreme aspect ratios, straight against the oracle
ASPECT = [(1, 65536), (65536, 1), (16, 65536), (65536, 16), (17, 65535)]


@pytest.fixture(scope="module")
def aspect_frames():
    rng = np.random.default_rng(30)
    frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ASPECT]
    oracle = {(i, q): c_oracle.analyze_frame(f, q) for i, f in enumerate(frames) for q in (90, 30)}
    return frames, oracle


@pytest.mark.usefixtures("block_stage")
def test_extreme_aspect_ratios(aspect_frames):
    import torch
    import v5ela

    frames, oracle = aspect_frames
    dev = [torch.from_numpy(f).cuda() for f in frames]
    for i, t in enumerate(dev):                                            # uniform, one frame each
        out = v5ela.analyze_batch(t[None], quality=90, want_residual=True)
        torch.cuda.synchronize()
        assert records_of(out["records"])[0].tobytes() == oracle[i, 90]["record"].tobytes(), ASPECT[i]
        assert np.array_equal(out["residual"][0].cpu().numpy(), oracle[i, 90]["residual"]), ASPECT[i]
    rng = np.random.default_rng(31)
    small = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in [(3, 5), (40, 33), (1, 1)]]
    mixed = [dev[0], torch.from_numpy(small[0]).cuda(), dev[1], dev[2], torch.from_numpy(small[1]).cuda(), dev[3], dev[4],
             torch.from_numpy(small[2]).cuda()]
    want = [oracle[0, 90], c_oracle.analyze_frame(small[0], 90), oracle[1, 90], oracle[2, 90], c_oracle.analyze_frame(small[1], 90),
            oracle[3, 90], oracle[4, 90], c_oracle.analyze_frame(small[2], 90)]
    rag = v5ela.analyze_ragged(mixed, quality=90, want_residual=True)
    sw = v5ela.analyze_sweep(dev, [90, 30], want_ghost=True)
    torch.cuda.synchronize()
    rr = records_of(rag["records"])
    for k, o in enumerate(want):
        assert rr[k].tobytes() == o["record"].tobytes(), k
        assert np.array_equal(rag["residual"][k].cpu().numpy(), o["residual"]), k
    srec = records_of(sw["records"]).reshape(2, len(dev))
    for k, q in enumerate((90, 30)):
        for i in range(len(dev)):
            assert srec[k, i].tobytes() == oracle[i, q]["record"].tobytes(), (q, ASPECT[i])
            assert np.array_equal(sw["ghost"][k][i].cpu().numpy(), ghost_of(oracle[i, q]["residual"])), (q, ASPECT[i])


# --------------------------------------------------------------------------------------------------------- 4. limit refusals
@pytest.mark.parametrize("hw", [(65537, 16), (16, 65537), (65536, 32768)])
def test_size_refusals_before_any_launch(hw):
    """A side of 65537, or h * w = 2^31, is refused by the uniform, ragged and sweep calls with V5ELA_ERR_INVALID and no launch.
    The descriptors point at a real allocation of the claimed size."""
    import torch
    from v5ela import _abi

    h, w = hw
    hd = handle()
    buf = torch.zeros(h * w * 3, dtype=torch.uint8, device="cuda")
    rec = torch.empty((2, 3144), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    before = hd.launch_count
    with pytest.raises(_abi.V5ElaError) as e:
        hd.analyze(buf.data_ptr(), 1, h, w, h * w * 3, w * 3, rec.data_ptr(), None, st)
    assert e.value.status == ERR_INVALID
    descs = (_abi.FrameDesc * 1)()
    descs[0].rgb, descs[0].height, descs[0].width, descs[0].row_stride_bytes = buf.data_ptr(), h, w, 3 * w
    with pytest.raises(_abi.V5ElaError) as e:
        hd.analyze_ragged(descs, 1, rec.data_ptr(), st)
    assert e.value.status == ERR_INVALID
    with pytest.raises(_abi.V5ElaError) as e:
        hd.analyze_sweep(descs, 1, [90, 50], rec.data_ptr(), None, st)
    assert e.value.status == ERR_INVALID
    torch.cuda.synchronize()
    assert hd.launch_count == before


# ------------------------------------------------------------------------------------------------- 5. spectrum at its limits
SPEC_SIZES = [(1, 65536), (65536, 1), (2, 65536), (65536, 3), (5, 65521), (65521, 4)]


def spec_check(got, gray, min_exact=0.999):
    ref = pil_oracle.fft_spectrum(gray)
    d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
    assert int(d.max()) <= 1, (gray.shape, int(d.max()))
    assert float((d == 0).mean()) >= min_exact, gray.shape


@pytest.fixture(scope="module")
def spec_images():
    rng = np.random.default_rng(50)
    return [rng.integers(0, 256, s, dtype=np.uint8) for s in SPEC_SIZES]


@pytest.mark.parametrize("fft", ["1", "0"])
def test_spectrum_side_limits(spec_images, fft, monkeypatch):
    """Uniform and one ragged call (with small crops) against NumPy; V5ELA_FFT=0 (exact-size DFT everywhere) likewise."""
    import torch
    import v5ela

    monkeypatch.setenv("V5ELA_FFT", fft)
    rng = np.random.default_rng(51)
    crops = [rng.integers(0, 256, s, dtype=np.uint8) for s in [(7, 9), (64, 48), (1, 1)]]
    dev = [torch.from_numpy(g).cuda() for g in spec_images]
    for g, t in zip(spec_images, dev):
        spec_check(v5ela.spectrum_batch(t[None])[0].cpu().numpy(), g)
    allimg = spec_images[:3] + crops + spec_images[3:]
    outs = v5ela.spectrum_ragged(dev[:3] + [torch.from_numpy(c).cuda() for c in crops] + dev[3:])
    torch.cuda.synchronize()
    for g, o in zip(allimg, outs):
        spec_check(o.cpu().numpy(), g, min_exact=0.99 if g.size < 1000 else 0.999)


def test_spectrum_70000_tiny_images():
    """70000 images of 6 x 10 in one uniform call: past the 65535-image chunk and the n <= 65535 FFT-path switch."""
    import torch
    import v5ela

    rng = np.random.default_rng(52)
    distinct = rng.integers(0, 256, (7, 6, 10), dtype=np.uint8)
    idx = np.arange(70000) % 7
    out = v5ela.spectrum_batch(torch.from_numpy(distinct).cuda()[torch.from_numpy(idx).cuda()]).cpu().numpy()
    ref = np.stack([pil_oracle.fft_spectrum(g) for g in distinct])
    d = np.abs(out.astype(np.int16) - ref[idx].astype(np.int16))
    assert int(d.max()) <= 1 and float((d == 0).mean()) >= 0.99
    for k in range(7):                                                     # every copy of an image is the same bytes
        assert (out[idx == k] == out[k]).all(), k


def test_spectrum_side_65537_refused():
    import torch
    from v5ela import _abi

    hd = handle()
    buf = torch.zeros(65537 * 2, dtype=torch.uint8, device="cuda")
    out = torch.empty(65537 * 2, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    before = hd.launch_count
    for h, w in [(65537, 2), (2, 65537)]:
        with pytest.raises(_abi.V5ElaError) as e:
            hd.spectrum(buf.data_ptr(), 1, h, w, h * w, w, out.data_ptr(), st)
        assert e.value.status == ERR_INVALID
        d = (_abi.GrayDesc * 1)()
        d[0].gray, d[0].height, d[0].width, d[0].row_stride_bytes, d[0].out = buf.data_ptr(), h, w, w, out.data_ptr()
        with pytest.raises(_abi.V5ElaError) as e:
            hd.spectrum_ragged(d, 1, st)
        assert e.value.status == ERR_INVALID
    torch.cuda.synchronize()
    assert hd.launch_count == before


# ------------------------------------------------------------------------------------------- 6. JPEG at 65535-pixel sides
# libjpeg (Pillow, OpenCV) writes sides up to JPEG_MAX_DIMENSION = 65500; the library's encoder goes to 65535, checked against the C
# oracle there and against Pillow at 65500.
def pil_file(img, q, **kw):
    from PIL import Image

    buf = io.BytesIO()
    Image.fromarray(img).save(buf, "JPEG", quality=q, **kw)
    return buf.getvalue()


def pil_rgb(data):
    from PIL import Image

    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


@pytest.mark.parametrize("hw", [(65535, 8), (8, 65535), (65500, 9), (9, 65500)])
@pytest.mark.parametrize("ch", [3, 1])
def test_jpeg_encode_65535_sides(hw, ch):
    from v5ela import jpeg

    h, w = hw
    rng = np.random.default_rng(60 + ch)
    img = rng.integers(0, 256, (h, w, 3) if ch == 3 else (h, w), dtype=np.uint8)
    for q in (1, 90, 100):
        got = jpeg.encode_host(img[None], q)[0]
        assert got == c_oracle.jpeg_encode(img, q), (hw, ch, q)
        if max(hw) <= 65500:
            assert got == pil_file(img, q), (hw, ch, q)


@pytest.mark.parametrize("hw", [(65500, 8), (8, 65500)])
def test_jpeg_decode_and_dct_stats_65535_sides(hw):
    """Pillow and OpenCV files of 65500-pixel sides (libjpeg's limit) in every layout, with restart intervals, and the library's
    own 65535-pixel files: pixels as Pillow (or the C oracle) decodes them, DCT histograms as NumPy counts them over the oracle's
    coefficients, and maps of ceil(H/8) x ceil(W/8) blocks."""
    import cv2
    from dct_helpers import np_hist
    from v5ela import jpeg

    h, w = hw
    rng = np.random.default_rng(61)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    gray = img[..., 0].copy()
    files = [pil_file(img, 90, subsampling=s) for s in (2, 1, 0)]
    files += [pil_file(img, 75, restart_marker_blocks=3), pil_file(gray, 95), pil_file(gray, 95, restart_marker_rows=1)]
    ok, enc = cv2.imencode(".jpg", img[..., ::-1], [cv2.IMWRITE_JPEG_QUALITY, 95])
    assert ok
    files.append(enc.tobytes())
    ok, enc = cv2.imencode(".jpg", gray, [cv2.IMWRITE_JPEG_QUALITY, 95, cv2.IMWRITE_JPEG_RST_INTERVAL, 7])
    assert ok
    files.append(enc.tobytes())
    n_libjpeg = len(files)
    big = rng.integers(0, 256, (65535, 7, 3) if h > w else (7, 65535, 3), dtype=np.uint8)
    files += [jpeg.encode_host(big[None], 90)[0], jpeg.encode_host(big[None, ..., 1], 100)[0]]
    dec = jpeg.decode_host(files)
    for k, (data, d) in enumerate(zip(files, dec)):
        want = pil_rgb(data) if k < n_libjpeg else c_oracle.jpeg_decode(data)["rgb"]
        assert np.array_equal(d["rgb"], want), (hw, k)
    st = jpeg.dct_stats_host(files, want_map=True)
    for k, data in enumerate(files):
        hh, ww, _ = c_oracle.jpeg_info(data)
        assert np.array_equal(st["hist"][k], np_hist(data)), (hw, k)
        assert st["map"][k].shape == (-(-hh // 8), -(-ww // 8)), (hw, k)


# ------------------------------------------------------------------------------------- 7. JPEG streams past 2^32 bits
@pytest.fixture(scope="module")
def giant_noise_files():
    """Pillow's q = 100 files of an 18000 x 18000 and a 15000 x 15000 noise image (~640 MB and ~445 MB)."""
    from PIL import Image

    Image.MAX_IMAGE_PIXELS = None
    rng = np.random.default_rng(70)
    out = {}
    for side in (18000, 15000):
        img = rng.integers(0, 256, (side, side, 3), dtype=np.uint8)
        out[side] = (img, pil_file(img, 100))
    return out


def test_jpeg_encode_past_2_32_bits(giant_noise_files):
    """The 18000 x 18000 q = 100 file has more than 2^32 entropy-coded bits; with the default capacity the GPU file must be
    Pillow's, byte for byte."""
    from v5ela import jpeg

    img, ref = giant_noise_files[18000]
    assert len(ref) * 8 > 2 ** 32 and len(ref) < jpeg.default_capacity(18000, 18000, 3)
    got = jpeg.encode_host(img[None], 100)[0]
    assert len(got) == len(ref)
    assert hashlib.sha256(got).hexdigest() == hashlib.sha256(ref).hexdigest()


def test_jpeg_decode_refuses_512mib_entropy_segment(giant_noise_files):
    """A file whose entropy-coded segment is 2^29 - 2^20 bytes or more is refused as unsupported, naming the file, before any
    upload or launch — by the decoder and by the DCT statistics."""
    import torch
    from v5ela import _abi, jpeg

    _, data = giant_noise_files[18000]
    assert len(data) > 2 ** 29
    small = pil_file(np.zeros((16, 16, 3), np.uint8), 90)
    hd = handle()
    before = hd.launch_count
    for call in (lambda: jpeg.decode_host([small, data]), lambda: jpeg.dct_stats([small, data])):
        with pytest.raises(_abi.V5ElaError) as e:
            call()
        assert e.value.status == ERR_UNSUPPORTED
        assert "entropy-coded segment" in str(e.value) and "(file 1)" in str(e.value)
    torch.cuda.synchronize()
    assert hd.launch_count == before


@pytest.mark.parametrize("path", ["one", "three"])
def test_jpeg_decode_445mb_file(giant_noise_files, path, monkeypatch):
    """The 15000 x 15000 q = 100 file (just under the limit) decodes pixel-identical to Pillow on both Huffman paths."""
    from v5ela import jpeg

    _, data = giant_noise_files[15000]
    monkeypatch.setenv("V5ELA_HUFF_PATH", path)
    assert np.array_equal(jpeg.decode_host([data])[0]["rgb"], pil_rgb(data))


# ------------------------------------------------------------------------------------ 8. enhancement and reduction grids
@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("hw", [(16, 16), (5, 7)])
def test_enhance_every_max_and_value(offset, hw):
    """256 records with ela_max = (m, 0, 0), m = 0..255, over residuals holding every value 0..255 (16 x 16: 768 bytes, the vector
    path) or 0..104 (5 x 7: 105 bytes, the scalar tail), at aligned and unaligned pointers; expected: the oracle's LUT of max(m, 1)."""
    import torch

    h, w = hw
    nb = h * w * 3
    recs = np.zeros(256, RECORD_DTYPE)
    recs["ela_max"][:, 0] = np.arange(256)
    res = np.tile(np.arange(nb, dtype=np.int64) % 256, (256, 1)).astype(np.uint8)
    lut = np.stack([c_oracle.enhance_lut(max(m, 1)) for m in range(256)])
    exp = np.stack([lut[m][res[m]] for m in range(256)])
    rb = torch.zeros(256 * nb + 16, dtype=torch.uint8, device="cuda")
    ob = torch.zeros(256 * nb + 16, dtype=torch.uint8, device="cuda")
    rb[offset:offset + 256 * nb] = torch.from_numpy(res.ravel()).cuda()
    dr = torch.from_numpy(recs.view(np.uint8)).cuda()
    handle().enhance(rb.data_ptr() + offset, dr.data_ptr(), 256, h, w, ob.data_ptr() + offset, torch.cuda.current_stream().cuda_stream)
    got = ob[offset:offset + 256 * nb].cpu().numpy().reshape(256, nb)
    assert np.array_equal(got, exp)


def test_enhance_70000_frames():
    import torch

    n = 70000
    m = np.arange(n) % 256
    recs = np.zeros(n, RECORD_DTYPE)
    recs["ela_max"][:, 1] = m
    res = np.tile(np.arange(768, dtype=np.int64) % 256, (n, 1)).astype(np.uint8)
    lut = np.stack([c_oracle.enhance_lut(max(k, 1)) for k in range(256)])
    dr = torch.from_numpy(recs.view(np.uint8)).cuda()
    rt = torch.from_numpy(res).cuda()
    out = torch.empty_like(rt)
    hd = handle()
    before = hd.launch_count
    hd.enhance(rt.data_ptr(), dr.data_ptr(), n, 16, 16, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    got = out.cpu().numpy()
    assert np.array_equal(got, lut[m][:, np.arange(768) % 256])
    assert hd.launch_count - before == 2                                    # 65535 + 4465 frames


@pytest.fixture(scope="module")
def seven_frames():
    rng = np.random.default_rng(80)
    frames = rng.integers(0, 256, (7, 16, 16, 3), dtype=np.uint8)
    frames[3] = 128                                                         # a flat frame: max_diff 0 -> 1
    oracle = [c_oracle.analyze_frame(f, 90) for f in frames]
    lut = [c_oracle.enhance_lut(max(int(o["record"]["ela_max"].max()), 1)) for o in oracle]
    enh = np.stack([lut[k][o["residual"]] for k, o in enumerate(oracle)])
    return frames, oracle, enh


def test_analyze_batch_enhanced_70000_frames(seven_frames):
    import torch
    import v5ela

    frames, oracle, enh = seven_frames
    idx = np.arange(70000) % 7
    t = torch.from_numpy(frames).cuda()[torch.from_numpy(idx).cuda()]
    out = v5ela.analyze_batch(t, quality=90, want_enhanced=True)
    recs = records_of(out["records"])
    got = out["enhanced"].cpu().numpy()
    for k in range(7):
        sel = idx == k
        assert (recs[sel].view(np.uint8).reshape(-1, 3144) == np.frombuffer(oracle[k]["record"].tobytes(), np.uint8)).all(), k
        assert (got[sel] == enh[k]).all(), k


def test_analyze_host_100000_frames_with_maps(seven_frames):
    from v5ela import host

    frames, oracle, enh = seven_frames
    idx = np.arange(100000) % 7
    recs, res, en = host.analyze_frames_host(frames[idx], 90, want_residual=True, want_enhanced=True)
    for k in range(7):
        sel = idx == k
        assert (recs[sel].view(np.uint8).reshape(-1, 3144) == np.frombuffer(oracle[k]["record"].tobytes(), np.uint8)).all(), k
        assert (res[sel] == oracle[k]["residual"]).all(), k
        assert (en[sel] == enh[k]).all(), k


def test_analyze_ragged_70000_descriptors(seven_frames):
    """70000 descriptors, every tenth with an enhanced map (and every seventh with a residual): records and maps are right."""
    import torch
    from v5ela import _abi

    frames, oracle, enh = seven_frames
    n = 70000
    idx = np.arange(n) % 7
    t = torch.from_numpy(frames).cuda()[torch.from_numpy(idx).cuda()].contiguous()
    res = torch.zeros_like(t)
    out = torch.zeros_like(t)
    rec = torch.empty((n, 3144), dtype=torch.uint8, device="cuda")
    descs = (_abi.FrameDesc * n)()
    fb = 16 * 16 * 3
    for i in range(n):
        d = descs[i]
        d.rgb, d.height, d.width, d.row_stride_bytes = t.data_ptr() + i * fb, 16, 16, 48
        d.residual = res.data_ptr() + i * fb if i % 7 == 0 else None
        d.enhanced = out.data_ptr() + i * fb if i % 10 == 0 else None
    handle().analyze_ragged(descs, n, rec.data_ptr(), torch.cuda.current_stream().cuda_stream)
    recs, res, out = records_of(rec), res.cpu().numpy(), out.cpu().numpy()
    for k in range(7):
        sel = idx == k
        assert (recs[sel].view(np.uint8).reshape(-1, 3144) == np.frombuffer(oracle[k]["record"].tobytes(), np.uint8)).all(), k
        e = sel & (np.arange(n) % 10 == 0)
        r = sel & (np.arange(n) % 7 == 0)
        assert (out[e] == enh[k]).all(), k
        assert (res[r] == oracle[k]["residual"]).all(), k
    assert not out[np.arange(n) % 10 != 0].any()


def test_reduce_records_saturation_and_64bit_sums():
    import torch
    import v5ela

    rng = np.random.default_rng(90)

    def reduce(recs, group):
        out = v5ela.reduce_records(torch.from_numpy(recs.view(np.uint8).reshape(-1, 3144).copy()).cuda(), group)
        return records_of(out)

    # bins that sum to exactly 2^32 - 1 (kept), 2^32 and 3 (2^32 - 1) (saturated); 64-bit sums up to just under 2^64
    recs = np.zeros(3, RECORD_DTYPE)
    recs["ela_hist"][0, 0, 0], recs["ela_hist"][1, 0, 0], recs["ela_hist"][2, 0, 0] = 2 ** 32 - 3, 1, 2
    recs["ela_hist"][:, 0, 1] = [2 ** 32 - 2, 1, 0]
    recs["ela_hist"][:, 1, 7] = [2 ** 31, 2 ** 31, 0]
    recs["ela_hist"][:, 2, 255] = 2 ** 32 - 1
    top = 2 ** 64 - 1
    recs["ela_sum"][:, 0] = [top // 3, top // 3, top // 3]
    recs["tex_sumsq"] = [top - 10, 5, 4]
    recs["tex_maxabs"] = [3, 1020, 7]
    recs["ela_max"] = [[1, 2, 3], [255, 0, 9], [4, 5, 6]]
    got = reduce(recs, 3)[0]
    assert got.tobytes() == combine(recs).tobytes()
    assert int(got["ela_hist"][0, 1]) == 2 ** 32 - 1 and int(got["ela_hist"][0, 0]) == 2 ** 32 - 1 and int(got["ela_hist"][1, 7]) == 2 ** 32 - 1
    assert int(got["ela_hist"][2, 255]) == 2 ** 32 - 1 and int(got["tex_sumsq"]) == top - 1
    # random records, group sizes 1, 3 and n; 70002 groups of one
    n = 70002
    recs = np.zeros(n, RECORD_DTYPE)
    raw = recs.view(np.uint8).reshape(n, 3144)
    raw[:, :3072] = rng.integers(0, 256, (n, 3072), dtype=np.uint8)
    recs["ela_sum"] = rng.integers(0, 2 ** 46, (n, 3), dtype=np.uint64)
    recs["tex_sumabs"] = rng.integers(0, 2 ** 40, n, dtype=np.uint64)
    recs["tex_maxabs"] = rng.integers(0, 1021, n)
    recs["ela_max"] = rng.integers(0, 256, (n, 3))
    for group in (1, 3, n):
        got = reduce(recs, group)
        assert len(got) == n // group
        if group == 1:
            assert got.tobytes() == recs.tobytes()
            continue
        want = np.stack([combine(recs[g * group:(g + 1) * group]) for g in range(n // group)])
        assert got.tobytes() == want.tobytes(), group
