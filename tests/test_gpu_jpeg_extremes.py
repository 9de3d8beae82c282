"""GPU: the JPEG decoder, the DCT statistics and the file-to-records path on coefficients at the limits of a baseline file
(tests/jpeg_craft.py, the same corpus as tests/test_jpeg_extremes_emu.py), against Pillow and OpenCV on x86-64 (libjpeg-turbo's SIMD
ISLOW path); and the fused ELA kernel on the frame built to drive its block stage to its extremes, under both block-stage builds."""
import io

import numpy as np
import pytest
from PIL import Image

import jpeg_craft as jc
from dct_helpers import np_hist, qtab_of
from helpers import adversarial_blocks_frame
from oracle import c_oracle
from test_jpeg_extremes_emu import CORPUS, FILES, reference
from v5ela.records import as_records
from v5ela.synth import gen_frame

pytestmark = pytest.mark.gpu


def normal_files():
    """Pixel-derived files of the corpus' sizes and layouts, to share a call with the crafted ones."""
    out = []
    for k, (layout, (h, w)) in enumerate(jc.SIZES.items()):
        buf = io.BytesIO()
        frame = gen_frame(k, h, w, 7)
        if layout == "gray":
            Image.fromarray(frame[..., 1]).save(buf, "JPEG", quality=85)
        else:
            Image.fromarray(frame).save(buf, "JPEG", quality=85, subsampling={"444": 0, "422": 1, "420": 2}[layout])
        out.append((f"normal_{layout}", buf.getvalue()))
    return out


@pytest.fixture(scope="module")
def mixed():
    import platform

    if platform.machine().lower() not in ("x86_64", "amd64"):
        pytest.skip(f"the reference is libjpeg-turbo's x86 SIMD inverse DCT; Pillow / OpenCV on {platform.machine()} run other code")
    normals, files = normal_files(), []
    for i, item in enumerate(FILES):                  # a normal file after every tenth crafted one
        files.append(item)
        if i % 10 == 0:
            files.append(normals[i // 10 % len(normals)])
    refs = [reference(data) for _, data in files]
    bad = [name for (name, _), r in zip(files, refs) if r is None]
    if bad:
        pytest.skip(f"Pillow and OpenCV decode {len(bad)} files differently (first: {bad[0]}): no single reference")
    return files, refs


@pytest.mark.parametrize("path", ["one", "three"])
def test_decode_host_equals_pillow_and_opencv(monkeypatch, mixed, path):
    """v5ela_jpeg_decode_host: every crafted file and the normal ones between them in one call."""
    from v5ela import jpeg

    monkeypatch.setenv("V5ELA_HUFF_PATH", path)
    files, refs = mixed
    outs = jpeg.decode_host([d for _, d in files], want_rgb=True, want_gray=True)
    for (name, _), o, r in zip(files, outs, refs):
        assert np.array_equal(o["rgb"], r["rgb"]), name
        assert np.array_equal(o["gray"], r["gray"]), name


@pytest.mark.parametrize("path", ["one", "three"])
def test_decode_on_device_equals_pillow_and_opencv(monkeypatch, mixed, path):
    """v5ela_jpeg_decode (one call per size: the device entry point takes files of one size)."""
    import torch
    from v5ela import jpeg

    monkeypatch.setenv("V5ELA_HUFF_PATH", path)
    files, refs = mixed
    groups = {}
    for item, r in zip(files, refs):
        groups.setdefault(r["gray"].shape, []).append((item, r))
    for shape, group in groups.items():
        out = jpeg.decode_batch([d for (_, d), _ in group], want_rgb=True, want_gray=True)
        torch.cuda.synchronize()
        assert (out["status"].cpu().numpy() == 0).all(), shape
        rgb, gray = out["rgb"].cpu().numpy(), out["gray"].cpu().numpy()
        for k, ((name, _), r) in enumerate(group):
            assert np.array_equal(rgb[k], r["rgb"]), name
            assert np.array_equal(gray[k], r["gray"]), name


@pytest.mark.parametrize("path", ["one", "three"])
def test_dct_stats_histograms_of_crafted_files(monkeypatch, path):
    """Independent of the inverse DCT: the coefficient histograms (+-64 saturating bins) of the crafted files equal NumPy's over
    the oracle's coefficients, and the tables read back are the files' own (16-bit ones included)."""
    import torch
    from v5ela import jpeg

    monkeypatch.setenv("V5ELA_HUFF_PATH", path)
    files = [d for _, d in FILES]
    out = jpeg.dct_stats(files)
    torch.cuda.synchronize()
    assert (out["status"].cpu().numpy() == 0).all()
    hist = out["hist"].cpu().numpy().view(np.uint32)
    qtab = out["qtab"].cpu().numpy()
    for i, (name, data) in enumerate(FILES):
        assert np.array_equal(hist[i], np_hist(data)), name
        assert np.array_equal(qtab[i], qtab_of(data)), name
    for i, e in enumerate(CORPUS):
        assert (qtab[i][0] == e["qt"]).all(), e["name"]


def test_analyze_jpeg_files_equals_pillow_then_oracle(mixed):
    """Crafted files of one size through decode + fused kernel on the GPU, against Pillow's decode through the C oracle."""
    import torch
    import v5ela

    files, _ = mixed
    h, w = jc.SIZES["420"]
    blobs = [d for _, d in files if Image.open(io.BytesIO(d)).size == (w, h)]
    assert len(blobs) > 100
    out = v5ela.analyze_jpeg_files(blobs, quality=90, want_residual=True)
    torch.cuda.synchronize()
    decoded = np.stack([np.asarray(Image.open(io.BytesIO(b)).convert("RGB")) for b in blobs])
    assert np.array_equal(out["rgb"].cpu().numpy(), decoded)
    recs, resid = c_oracle.analyze(decoded, 90, want_residual=True)
    assert np.array_equal(out["residual"].cpu().numpy(), resid)
    assert as_records(out["records"].cpu()).tobytes() == recs.tobytes()
    assert (out["status"].cpu().numpy() == 0).all()


# ------------------------------------------------------------------------------------- the fused kernel's extreme blocks
def _ghost_of(residual):
    h, w, _ = residual.shape
    mh, mw = -(-h // 16), -(-w // 16)
    sq = np.zeros((16 * mh, 16 * mw), np.int64)
    sq[:h, :w] = (residual.astype(np.int64) ** 2).sum(axis=2)
    return sq.reshape(mh, 16, mw, 16).sum(axis=(1, 3))


def test_adversarial_blocks_sweep_every_quality(block_stage):
    """The frames built to maximise the block stage's 16-bit hand-offs (DESIGN.md 4.1), at every quality 1..100 in one sweep with
    ghost maps: records equal the C oracle's, maps the NumPy block sums of its residual."""
    import torch
    import v5ela

    frames = list(adversarial_blocks_frame())
    qualities = list(range(1, 101))
    out = v5ela.analyze_sweep([torch.from_numpy(f).cuda() for f in frames], qualities, want_ghost=True)
    torch.cuda.synchronize()
    for q, qual in enumerate(qualities):
        got = as_records(out["records"][q].cpu())
        for i, f in enumerate(frames):
            o = c_oracle.analyze_frame(f, qual)
            assert got[i].tobytes() == o["record"].tobytes(), (qual, i)
            assert np.array_equal(out["ghost"][q][i].cpu().numpy(), _ghost_of(o["residual"])), (qual, i)


@pytest.mark.parametrize("q", [1, 2, 50, 100])
def test_adversarial_blocks_records_only_fast(block_stage, q):
    """Records-only calls on the adversarial frames (widths multiples of 16) take the FAST instantiation and equal the oracle."""
    import torch
    import v5ela
    from v5ela.batch import get_handle

    hd = get_handle(torch.cuda.current_device())
    for f in adversarial_blocks_frame():
        rec = as_records(v5ela.analyze_batch(torch.from_numpy(f).cuda()[None], quality=q)["records"].cpu())
        assert hd.last_instantiation == "fast"
        assert rec[0].tobytes() == c_oracle.analyze_frame(f, q)["record"].tobytes()
