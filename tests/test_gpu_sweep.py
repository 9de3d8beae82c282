"""GPU: quality sweeps (v5ela_analyze_sweep / _host, include/v5ela.h) — every frame at many JPEG qualities in one launch sequence, with
the JPEG-ghost maps. Byte identity with the per-quality calls, the C oracle and NumPy block sums of its residual; both block-stage
builds."""
import io

import numpy as np
import pytest

from oracle import c_oracle
from v5ela.records import RECORD_DTYPE, as_records, ghost_curve
from v5ela.synth import gen_frame

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("block_stage")]

SIZES = [(1, 1), (17, 33), (257, 301), (45, 61), (100, 1000), (360, 640), (271, 481), (9, 976)]


def ghost_of(residual):
    h, w, _ = residual.shape
    mh, mw = -(-h // 16), -(-w // 16)
    sq = np.zeros((16 * mh, 16 * mw), np.int64)
    sq[:h, :w] = (residual.astype(np.int64) ** 2).sum(axis=2)
    return sq.reshape(mh, 16, mw, 16).sum(axis=(1, 3))


def mixed_frames(seed=0):
    rng = np.random.default_rng(seed)
    return [gen_frame(k, h, w, seed) if k % 2 == 0 else rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for k, (h, w) in enumerate(SIZES)]


def handle():
    import torch
    from v5ela.batch import get_handle

    return get_handle(torch.cuda.current_device())


def test_sweep_equals_ragged_calls_mixed_sizes():
    import torch
    import v5ela

    qualities = [30, 75, 90, 75, 100]
    dev = [torch.from_numpy(f).cuda() for f in mixed_frames(1)]
    out = v5ela.analyze_sweep(dev, qualities, want_ghost=True)
    for q, qual in enumerate(qualities):
        ref = v5ela.analyze_ragged(dev, quality=qual)["records"]
        torch.cuda.synchronize()
        assert torch.equal(out["records"][q], ref), qual
    assert len(out["ghost"]) == len(qualities) and all(len(g) == len(dev) for g in out["ghost"])


def test_sweep_views_into_one_keyframe():
    """Crops as strided, unaligned views of a device-resident keyframe, as analyze_ragged takes them."""
    import torch
    import v5ela

    t = torch.from_numpy(gen_frame(3, 720, 1280, 2)).cuda()
    boxes = [(0, 0, 720, 1280), (13, 7, 300, 411), (100, 100, 101, 101), (5, 640, 250, 1279), (333, 222, 590, 523)]
    views = [t[y1:y2, x1:x2] for (y1, x1, y2, x2) in boxes]
    qualities = [60, 90]
    out = v5ela.analyze_sweep(views, qualities)
    for q, qual in enumerate(qualities):
        ref = v5ela.analyze_ragged(views, quality=qual)["records"]
        torch.cuda.synchronize()
        assert torch.equal(out["records"][q], ref), qual


def test_sweep_1080p_equals_uniform_batches():
    """8 x 1080p at {75, 85, 90, 95}: the same bytes as four analyze_batch calls (which take the FAST instantiation)."""
    import torch
    import v5ela
    from v5ela.synth import gen_batch_torch

    t = gen_batch_torch(0, 8, 1080, 1920, seed=5)
    qualities = [75, 85, 90, 95]
    out = v5ela.analyze_sweep(t, qualities, want_ghost=True)
    assert out["ghost"].shape == (4, 8, 68, 120) and out["ghost"].dtype == torch.int32
    for q, qual in enumerate(qualities):
        ref = v5ela.analyze_batch(t, quality=qual)["records"]
        torch.cuda.synchronize()
        assert torch.equal(out["records"][q], ref), qual
    # the ghost maps add up to the records' ela_sumsq
    recs = as_records(out["records"].reshape(-1, 3144)).reshape(4, 8)
    sums = out["ghost"].to(torch.int64).sum(dim=(2, 3)).cpu().numpy()
    assert np.array_equal(sums, recs["ela_sumsq"].sum(axis=-1).astype(np.int64))


def test_sweep_vs_oracle_records_and_ghost_maps():
    import torch
    import v5ela

    frames = mixed_frames(2)
    qualities = [1, 50, 90, 100]
    out = v5ela.analyze_sweep([torch.from_numpy(f).cuda() for f in frames], qualities, want_ghost=True)
    torch.cuda.synchronize()
    recs = as_records(out["records"].reshape(-1, 3144)).reshape(len(qualities), len(frames))
    for q, qual in enumerate(qualities):
        for i, f in enumerate(frames):
            o = c_oracle.analyze_frame(f, qual)
            assert recs[q, i].tobytes() == o["record"].tobytes(), (qual, f.shape)
            assert np.array_equal(out["ghost"][q][i].cpu().numpy(), ghost_of(o["residual"])), (qual, f.shape)


def test_host_and_device_entry_points_agree():
    import torch
    import v5ela
    from v5ela import host

    frames = mixed_frames(3)
    qualities = [95, 70, 70, 40]
    dev = v5ela.analyze_sweep([torch.from_numpy(f).cuda() for f in frames], qualities, want_ghost=True)
    torch.cuda.synchronize()
    recs, ghost = host.analyze_sweep_host(frames, qualities, want_ghost=True)
    assert recs.shape == (4, len(frames))
    assert recs.tobytes() == dev["records"].cpu().numpy().tobytes()
    for q in range(len(qualities)):
        for i in range(len(frames)):
            assert np.array_equal(ghost[q][i].view(np.int32), dev["ghost"][q][i].cpu().numpy())
    # a uniform array: the (nq, N, mh, mw) layout, and records without maps
    batch = np.stack([gen_frame(k, 64, 96, 1) for k in range(3)])
    r2, g2 = host.analyze_sweep_host(batch, [90, 50], want_ghost=True)
    r3, g3 = host.analyze_sweep_host(batch, [90, 50])
    assert g2.shape == (2, 3, 4, 6) and g3 is None and r2.tobytes() == r3.tobytes()
    d2 = v5ela.analyze_sweep(torch.from_numpy(batch).cuda(), [90, 50], want_ghost=True)
    torch.cuda.synchronize()
    assert r2.tobytes() == d2["records"].cpu().numpy().tobytes()
    assert np.array_equal(g2.view(np.int32), d2["ghost"].cpu().numpy())


@pytest.mark.parametrize("nq", [1, 20])
def test_two_launches_per_call(nq):
    import torch
    import v5ela

    hd = handle()
    dev = [torch.from_numpy(f).cuda() for f in mixed_frames(4)]
    inst = hd.last_instantiation
    quality = hd.quality
    for want_ghost in (False, True):
        before = hd.launch_count
        v5ela.analyze_sweep(dev, list(range(5, 5 + 5 * nq, 5)), want_ghost=want_ghost)
        assert hd.launch_count == before + 2
    torch.cuda.synchronize()
    assert hd.last_instantiation == inst and hd.quality == quality


def test_refusals_launch_nothing():
    import torch
    from v5ela import _abi

    hd = handle()
    frames = [torch.from_numpy(f).cuda() for f in mixed_frames(5)[:3]]
    n = len(frames)
    records = torch.full((2, n, 3144), 0x5A, dtype=torch.uint8, device="cuda")

    def descs():
        d = (_abi.FrameDesc * n)()
        for i, f in enumerate(frames):
            d[i].rgb, d[i].height, d[i].width, d[i].row_stride_bytes = f.data_ptr(), f.shape[0], f.shape[1], f.stride(0)
        return d

    cases = []
    d = descs()
    cases.append((d, [90, 101], "quality 1"))
    cases.append((d, [0, 90], "quality 0"))
    cases.append((d, [], "nq"))
    cases.append((d, [90] * 101, "nq"))
    d = descs(); d[2].width = 0
    cases.append((d, [90, 75], "frame 2"))
    d = descs(); d[1].row_stride_bytes = 3 * frames[1].shape[1] - 1
    cases.append((d, [90, 75], "frame 1"))
    d = descs(); d[0].residual = records.data_ptr()
    cases.append((d, [90, 75], "frame 0"))
    d = descs(); d[1].enhanced = records.data_ptr()
    cases.append((d, [90, 75], "frame 1"))
    for d, qualities, where in cases:
        before = hd.launch_count
        with pytest.raises(_abi.V5ElaError) as ei:
            hd.analyze_sweep(d, n, qualities, records.data_ptr(), None, torch.cuda.current_stream().cuda_stream)
        assert ei.value.status == -1 and where in str(ei.value), (where, str(ei.value))
        assert hd.launch_count == before
        with pytest.raises(_abi.V5ElaError):
            hd.analyze_sweep(d, -1, [90], records.data_ptr(), None, None)
    torch.cuda.synchronize()
    assert bool((records == 0x5A).all())
    host_recs = np.zeros((2, n), RECORD_DTYPE)
    hframes = mixed_frames(5)[:3]
    hd_ = (_abi.FrameDesc * n)()
    for i, f in enumerate(hframes):
        hd_[i].rgb, hd_[i].height, hd_[i].width, hd_[i].row_stride_bytes = f.ctypes.data, f.shape[0], f.shape[1], f.strides[0]
    hd_[1].residual = host_recs.ctypes.data
    before = hd.launch_count
    with pytest.raises(_abi.V5ElaError) as ei:
        hd.analyze_sweep_host(hd_, n, [90, 75], host_recs.ctypes.data, None)
    assert "frame 1" in str(ei.value) and hd.launch_count == before and not host_recs.tobytes().strip(b"\0")


def test_one_handle_on_two_streams():
    """Sweeps on one stream, analyze_batch on another, alternately through one handle: the handle-owned ticket counter and tables
    are reused by every call, so each call waits for the previous one's kernels. Results against serial runs."""
    import torch
    import v5ela
    from v5ela.synth import gen_batch_torch

    big = gen_batch_torch(0, 24, 720, 1280, seed=3)
    small = [t for t in gen_batch_torch(7, 3, 96, 160, seed=4)]
    qualities = [60, 75, 90]
    ref_big = v5ela.analyze_batch(big)["records"].clone()
    ref_sweep = v5ela.analyze_sweep(small, qualities, want_ghost=True)
    ref_rec, ref_ghost = ref_sweep["records"].clone(), [[g.clone() for g in gq] for gq in ref_sweep["ghost"]]
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    outs = []
    for _ in range(10):
        with torch.cuda.stream(s1):
            a = v5ela.analyze_batch(big)["records"]
        with torch.cuda.stream(s2):
            b = v5ela.analyze_sweep(small, qualities, want_ghost=True)
        outs.append((a, b))
    torch.cuda.synchronize()
    for a, b in outs:
        assert torch.equal(a, ref_big) and torch.equal(b["records"], ref_rec)
        assert all(torch.equal(b["ghost"][q][i], ref_ghost[q][i]) for q in range(3) for i in range(3))


def test_spliced_frame_ghost_map():
    """Left half from a q60 file, right half from a q90 file, the whole saved at q95: re-saved at q60, the left half's ghost map is
    lower than the right half's."""
    import torch
    import v5ela
    from PIL import Image

    def jpeg_roundtrip(a, q):
        buf = io.BytesIO()
        Image.fromarray(a).save(buf, "JPEG", quality=q)
        return np.array(Image.open(io.BytesIO(buf.getvalue())).convert("RGB"))

    src = gen_frame(0, 288, 352, 0)
    spliced = np.concatenate([jpeg_roundtrip(src, 60)[:, :176], jpeg_roundtrip(src, 90)[:, 176:]], axis=1)
    frame = jpeg_roundtrip(np.ascontiguousarray(spliced), 95)
    out = v5ela.analyze_sweep([torch.from_numpy(frame).cuda()], [60, 75, 90], want_ghost=True)
    torch.cuda.synchronize()
    g60 = out["ghost"][0][0].cpu().numpy().astype(np.float64)
    assert g60.shape == (18, 22)
    assert g60[:, :11].mean() < g60[:, 11:].mean()
    recs = as_records(out["records"].reshape(-1, 3144)).reshape(3, 1)
    assert ghost_curve(recs, 288 * 352).shape == (3, 1)
