"""GPU: a handle owns what its entry points allocate. The device workspaces, pinned staging buffers, streams and events live in
members of the handle (csrc/v5ela_handle.h), so v5ela_destroy releases all of them."""
import hashlib

import numpy as np
import pytest

from v5ela.synth import gen_batch, gen_frame

pytestmark = pytest.mark.gpu

GB, MB = 1 << 30, 1 << 20
BIG = (64, 1080, 1920)                     # analyze_host batch: d_in, d_res and d_enh of the handle are ~400 MB each
SMALL = (4, 256, 384)
CROPS = [(257, 301), (96, 160), (33, 47)]


def _inputs():
    """Every input and device output buffer of a cycle, allocated once, so that a cycle allocates nothing but the handle's own."""
    import torch

    from v5ela import jpeg

    n, h, w = SMALL
    cap = jpeg.default_capacity(h, w, 3)
    rgb = gen_batch(0, n, h, w, seed=5)
    crops = [gen_frame(i, ch, cw, 6) for i, (ch, cw) in enumerate(CROPS)]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    dz = lambda shape, dt=torch.uint8: torch.zeros(shape, dtype=dt, device="cuda")  # noqa: E731
    return {
        "big": np.random.default_rng(7).integers(0, 256, BIG + (3,), dtype=np.uint8),
        "rgb": rgb, "d_rgb": dev(rgb), "gray": np.ascontiguousarray(rgb[..., 1]), "d_gray": dev(rgb[..., 1]),
        "crops": crops, "d_crops": [dev(c) for c in crops], "cap": cap,
        "d_rec": dz((n, 3144)), "d_rec_ex": dz((n, 3144)), "d_res_ex": dz((n, h, w, 3)), "d_hist": dz((n, 256), torch.int32),
        "d_rec_rag": dz((len(CROPS), 3144)), "d_enh_rag": dz(CROPS[0] + (3,)), "d_spec": dz((n, h, w)),
        "d_enc": dz((n, cap)), "d_sizes": dz(n, torch.int32), "d_dec": dz((n, h, w, 3)), "d_status": dz(n, torch.int32),
    }


def _descs(frames, enhanced):
    from v5ela import _abi

    descs = (_abi.FrameDesc * len(frames))()
    for i, f in enumerate(frames):
        host = isinstance(f, np.ndarray)
        descs[i].rgb = f.ctypes.data if host else f.data_ptr()
        descs[i].height, descs[i].width = f.shape[0], f.shape[1]
        descs[i].row_stride_bytes = f.strides[0] if host else f.stride(0)
        e = enhanced[i]
        descs[i].enhanced = None if e is None else (e.ctypes.data if host else e.data_ptr())
    return descs


def _cycle(inp):
    """Creates a handle, drives every entry point that owns a workspace, closes the handle.
    -> (device bytes the open handle held, {output name: bytes})"""
    import torch

    from v5ela import _abi, jpeg

    n, h, w = SMALL
    cap = inp["cap"]
    out = {}
    torch.cuda.synchronize()
    free_before = torch.cuda.mem_get_info()[0]
    hd = _abi.Handle(torch.cuda.current_device())
    stream = torch.cuda.current_stream().cuda_stream
    hd.profile_enable(True)
    hd.profile_read(True)

    d_rgb, fs, rs = inp["d_rgb"], inp["d_rgb"].stride(0), inp["d_rgb"].stride(1)
    hd.analyze(d_rgb.data_ptr(), n, h, w, fs, rs, inp["d_rec"].data_ptr(), None, stream)
    hd.analyze(d_rgb.data_ptr(), n, h, w, fs, rs, inp["d_rec_ex"].data_ptr(), inp["d_res_ex"].data_ptr(), stream,
               d_tex_hist=inp["d_hist"].data_ptr())
    hd.analyze_ragged(_descs(inp["d_crops"], [inp["d_enh_rag"], None, None]), len(CROPS), inp["d_rec_rag"].data_ptr(), stream)
    rag_recs = np.zeros((len(CROPS), 3144), np.uint8)
    rag_enh = [np.zeros_like(c) for c in inp["crops"]]
    hd.analyze_ragged_host(_descs(inp["crops"], rag_enh), len(CROPS), rag_recs.ctypes.data)
    out["ragged_host"] = rag_recs.tobytes() + b"".join(e.tobytes() for e in rag_enh)

    big = inp["big"]
    for label, st in (("sync", None), ("stream", stream)):
        recs, res, enh = np.zeros((BIG[0], 3144), np.uint8), np.empty_like(big), np.empty_like(big)
        hd.analyze_host(big.ctypes.data, *BIG, recs.ctypes.data, res.ctypes.data, enh.ctypes.data, stream=st)
        torch.cuda.synchronize()
        out[f"analyze_host_{label}"] = recs.tobytes() + hashlib.sha256(res).digest() + hashlib.sha256(enh).digest()

    d_gray = inp["d_gray"]
    hd.spectrum(d_gray.data_ptr(), n, h, w, d_gray.stride(0), d_gray.stride(1), inp["d_spec"].data_ptr(), stream)
    spec = np.empty_like(inp["gray"])
    hd.spectrum_host(inp["gray"].ctypes.data, n, h, w, spec.ctypes.data)
    out["spectrum_host"] = spec.tobytes()

    hd.jpeg_encode(d_rgb.data_ptr(), n, h, w, 3, fs, rs, 90, inp["d_enc"].data_ptr(), cap, inp["d_sizes"].data_ptr(), stream)
    enc, sizes = np.zeros((n, cap), np.uint8), np.zeros(n, np.int32)
    hd.jpeg_encode_host(inp["rgb"].ctypes.data, n, h, w, 3, 90, enc.ctypes.data, cap, sizes.ctypes.data)
    files = [enc[i, :sizes[i]].tobytes() for i in range(n)]
    out["jpeg_encode_host"] = b"".join(files)
    keep, ptrs, lens = jpeg._file_table(files)
    hd.jpeg_decode(ptrs, lens, n, inp["d_dec"].data_ptr(), None, None, None, inp["d_status"].data_ptr(), stream)
    rgb, gray = np.zeros((n, h, w, 3), np.uint8), np.zeros((n, h, w), np.uint8)
    hd.jpeg_decode_host(ptrs, lens, n, rgb.ctypes.data, None, gray.ctypes.data, None)
    out["jpeg_decode_host"] = rgb.tobytes() + gray.tobytes()
    del keep

    out["profiled_launches"] = str(hd.profile_read(True)[1]).encode()
    torch.cuda.synchronize()
    held = free_before - torch.cuda.mem_get_info()[0]
    hd.close()
    for k in ("d_rec", "d_rec_ex", "d_res_ex", "d_hist", "d_rec_rag", "d_enh_rag", "d_spec", "d_sizes", "d_dec", "d_status"):
        out[k] = inp[k].cpu().numpy().tobytes()
    sz = inp["d_sizes"].cpu().numpy()
    out["d_enc"] = b"".join(inp["d_enc"][i, :int(sz[i])].cpu().numpy().tobytes() for i in range(n))
    return held, out


def test_destroy_releases_what_the_handle_held():
    """Three cycles of create / every workspace-owning entry point / close leave free device memory where it was, and give the
    same results each time. Free memory is read for the whole device, which other processes share: the handle is made to hold
    at least 1 GB and the cycles may leave at most 256 MB behind, so that another process's allocations during the test are
    unlikely to decide it either way."""
    import torch

    inp = _inputs()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    baseline = torch.cuda.mem_get_info()[0]
    results = []
    for _ in range(3):
        held, out = _cycle(inp)
        assert held >= GB, f"the open handle held only {held / MB:.0f} MB"
        results.append(out)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    lost = baseline - torch.cuda.mem_get_info()[0]
    assert lost <= 256 * MB, f"{lost / MB:.0f} MB of device memory not released by three closed handles"
    assert results[0].keys() == results[-1].keys()
    for k in results[0]:
        assert results[0][k] == results[-1][k], k
