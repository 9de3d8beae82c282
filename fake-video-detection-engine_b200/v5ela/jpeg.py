"""Codec rows on the GPU (include/v5ela.h, v5ela_jpeg_*): the JPEG files on either side of the ELA arithmetic.

  decode_host / decode_batch  : Image.open(crop).convert('RGB') and cv2.imread(crop, IMREAD_GRAYSCALE)
                                (reference v5_texture_ela.py:64, :83) — pixel-identical
  encode_host / encode_batch  : Image.save(.., 'JPEG', quality=q) and cv2.imwrite('.jpg', gray)
                                (reference v5_texture_ela.py:66-67, :80-81, :90-91) — byte-identical
  dct_stats / dct_stats_host  : per-frequency histograms of the files' quantised DCT coefficients, their quantisation tables
                                and a per-block map of aligned double compression (DESIGN.md §4.8)
  ijg_quality                 : the IJG quality whose tables a file's DQT equals
No CPU implementation exists behind these; files outside the decoder's supported set raise V5ElaError(status -5).
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _abi

UNSUPPORTED = -5


def info(data: bytes):
    """-> (height, width, channels) from the file's headers; raises V5ElaError for corrupt / unsupported files."""
    lib = _abi.load()
    h, w, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    buf = np.frombuffer(data, np.uint8)                                    # no copy
    rc = lib.v5ela_jpeg_info(buf.ctypes.data, len(data), ctypes.byref(h), ctypes.byref(w), ctypes.byref(c))
    if rc != 0:
        raise _abi.V5ElaError(rc, lib.v5ela_status_string(rc).decode())
    return h.value, w.value, c.value


def info_batch(files, table=None):
    """-> int32 array (N, 3) of (height, width, channels), one library call for the whole list."""
    lib = _abi.load()
    n = len(files)
    keep, ptrs, lens = table or _file_table(files)
    dims = np.zeros((n, 3), np.int32)
    bad = ctypes.c_int(-1)
    rc = lib.v5ela_jpeg_info_batch(ptrs, lens, n, dims.ctypes.data, ctypes.byref(bad))
    if rc != 0:
        raise _abi.V5ElaError(rc, f"{lib.v5ela_status_string(rc).decode()} (file {bad.value})")
    return dims


def _file_table(files):
    """ctypes arrays (pointers, lengths) over a list of bytes objects / uint8 arrays (e.g. views into one pinned arena); the
    first return value keeps the buffers alive."""
    n = len(files)
    keep = [f if isinstance(f, np.ndarray) else np.frombuffer(f, np.uint8) for f in files]
    ptrs = (ctypes.c_void_p * n)(*[k.ctypes.data for k in keep])
    lens = (ctypes.c_int64 * n)(*[len(f) for f in files])
    return keep, ptrs, lens


def default_capacity(h: int, w: int, channels: int) -> int:
    """Output bytes reserved per image by the wrappers: two bytes per sample plus the header; files that need more are
    reported, never truncated silently (re-run with capacity=bound(...))."""
    blocks = ((h + 15) // 16) * ((w + 15) // 16) * 6 if channels == 3 else ((h + 7) // 8) * ((w + 7) // 8)
    return blocks * 128 + 4096


def bound(h: int, w: int, channels: int) -> int:
    return int(_abi.load().v5ela_jpeg_bound(h, w, channels))


def encode_host(images: np.ndarray, quality: int, device: int = 0, capacity: int | None = None):
    """images: (N, H, W) gray or (N, H, W, 3) RGB uint8 host array -> list of N bytes objects (complete JPEG files)."""
    img = np.ascontiguousarray(images, dtype=np.uint8)
    if img.ndim not in (3, 4) or (img.ndim == 4 and img.shape[-1] != 3):
        raise ValueError("images must have shape (N, H, W) or (N, H, W, 3)")
    n, h, w = img.shape[:3]
    ch = 3 if img.ndim == 4 else 1
    if n == 0:
        return []
    cap = int(capacity or default_capacity(h, w, ch))
    out = np.empty((n, cap), np.uint8)
    sizes = np.zeros(n, np.int32)
    _abi.get_handle(device).jpeg_encode_host(img.ctypes.data, n, h, w, ch, int(quality), out.ctypes.data, cap, sizes.ctypes.data)
    if (sizes > cap).any():
        if capacity is None:
            return encode_host(images, quality, device, bound(h, w, ch))
        raise _abi.V5ElaError(-1, f"JPEG capacity {cap} too small (needed up to {int(sizes.max())})")
    return [out[i, :sizes[i]].tobytes() for i in range(n)]


def encode_batch(images, quality: int, capacity: int | None = None):
    """images: uint8 CUDA tensor (N, H, W) or (N, H, W, 3) (inner dims dense) -> (files uint8 [N, capacity], sizes int32 [N])
    on the same device, asynchronous on the current stream. sizes[i] > capacity marks a file that did not fit."""
    import torch

    if not images.is_cuda or images.dtype != torch.uint8:
        raise ValueError("encode_batch needs a uint8 CUDA tensor")
    ch = 3 if images.dim() == 4 else 1
    if images.dim() not in (3, 4) or (ch == 3 and (images.shape[-1] != 3 or images.stride(-1) != 1 or images.stride(-2) != 3)) or \
            (ch == 1 and images.stride(-1) != 1):
        raise ValueError("images must be (N, H, W) or (N, H, W, 3) with dense pixels")
    n, h, w = images.shape[:3]
    cap = int(capacity or default_capacity(h, w, ch))
    out = torch.empty((n, cap), dtype=torch.uint8, device=images.device)
    sizes = torch.zeros(n, dtype=torch.int32, device=images.device)
    if n:
        hd = _abi.get_handle(images.device.index or 0)
        hd.jpeg_encode(images.data_ptr(), n, h, w, ch, images.stride(0), images.stride(1), int(quality), out.data_ptr(), cap,
                       sizes.data_ptr(), torch.cuda.current_stream(images.device).cuda_stream)
    return out, sizes


def decode_host(files, want_rgb: bool = True, want_gray: bool = False, device: int = 0):
    """files: list of bytes -> list of dicts {'rgb': (H,W,3), 'gray': (H,W)} (keys as requested), host arrays."""
    n = len(files)
    if n == 0:
        return []
    table = _file_table(files)
    dims = [tuple(int(v) for v in d) for d in info_batch(files, table)]
    px = np.array([h * w for h, w, _ in dims], np.int64)
    offs = np.concatenate([[0], np.cumsum(px)])
    rgb = np.empty(3 * int(offs[-1]), np.uint8) if want_rgb else None
    gray = np.empty(int(offs[-1]), np.uint8) if want_gray else None
    keep, ptrs, lens = table
    _abi.get_handle(device).jpeg_decode_host(ptrs, lens, n, rgb.ctypes.data if want_rgb else None, None,
                                     gray.ctypes.data if want_gray else None, None)
    del keep
    out = []
    for i, (h, w, _) in enumerate(dims):
        d = {}
        if want_rgb:
            d["rgb"] = rgb[3 * offs[i]:3 * offs[i + 1]].reshape(h, w, 3)
        if want_gray:
            d["gray"] = gray[offs[i]:offs[i + 1]].reshape(h, w)
        out.append(d)
    return out


def decode_batch(files, device=0, want_rgb: bool = True, want_gray: bool = False, handle=None):
    """files: list of bytes (or uint8 arrays), all the same size -> {'rgb': uint8 CUDA tensor [N,H,W,3], 'gray': [N,H,W],
    'status': int32 [N]}, asynchronous on the current stream. Header parsing happens on the calling thread; pageable files are
    staged before the call returns, files that are views into pinned memory are read asynchronously (keep the arena alive)."""
    import torch

    n = len(files)
    dev = torch.device("cuda", device) if not isinstance(device, torch.device) else device
    table = _file_table(files)
    dims = info_batch(files, table)
    if n == 0 or (dims[:, :2] != dims[0, :2]).any():
        raise ValueError("decode_batch needs at least one file and files of one size; use decode_host for mixed sizes")
    h, w = int(dims[0, 0]), int(dims[0, 1])
    out = {"status": torch.zeros(n, dtype=torch.int32, device=dev)}
    if want_rgb:
        out["rgb"] = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    if want_gray:
        out["gray"] = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
    keep, ptrs, lens = table
    (handle or _abi.get_handle(dev.index or 0)).jpeg_decode(ptrs, lens, n, out["rgb"].data_ptr() if want_rgb else None, None,
                                           out["gray"].data_ptr() if want_gray else None, None, out["status"].data_ptr(),
                                           torch.cuda.current_stream(dev).cuda_stream)
    del keep
    return out


DQ_HIST_SHAPE = (3, 64, 129)


def _map_layout(files, table):
    """(per-file map shapes (ceil(H/8), ceil(W/8)), packed element offsets (N + 1))"""
    shapes = [((int(h) + 7) // 8, (int(w) + 7) // 8) for h, w, _ in info_batch(files, table)]
    offs = np.concatenate([[0], np.cumsum([a * b for a, b in shapes])]).astype(np.int64)
    return shapes, offs


def dct_stats(files, want_qtab: bool = True, want_map: bool = False, device=0, handle=None):
    """files: list of bytes (or uint8 arrays; any mix of sizes and layouts) -> dict of CUDA tensors, asynchronous on the current
    stream:
      'hist'   int32 (N, 3, 64, 129): [i][c][k][v + 64] counts the real blocks of component c of file i whose quantised coefficient
               at natural-order position k is v, clamped to -64..64 (the counts are uint32 in the library; int32 is a view)
      'qtab'   uint16 (N, 3, 64): each component's quantisation table, natural order (want_qtab)
      'map'    list of N float32 (ceil(H/8), ceil(W/8)) views into one arena: per luma block, the posterior that the block was not
               aligned-double-compressed (want_map)
      'status' int32 (N): 0, or -1 for a file whose entropy-coded data ends early
    Header parsing happens on the calling thread; files that are views into pinned memory are read asynchronously."""
    import torch

    n = len(files)
    dev = torch.device("cuda", device) if not isinstance(device, torch.device) else device
    out = {"hist": torch.zeros((n,) + DQ_HIST_SHAPE, dtype=torch.int32, device=dev),
           "status": torch.zeros(n, dtype=torch.int32, device=dev)}
    if want_qtab:
        out["qtab"] = torch.zeros((n, 3, 64), dtype=torch.uint16, device=dev)
    if n == 0:
        if want_map:
            out["map"] = []
        return out
    table = _file_table(files)
    arena = None
    if want_map:
        shapes, offs = _map_layout(files, table)
        arena = torch.empty(int(offs[-1]), dtype=torch.float32, device=dev)
        out["map"] = [arena[int(offs[i]):int(offs[i + 1])].view(shapes[i]) for i in range(n)]
    keep, ptrs, lens = table
    (handle or _abi.get_handle(dev.index or 0)).jpeg_dct_stats(
        ptrs, lens, n, out["hist"].data_ptr(), out["qtab"].data_ptr() if want_qtab else None,
        arena.data_ptr() if want_map else None, None, out["status"].data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    del keep
    return out


def dct_stats_host(files, want_qtab: bool = True, want_map: bool = False, device=0, handle=None):
    """The same as NumPy arrays ('hist' uint32, 'qtab' uint16, 'map' list of float32 views into one array); synchronous, and a file
    whose entropy-coded data ends early raises V5ElaError(-1)."""
    n = len(files)
    out = {"hist": np.zeros((n,) + DQ_HIST_SHAPE, np.uint32)}
    if want_qtab:
        out["qtab"] = np.zeros((n, 3, 64), np.uint16)
    if n == 0:
        if want_map:
            out["map"] = []
        return out
    table = _file_table(files)
    arena = None
    if want_map:
        shapes, offs = _map_layout(files, table)
        arena = np.empty(int(offs[-1]), np.float32)
        out["map"] = [arena[offs[i]:offs[i + 1]].reshape(shapes[i]) for i in range(n)]
    keep, ptrs, lens = table
    (handle or _abi.get_handle(device)).jpeg_dct_stats_host(ptrs, lens, n, out["hist"].ctypes.data,
                                                            out["qtab"].ctypes.data if want_qtab else None,
                                                            arena.ctypes.data if want_map else None, None)
    del keep
    return out


def ijg_quality(qtab):
    """qtab: one file's quantisation tables, natural order — (3, 64) as dct_stats returns them (components a one-component file
    lacks are zero), (2, 64) luma + chroma, or (64,) luma alone; a tensor or an array. -> the IJG quality 1..100 whose
    jpeg_set_quality tables (what libjpeg, and so PIL and OpenCV, write for `quality`) equal them, or None. Host only."""
    if hasattr(qtab, "detach"):
        qtab = qtab.detach().cpu().numpy()
    q = np.ascontiguousarray(np.asarray(qtab).reshape(-1, 64), dtype=np.uint16)
    if q.shape[0] not in (1, 2, 3):
        raise ValueError("qtab must hold one, two or three tables of 64 entries")
    chroma = None
    if q.shape[0] >= 2 and q[1:].any():
        if q.shape[0] == 3 and not np.array_equal(q[1], q[2]):
            return None                                                   # the IJG tables give Cb and Cr the same table
        chroma = q[1]
    r = _abi.load().v5ela_jpeg_ijg_quality(q[0].ctypes.data, chroma.ctypes.data if chroma is not None else None)
    if r < 0:
        raise _abi.V5ElaError(r, "v5ela_jpeg_ijg_quality: bad table")
    return int(r) or None
