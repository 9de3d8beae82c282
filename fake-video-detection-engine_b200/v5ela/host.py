"""NumPy-level entry point over ``v5ela_analyze_host`` (include/v5ela.h): host arrays in, host arrays out.

This is what the drop-in node uses (it needs no torch): frames are copied to the GPU, analysed by the fused kernel and
the records / residual / enhanced maps copied back. No CPU implementation exists behind it.
"""
from __future__ import annotations

import numpy as np

from ._abi import get_handle
from .records import RECORD_DTYPE


def analyze_frames_host(frames: np.ndarray, quality: int = 90, want_residual: bool = False, want_enhanced: bool = False,
                        device: int = 0):
    """frames: (N, H, W, 3) uint8 host array -> (records[N] structured, residual | None, enhanced | None)."""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    if frames.ndim != 4 or frames.shape[-1] != 3:
        raise ValueError("frames must have shape (N, H, W, 3)")
    n, h, w, _ = frames.shape
    recs = np.zeros(n, dtype=RECORD_DTYPE)
    residual = np.empty_like(frames) if want_residual else None
    enhanced = np.empty_like(frames) if want_enhanced else None
    if n == 0 or h == 0 or w == 0:
        return recs, residual, enhanced
    hd = get_handle(device)
    if hd.quality != quality:
        hd.set_quality(quality)
    hd.analyze_host(frames.ctypes.data, n, h, w, recs.ctypes.data,
                    residual.ctypes.data if residual is not None else None,
                    enhanced.ctypes.data if enhanced is not None else None, None)
    return recs, residual, enhanced


def analyze_ragged_host(frames, quality: int = 90, want_residual: bool = False, want_enhanced: bool = False, device: int = 0):
    """frames: sequence of (H_i, W_i, 3) uint8 host arrays of different sizes -> (records[N] structured, [residual_i] | None,
    [enhanced_i] | None) through ``v5ela_analyze_ragged_host``: one upload, one launch sequence, one download for the whole batch
    (the node's <= 3 face crops, v5_texture_ela.py:42,56-64)."""
    from ._abi import FrameDesc

    arrs = [np.ascontiguousarray(f, dtype=np.uint8) for f in frames]
    n = len(arrs)
    for a in arrs:
        if a.ndim != 3 or a.shape[-1] != 3 or a.shape[0] == 0 or a.shape[1] == 0:
            raise ValueError("frames must be non-empty (H, W, 3) arrays")
    recs = np.zeros(n, dtype=RECORD_DTYPE)
    residual = [np.empty_like(a) for a in arrs] if want_residual else None
    enhanced = [np.empty_like(a) for a in arrs] if want_enhanced else None
    if n == 0:
        return recs, residual, enhanced
    descs = (FrameDesc * n)()
    for i, a in enumerate(arrs):
        descs[i].rgb = a.ctypes.data
        descs[i].height, descs[i].width = a.shape[0], a.shape[1]
        descs[i].row_stride_bytes = a.strides[0]
        descs[i].residual = residual[i].ctypes.data if residual is not None else None
        descs[i].enhanced = enhanced[i].ctypes.data if enhanced is not None else None
    hd = get_handle(device)
    if hd.quality != quality:
        hd.set_quality(quality)
    hd.analyze_ragged_host(descs, n, recs.ctypes.data)
    return recs, residual, enhanced


def spectrum_host(gray: np.ndarray, device: int = 0) -> np.ndarray:
    """FFT log-magnitude spectrum image(s) (v5_texture_ela.py:84-88) of (H, W) or (N, H, W) uint8 host arrays."""
    g = np.ascontiguousarray(gray, dtype=np.uint8)
    single = g.ndim == 2
    if single:
        g = g[None]
    if g.ndim != 3:
        raise ValueError("gray must have shape (H, W) or (N, H, W)")
    out = np.empty_like(g)
    n, h, w = g.shape
    if n and h and w:
        get_handle(device).spectrum_host(g.ctypes.data, n, h, w, out.ctypes.data)
    return out[0] if single else out
