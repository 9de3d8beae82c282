"""Batch entry point: ``analyze_batch(frames_u8[N,H,W,3]) -> records (+ residual / enhanced maps)`` on one B200.

PyTorch is plumbing here (device memory, streams); the work is one call into libv5ela.so (include/v5ela.h).
There is no CPU path: tensors must live on a CUDA device and the library must load.
"""
from __future__ import annotations

from . import _abi
from ._abi import get_handle
from .records import RECORD_BYTES


def analyze_batch(frames, quality: int = 90, want_residual: bool = False, want_enhanced: bool = False,
                  records_out=None, residual_out=None, handle=None, want_tex_hist: bool = False):
    """Run the fused ELA + texture kernel over a batch of RGB frames.

    frames : torch.uint8 CUDA tensor, shape (N, H, W, 3), innermost two dims dense (row/frame strides may be padded).
    Returns a dict: ``records`` uint8 (N, 3144) on the same device (view with ``records.as_records`` on the host),
    and, when asked, ``residual`` (= the reference's ``diff``, v5_texture_ela.py:70) and ``enhanced``
    (= ``ImageEnhance.Brightness(diff).enhance(scale)``, v5…:78), both uint8 (N, H, W, 3); with ``want_tex_hist`` also
    ``tex_hist`` int32 (N, 256), the histogram of min(|Laplacian of the luma|, 255) (SURVEY.md §8a, optional field).
    Asynchronous on torch's current stream.
    """
    import torch

    if not isinstance(frames, torch.Tensor) or frames.dtype != torch.uint8:
        raise TypeError("frames must be a torch.uint8 tensor")
    if frames.dim() != 4 or frames.shape[-1] != 3:
        raise ValueError("frames must have shape (N, H, W, 3)")
    if not frames.is_cuda:
        raise ValueError("frames must be a CUDA tensor (this path has no CPU implementation)")
    if frames.stride(3) != 1 or frames.stride(2) != 3:
        frames = frames.contiguous()
    n, h, w, _ = frames.shape
    dev = frames.device
    hd = handle or get_handle(dev.index if dev.index is not None else torch.cuda.current_device())
    if hd.quality != quality:
        hd.set_quality(quality)
    records = records_out if records_out is not None else torch.empty((n, RECORD_BYTES), dtype=torch.uint8, device=dev)
    out = {"records": records}
    residual = None
    if want_residual or want_enhanced:
        residual = residual_out if residual_out is not None else torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    tex_hist = torch.zeros((n, 256), dtype=torch.int32, device=dev) if want_tex_hist else None
    if tex_hist is not None:
        out["tex_hist"] = tex_hist
    if n == 0 or h == 0 or w == 0:
        if residual is not None:
            out["residual"] = residual
            if want_enhanced:
                out["enhanced"] = torch.empty_like(residual)
        return out
    stream = torch.cuda.current_stream(dev).cuda_stream
    hd.analyze(frames.data_ptr(), n, h, w, frames.stride(0), frames.stride(1), records.data_ptr(),
               residual.data_ptr() if residual is not None else None, stream,
               tex_hist.data_ptr() if tex_hist is not None else None)
    if residual is not None:
        out["residual"] = residual
    if want_enhanced:
        enhanced = torch.empty_like(residual)
        hd.enhance(residual.data_ptr(), records.data_ptr(), n, h, w, enhanced.data_ptr(), stream)
        out["enhanced"] = enhanced
    return out


def analyze_ragged(frames, quality: int = 90, want_residual: bool = False, want_enhanced: bool = False, records_out=None, handle=None):
    """The fused kernel over frames of DIFFERENT sizes in one launch (v5ela_analyze_ragged) — the reference node's real input: face
    crops (v5_texture_ela.py:56-64), here as they lie on the device, e.g. strided views into decoded keyframes (v5ela.handoff).

    frames : sequence of torch.uint8 CUDA tensors (H_i, W_i, 3), pixels dense (stride 3 / 1), any row stride, all on one device.
    Returns ``records`` uint8 (N, 3144) and, when asked, lists ``residual`` / ``enhanced`` of (H_i, W_i, 3) tensors. Asynchronous on
    torch's current stream; no per-frame launches and no host synchronisation.
    """
    import torch

    n = len(frames)
    if n == 0:
        dev = torch.device("cuda", torch.cuda.current_device())
        out = {"records": torch.empty((0, RECORD_BYTES), dtype=torch.uint8, device=dev)}
        if want_residual:
            out["residual"] = []
        if want_enhanced:
            out["enhanced"] = []
        return out
    dev = frames[0].device
    views = []
    for f in frames:
        if not isinstance(f, torch.Tensor) or f.dtype != torch.uint8 or not f.is_cuda or f.dim() != 3 or f.shape[-1] != 3:
            raise ValueError("frames must be torch.uint8 CUDA tensors of shape (H, W, 3)")
        if f.device != dev:
            raise ValueError("all frames must live on one device")
        if f.shape[0] == 0 or f.shape[1] == 0:
            raise ValueError("empty frame in a ragged batch")
        if f.stride(2) != 1 or f.stride(1) != 3:
            f = f.contiguous()
        views.append(f)
    hd = handle or get_handle(dev.index if dev.index is not None else torch.cuda.current_device())
    if hd.quality != quality:
        hd.set_quality(quality)
    records = records_out if records_out is not None else torch.empty((n, RECORD_BYTES), dtype=torch.uint8, device=dev)
    out = {"records": records}
    resid = enh = None
    if want_residual:                                           # one arena per kind, the maps are views into it
        sizes = [f.shape[0] * f.shape[1] * 3 for f in views]
        offs = [0]
        for s_ in sizes:
            offs.append(offs[-1] + (s_ + 255) // 256 * 256)
        arena = torch.empty(offs[-1], dtype=torch.uint8, device=dev)
        resid = [arena[offs[i]:offs[i] + sizes[i]].view(views[i].shape[0], views[i].shape[1], 3) for i in range(n)]
        out["residual"] = resid
    if want_enhanced:
        sizes = [f.shape[0] * f.shape[1] * 3 for f in views]
        offs = [0]
        for s_ in sizes:
            offs.append(offs[-1] + (s_ + 255) // 256 * 256)
        arena_e = torch.empty(offs[-1], dtype=torch.uint8, device=dev)
        enh = [arena_e[offs[i]:offs[i] + sizes[i]].view(views[i].shape[0], views[i].shape[1], 3) for i in range(n)]
        out["enhanced"] = enh
    descs = (_abi.FrameDesc * n)()
    for i, f in enumerate(views):
        descs[i].rgb = f.data_ptr()
        descs[i].height, descs[i].width = int(f.shape[0]), int(f.shape[1])
        descs[i].row_stride_bytes = int(f.stride(0))
        descs[i].residual = resid[i].data_ptr() if resid is not None else None
        descs[i].enhanced = enh[i].data_ptr() if enh is not None else None
    hd.analyze_ragged(descs, n, records.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    out["_keepalive"] = views                                   # contiguous copies (if any) must outlive the asynchronous launch
    return out


def reduce_records(records, group: int, handle=None):
    """Per-video aggregation on the device: (N, 3144) -> (N // group, 3144)."""
    import torch

    n = records.shape[0]
    dev = records.device
    hd = handle or get_handle(dev.index if dev.index is not None else torch.cuda.current_device())
    out = torch.empty((n // group, RECORD_BYTES), dtype=torch.uint8, device=dev)
    if n:
        hd.reduce_records(records.data_ptr(), n, group, out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    return out


def spectrum_batch(gray, handle=None):
    """FFT log-magnitude spectrum images of a torch.uint8 CUDA tensor (N, H, W) -> uint8 (N, H, W); see include/v5ela.h."""
    import torch

    if not isinstance(gray, torch.Tensor) or gray.dtype != torch.uint8 or gray.dim() != 3 or not gray.is_cuda:
        raise ValueError("gray must be a torch.uint8 CUDA tensor of shape (N, H, W)")
    if gray.stride(2) != 1:
        gray = gray.contiguous()
    n, h, w = gray.shape
    dev = gray.device
    hd = handle or get_handle(dev.index if dev.index is not None else torch.cuda.current_device())
    out = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
    if n and h and w:
        hd.spectrum(gray.data_ptr(), n, h, w, gray.stride(0), gray.stride(1), out.data_ptr(),
                    torch.cuda.current_stream(dev).cuda_stream)
    return out


def analyze_jpeg_files(files, quality: int = 90, device=0, want_residual: bool = False, want_enhanced: bool = False, handle=None):
    """Keyframes / crops as the reference holds them — JPEG files (bytes), all of one size — decoded on the GPU (pixel-identical
    to Image.open(..).convert('RGB'), v5_texture_ela.py:64) and analysed without the pixels ever crossing PCIe: only the
    compressed bytes go up and the records come down. Returns analyze_batch's dict plus ``rgb`` (the decoded frames) and
    ``status`` (int32 per file, 0 = ok)."""
    from . import jpeg

    dec = jpeg.decode_batch(files, device=device, want_rgb=True, handle=handle)
    out = analyze_batch(dec["rgb"], quality=quality, want_residual=want_residual, want_enhanced=want_enhanced, handle=handle)
    out["rgb"] = dec["rgb"]
    out["status"] = dec["status"]
    return out

