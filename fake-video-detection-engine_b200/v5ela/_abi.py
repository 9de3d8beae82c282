"""ctypes binding of libv5ela.so (include/v5ela.h). No CPU fallback: a missing or unloadable library is an error."""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# V5ELA_LIB: development knob — load another build of the SAME library (kernel-tuning variants under profiles/variants/).
LIB_PATH = os.environ.get("V5ELA_LIB") or os.path.join(_HERE, "libv5ela.so")

# Every symbol include/v5ela.h declares; tests assert the built library exports exactly these.
EXPORTS = (
    "v5ela_abi_version", "v5ela_record_bytes", "v5ela_status_string", "v5ela_create", "v5ela_destroy",
    "v5ela_last_error", "v5ela_set_quality", "v5ela_get_quality", "v5ela_get_quant_tables", "v5ela_analyze", "v5ela_analyze_ex",
    "v5ela_enhance", "v5ela_reduce_records", "v5ela_analyze_host", "v5ela_launch_count", "v5ela_profile_enable",
    "v5ela_profile_read", "v5ela_spectrum", "v5ela_spectrum_host", "v5ela_jpeg_bound", "v5ela_jpeg_encode",
    "v5ela_jpeg_encode_host", "v5ela_jpeg_info", "v5ela_jpeg_info_batch", "v5ela_jpeg_decode", "v5ela_jpeg_decode_host",
    "v5ela_last_instantiation", "v5ela_set_block_stage", "v5ela_get_block_stage", "v5ela_analyze_ragged", "v5ela_analyze_ragged_host",
    "v5ela_spectrum_ragged", "v5ela_spectrum_ragged_host", "v5ela_analyze_sweep", "v5ela_analyze_sweep_host",
)
BLOCK_STAGES = {"smem": 0, "mma": 1}
INSTANTIATIONS = {0: "general", 1: "fast", 2: "texhist", -1: None}


class FrameDesc(ctypes.Structure):
    """v5ela_frame_desc (include/v5ela.h): one frame of a ragged batch."""
    _fields_ = [("rgb", ctypes.c_void_p), ("height", ctypes.c_int32), ("width", ctypes.c_int32), ("row_stride_bytes", ctypes.c_int64),
                ("residual", ctypes.c_void_p), ("enhanced", ctypes.c_void_p)]


class GrayDesc(ctypes.Structure):
    """v5ela_gray_desc (include/v5ela.h): one image of a ragged spectrum batch."""
    _fields_ = [("gray", ctypes.c_void_p), ("height", ctypes.c_int32), ("width", ctypes.c_int32), ("row_stride_bytes", ctypes.c_int64),
                ("out", ctypes.c_void_p)]


class V5ElaError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"v5ela error {status}: {message}")
        self.status = status


_lib = None


def load() -> ctypes.CDLL:
    """Load libv5ela.so, building it in-tree with nvcc when it is absent. Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build

        _build.build_library()
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # loud: there is no other implementation to fall back to
        raise ImportError(f"cannot load {LIB_PATH}: {e}. Build it with `python __graft_entry__.py` "
                          f"(nvcc -gencode arch=compute_100a,code=sm_100a).") from e
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    lib.v5ela_abi_version.restype = i32
    lib.v5ela_record_bytes.restype = ctypes.c_size_t
    lib.v5ela_status_string.restype = ctypes.c_char_p
    lib.v5ela_status_string.argtypes = [i32]
    lib.v5ela_create.argtypes = [i32, ctypes.POINTER(vp)]
    lib.v5ela_destroy.argtypes = [vp]
    lib.v5ela_last_error.restype = ctypes.c_char_p
    lib.v5ela_last_error.argtypes = [vp]
    lib.v5ela_set_quality.argtypes = [vp, i32]
    lib.v5ela_get_quality.argtypes = [vp]
    lib.v5ela_get_quant_tables.argtypes = [vp, ctypes.POINTER(ctypes.c_uint16), ctypes.POINTER(ctypes.c_uint16)]
    lib.v5ela_analyze.argtypes = [vp, vp, i32, i32, i32, i64, i64, vp, vp, vp]
    lib.v5ela_analyze_ex.argtypes = [vp, vp, i32, i32, i32, i64, i64, vp, vp, vp, vp]
    lib.v5ela_analyze_ragged.argtypes = [vp, ctypes.POINTER(FrameDesc), i32, vp, vp]
    lib.v5ela_analyze_ragged_host.argtypes = [vp, ctypes.POINTER(FrameDesc), i32, vp]
    lib.v5ela_analyze_sweep.argtypes = [vp, ctypes.POINTER(FrameDesc), i32, ctypes.POINTER(i32), i32, vp, vp, vp]
    lib.v5ela_analyze_sweep_host.argtypes = [vp, ctypes.POINTER(FrameDesc), i32, ctypes.POINTER(i32), i32, vp, vp]
    lib.v5ela_enhance.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    lib.v5ela_reduce_records.argtypes = [vp, vp, i32, i32, vp, vp]
    lib.v5ela_analyze_host.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp]
    lib.v5ela_spectrum.argtypes = [vp, vp, i32, i32, i32, i64, i64, vp, vp]
    lib.v5ela_spectrum_host.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.v5ela_spectrum_ragged.argtypes = [vp, ctypes.POINTER(GrayDesc), i32, vp]
    lib.v5ela_spectrum_ragged_host.argtypes = [vp, ctypes.POINTER(GrayDesc), i32]
    lib.v5ela_jpeg_bound.restype = i64
    lib.v5ela_jpeg_bound.argtypes = [i32, i32, i32]
    lib.v5ela_jpeg_encode.argtypes = [vp, vp, i32, i32, i32, i32, i64, i64, i32, vp, i64, vp, vp]
    lib.v5ela_jpeg_encode_host.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp, i64, vp]
    lib.v5ela_jpeg_info.argtypes = [vp, i64, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32)]
    lib.v5ela_jpeg_info_batch.argtypes = [vp, vp, i32, vp, ctypes.POINTER(i32)]
    lib.v5ela_jpeg_decode.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.v5ela_jpeg_decode_host.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    lib.v5ela_profile_enable.argtypes = [vp, i32]
    lib.v5ela_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(i64), i32]
    lib.v5ela_last_instantiation.argtypes = [vp]
    lib.v5ela_set_block_stage.argtypes = [vp, i32]
    lib.v5ela_get_block_stage.argtypes = [vp]
    lib.v5ela_launch_count.restype = i64
    lib.v5ela_launch_count.argtypes = [vp]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int and name not in ("v5ela_abi_version", "v5ela_jpeg_bound"):
            fn.restype = i32
    if lib.v5ela_abi_version() != 1:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.v5ela_abi_version()} != 1")
    _lib = lib
    return lib


class Handle:
    """Owns one v5ela_handle (one CUDA device, one thread)."""

    def __init__(self, device: int = 0, quality: int = 90):
        self._lib = load()
        self._h = ctypes.c_void_p()
        rc = self._lib.v5ela_create(int(device), ctypes.byref(self._h))
        if rc != 0:
            raise V5ElaError(rc, self._lib.v5ela_status_string(rc).decode())
        self.device = int(device)
        self._quality = 90
        if quality != 90:
            self.set_quality(quality)

    def _check(self, rc: int):
        if rc != 0:
            msg = self._lib.v5ela_last_error(self._h).decode() or self._lib.v5ela_status_string(rc).decode()
            raise V5ElaError(rc, msg)

    @property
    def quality(self) -> int:
        return self._quality

    def set_quality(self, quality: int):
        self._check(self._lib.v5ela_set_quality(self._h, int(quality)))
        self._quality = int(quality)

    def quant_tables(self):
        import numpy as np

        lu, ch = np.zeros(64, np.uint16), np.zeros(64, np.uint16)
        u16p = ctypes.POINTER(ctypes.c_uint16)
        self._check(self._lib.v5ela_get_quant_tables(self._h, lu.ctypes.data_as(u16p), ch.ctypes.data_as(u16p)))
        return lu.reshape(8, 8), ch.reshape(8, 8)

    def analyze(self, d_rgb: int, n: int, h: int, w: int, frame_stride: int, row_stride: int, d_records: int,
                d_residual: int | None, stream: int | None, d_tex_hist: int | None = None):
        if d_tex_hist:
            self._check(self._lib.v5ela_analyze_ex(self._h, d_rgb, n, h, w, frame_stride, row_stride, d_records,
                                                   d_residual or None, d_tex_hist, stream or None))
        else:
            self._check(self._lib.v5ela_analyze(self._h, d_rgb, n, h, w, frame_stride, row_stride, d_records,
                                                d_residual or None, stream or None))

    def analyze_ragged(self, descs, n: int, d_records: int, stream: int | None):
        """descs: ctypes array of FrameDesc holding DEVICE pointers; one launch for frames of different sizes."""
        self._check(self._lib.v5ela_analyze_ragged(self._h, descs, n, d_records, stream or None))

    def analyze_ragged_host(self, descs, n: int, records_host: int):
        """descs: ctypes array of FrameDesc holding HOST pointers; synchronous."""
        self._check(self._lib.v5ela_analyze_ragged_host(self._h, descs, n, records_host))

    def analyze_sweep(self, descs, n: int, qualities, d_records: int, d_ghost: int | None, stream: int | None):
        """descs: ctypes array of FrameDesc holding DEVICE pointers, analysed at every quality of `qualities` in one launch sequence
        (records quality-major); the handle's quality is left as it is."""
        qs = (ctypes.c_int * len(qualities))(*[int(q) for q in qualities])
        self._check(self._lib.v5ela_analyze_sweep(self._h, descs, n, qs, len(qualities), d_records, d_ghost or None, stream or None))

    def analyze_sweep_host(self, descs, n: int, qualities, records_host: int, ghost_host: int | None):
        """descs: ctypes array of FrameDesc holding HOST pointers; synchronous."""
        qs = (ctypes.c_int * len(qualities))(*[int(q) for q in qualities])
        self._check(self._lib.v5ela_analyze_sweep_host(self._h, descs, n, qs, len(qualities), records_host, ghost_host or None))

    def enhance(self, d_residual: int, d_records: int, n: int, h: int, w: int, d_enhanced: int, stream: int | None):
        self._check(self._lib.v5ela_enhance(self._h, d_residual, d_records, n, h, w, d_enhanced, stream or None))

    def reduce_records(self, d_records: int, n: int, group: int, d_out: int, stream: int | None):
        self._check(self._lib.v5ela_reduce_records(self._h, d_records, n, group, d_out, stream or None))

    def analyze_host(self, rgb_host: int, n: int, h: int, w: int, records_host: int, residual_host: int | None = None,
                     enhanced_host: int | None = None, stream: int | None = None):
        """Host-buffer entry point; synchronous when `stream` is None, else asynchronous on that stream."""
        self._check(self._lib.v5ela_analyze_host(self._h, rgb_host, n, h, w, records_host, residual_host or None,
                                                 enhanced_host or None, stream or None))

    def spectrum(self, d_gray: int, n: int, h: int, w: int, frame_stride: int, row_stride: int, d_out: int,
                 stream: int | None):
        self._check(self._lib.v5ela_spectrum(self._h, d_gray, n, h, w, frame_stride, row_stride, d_out, stream or None))

    def spectrum_host(self, gray_host: int, n: int, h: int, w: int, out_host: int):
        self._check(self._lib.v5ela_spectrum_host(self._h, gray_host, n, h, w, out_host))

    def spectrum_ragged(self, descs, n: int, stream: int | None):
        """descs: ctypes array of GrayDesc holding DEVICE pointers; one launch sequence for images of different sizes."""
        self._check(self._lib.v5ela_spectrum_ragged(self._h, descs, n, stream or None))

    def spectrum_ragged_host(self, descs, n: int):
        """descs: ctypes array of GrayDesc holding HOST pointers; synchronous."""
        self._check(self._lib.v5ela_spectrum_ragged_host(self._h, descs, n))

    def jpeg_encode(self, d_img: int, n: int, h: int, w: int, channels: int, frame_stride: int, row_stride: int, quality: int,
                    d_out: int, out_stride: int, d_sizes: int, stream: int | None):
        self._check(self._lib.v5ela_jpeg_encode(self._h, d_img, n, h, w, channels, frame_stride, row_stride, quality, d_out,
                                                out_stride, d_sizes, stream or None))

    def jpeg_encode_host(self, img_host: int, n: int, h: int, w: int, channels: int, quality: int, out_host: int,
                         out_stride: int, sizes_host: int):
        self._check(self._lib.v5ela_jpeg_encode_host(self._h, img_host, n, h, w, channels, quality, out_host, out_stride,
                                                     sizes_host))

    def jpeg_decode(self, files, lens, n: int, d_rgb: int | None, rgb_offsets, d_gray: int | None, gray_offsets,
                    d_status: int | None, stream: int | None):
        self._check(self._lib.v5ela_jpeg_decode(self._h, files, lens, n, d_rgb or None, rgb_offsets, d_gray or None, gray_offsets,
                                                d_status or None, stream or None))

    def jpeg_decode_host(self, files, lens, n: int, rgb_host: int | None, rgb_offsets, gray_host: int | None, gray_offsets):
        self._check(self._lib.v5ela_jpeg_decode_host(self._h, files, lens, n, rgb_host or None, rgb_offsets, gray_host or None,
                                                     gray_offsets))

    def profile_enable(self, enable: bool = True):
        self._check(self._lib.v5ela_profile_enable(self._h, 1 if enable else 0))

    def profile_read(self, reset: bool = True):
        """-> (summed fused-kernel milliseconds, launches) since the last reset (waits for the recorded events)."""
        ms, cnt = ctypes.c_double(0.0), ctypes.c_int64(0)
        self._check(self._lib.v5ela_profile_read(self._h, ctypes.byref(ms), ctypes.byref(cnt), 1 if reset else 0))
        return ms.value, cnt.value

    @property
    def last_instantiation(self):
        """'general' | 'fast' | 'texhist' — the fused-kernel instantiation the last analyze call launched (None before any)."""
        return INSTANTIATIONS[int(self._lib.v5ela_last_instantiation(self._h))]

    @property
    def block_stage(self) -> str:
        """'smem' | 'mma' — which build of the fused kernel's 8x8 block stage this handle launches (include/v5ela.h)."""
        v = int(self._lib.v5ela_get_block_stage(self._h))
        return {n: k for k, n in BLOCK_STAGES.items()}[v]

    @block_stage.setter
    def block_stage(self, name: str):
        self._check(self._lib.v5ela_set_block_stage(self._h, BLOCK_STAGES[name]))

    @property
    def launch_count(self) -> int:
        return int(self._lib.v5ela_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.v5ela_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_tls = threading.local()


def get_handle(device_index: int) -> Handle:
    """One library handle per (thread, device), shared by every entry point of the package; handles are not thread-safe
    (include/v5ela.h)."""
    cache = getattr(_tls, "handles", None)
    if cache is None:
        cache = _tls.handles = {}
    h = cache.get(device_index)
    if h is None:
        h = cache[device_index] = Handle(device_index)
    return h
