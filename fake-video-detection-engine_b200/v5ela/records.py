"""The V5F v1 per-frame record (include/v5ela.h `v5ela_record`) on the host, and the float features derived from it."""
from __future__ import annotations

import numpy as np

RECORD_DTYPE = np.dtype(
    [
        ("ela_hist", "<u4", (3, 256)),
        ("ela_sum", "<u8", (3,)),
        ("ela_sumsq", "<u8", (3,)),
        ("tex_sumabs", "<u8"),
        ("tex_sumsq", "<u8"),
        ("tex_maxabs", "<u2"),
        ("ela_max", "u1", (3,)),
        ("pad", "u1", (3,)),
    ]
)
RECORD_BYTES = RECORD_DTYPE.itemsize
assert RECORD_BYTES == 3144


def as_records(raw) -> np.ndarray:
    """uint8 array/tensor of shape (N, 3144) (host) -> structured array of N records (a view, no copy)."""
    if hasattr(raw, "detach"):
        raw = raw.detach().cpu().numpy()
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    return raw.reshape(-1, RECORD_BYTES).view(RECORD_DTYPE).reshape(-1)


def combine(records: np.ndarray) -> np.ndarray:
    """Host mirror of v5ela_reduce_records: one record aggregating `records` (sums add, maxima max)."""
    out = np.zeros((), dtype=RECORD_DTYPE)
    out["ela_hist"] = np.minimum(records["ela_hist"].sum(axis=0, dtype=np.uint64), 0xFFFFFFFF).astype(np.uint32)   # saturating, like the kernel
    for k in ("ela_sum", "ela_sumsq", "tex_sumabs", "tex_sumsq"):
        out[k] = records[k].sum(axis=0, dtype=np.uint64)
    out["tex_maxabs"] = records["tex_maxabs"].max()
    out["ela_max"] = records["ela_max"].max(axis=0)
    return out


def ghost_curve(records, pixels) -> np.ndarray:
    """The JPEG-ghost curve of sweep records (v5ela.analyze_sweep): the mean squared residual sum_c ela_sumsq / (3 * pixels) as
    float64, one value per record. ``records`` is a structured array of any shape, e.g. (nq, N); ``pixels`` is H*W, or an array that
    broadcasts against it, e.g. the (N,) pixel counts of the frames. Its minimum over the qualities estimates a frame's earlier
    JPEG quality."""
    return records["ela_sumsq"].sum(axis=-1, dtype=np.uint64).astype(np.float64) / (3.0 * np.asarray(pixels, dtype=np.float64))


def features(rec, n_pixels: int) -> dict:
    """Float64 features of one record over `n_pixels` pixels (H*W of the frame, or the sum over a video's frames).

    ``ela_max`` / ``ela_scale`` are the reference's ``max_diff`` (with its 0 -> 1 fix) and ``scale``
    (v5_texture_ela.py:72-76); everything else is the build-defined statistics of SURVEY.md §8a.
    """
    n = float(n_pixels)
    s = rec["ela_sum"].astype(np.float64)
    sq = rec["ela_sumsq"].astype(np.float64)
    mean = s / n
    max_diff = int(rec["ela_max"].max())
    tex_mean_abs = float(rec["tex_sumabs"]) / n
    return {
        "ela_max_rgb": [int(v) for v in rec["ela_max"]],
        "ela_max": max_diff,
        "ela_scale": 255.0 / (max_diff if max_diff else 1),
        "ela_mean_rgb": [float(v) for v in mean],
        "ela_var_rgb": [float(v) for v in (sq / n - mean * mean)],
        "ela_mean": float(s.sum() / (3.0 * n)),
        "ela_nonzero_frac_rgb": [float(1.0 - rec["ela_hist"][c][0] / n) for c in range(3)],
        "tex_mean_abs": tex_mean_abs,
        "tex_mean_sq": float(rec["tex_sumsq"]) / n,
        "tex_max_abs": int(rec["tex_maxabs"]),
    }
