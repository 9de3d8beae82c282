"""The V5F v1 per-frame record (include/v5ela.h `v5ela_record`) on the host, and the float features derived from it."""
from __future__ import annotations

import math

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


# ------------------------------------------------------------------------------------------------ DCT statistics
# NumPy restatement of the double-compression estimator of v5ela_jpeg_dct_stats (include/v5ela.h, csrc/v5jpeg_dct.cuh,
# DESIGN.md §4.8). The period decision is computed with the same double operations in the same order as the kernel, so that
# p_k comes out identical; the map agrees to rounding.
DQ_TAU, DQ_RHO, DQ_MIN_COUNT, DQ_PMAX, DQ_FREQS = 0.5, 0.05, 64, 12, 15
# cos / sin (2 pi j / p), p = 2..12, j = 0..p-1, p-major: the literals of csrc/v5jpeg_dct.cuh
DQ_COS = (
    1.0, -1.0,
    1.0, -0.5, -0.5,
    1.0, 0.0, -1.0, 0.0,
    1.0, 0.30901699437494745, -0.8090169943749475, -0.8090169943749475, 0.30901699437494745,
    1.0, 0.5, -0.5, -1.0, -0.5, 0.5,
    1.0, 0.6234898018587335, -0.2225209339563144, -0.9009688679024191, -0.9009688679024191, -0.2225209339563144, 0.6234898018587335,
    1.0, 0.7071067811865476, 0.0, -0.7071067811865476, -1.0, -0.7071067811865476, 0.0, 0.7071067811865476,
    1.0, 0.766044443118978, 0.17364817766693036, -0.5, -0.9396926207859084, -0.9396926207859084, -0.5, 0.17364817766693036, 0.766044443118978,
    1.0, 0.8090169943749475, 0.30901699437494745, -0.30901699437494745, -0.8090169943749475, -1.0, -0.8090169943749475, -0.30901699437494745,
    0.30901699437494745, 0.8090169943749475,
    1.0, 0.8412535328311812, 0.41541501300188644, -0.14231483827328514, -0.6548607339452851, -0.9594929736144974, -0.9594929736144974,
    -0.6548607339452851, -0.14231483827328514, 0.41541501300188644, 0.8412535328311812,
    1.0, 0.8660254037844386, 0.5, 0.0, -0.5, -0.8660254037844386, -1.0, -0.8660254037844386, -0.5, 0.0, 0.5, 0.8660254037844386,
)
DQ_SIN = (
    0.0, 0.0,
    0.0, 0.8660254037844386, -0.8660254037844386,
    0.0, 1.0, 0.0, -1.0,
    0.0, 0.9510565162951535, 0.5877852522924731, -0.5877852522924731, -0.9510565162951535,
    0.0, 0.8660254037844386, 0.8660254037844386, 0.0, -0.8660254037844386, -0.8660254037844386,
    0.0, 0.7818314824680298, 0.9749279121818236, 0.4338837391175581, -0.4338837391175581, -0.9749279121818236, -0.7818314824680298,
    0.0, 0.7071067811865476, 1.0, 0.7071067811865476, 0.0, -0.7071067811865476, -1.0, -0.7071067811865476,
    0.0, 0.6427876096865394, 0.984807753012208, 0.8660254037844386, 0.3420201433256687, -0.3420201433256687, -0.8660254037844386,
    -0.984807753012208, -0.6427876096865394,
    0.0, 0.5877852522924731, 0.9510565162951535, 0.9510565162951535, 0.5877852522924731, 0.0, -0.5877852522924731, -0.9510565162951535,
    -0.9510565162951535, -0.5877852522924731,
    0.0, 0.5406408174555976, 0.9096319953545183, 0.9898214418809327, 0.7557495743542583, 0.28173255684142967, -0.28173255684142967,
    -0.7557495743542583, -0.9898214418809327, -0.9096319953545183, -0.5406408174555976,
    0.0, 0.5, 0.8660254037844386, 1.0, 0.8660254037844386, 0.5, 0.0, -0.5, -0.8660254037844386, -1.0, -0.8660254037844386, -0.5,
)
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                   35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55,
                   62, 63])                              # natural-order position of zigzag position z


def _dq_period(h) -> int:
    """p_k of one frequency's 129-bin histogram h (value v at h[v + 64])."""
    g = [0] + [int(h[64 + v]) + int(h[64 - v]) for v in range(1, 64)]
    n = sum(g)
    if n < DQ_MIN_COUNT:
        return 1
    r2 = {v: 2 * g[v] - g[v - 1] - g[v + 1] for v in range(2, 63)}           # twice the residual r(v)
    abs2r = sum(abs(x) for x in r2.values())
    best, s_best = 0, -1.0
    for p in range(2, DQ_PMAX + 1):
        base = p * (p - 1) // 2 - 1
        re = im = 0.0
        for j in range(p):
            rj = float(sum(x for v, x in r2.items() if v % p == j))
            re = re + rj * DQ_COS[base + j]
            im = im + rj * DQ_SIN[base + j]
        s = math.sqrt(re * re + im * im) / float(max(abs2r, 2))
        if s > s_best:                                                           # the smaller p wins ties
            best, s_best = p, s
    return best if s_best >= DQ_TAU and 0.5 * abs2r >= DQ_RHO * n else 1


def _dq_lut(h, p: int) -> np.ndarray:
    """log P_u of the 129 bins for period p, then log P_t = -log p."""
    out = np.empty(130)
    for b in range(129):
        v = min(max(b - 64, -63), 63)                                            # the end bins take the entries of +-63
        s = p * (v // p)
        mass = sum(int(h[64 + u]) for u in range(s, s + p) if -63 <= u <= 63)
        out[b] = -math.log(p) if mass == 0 else (math.log(int(h[64 + v]) / mass) if h[64 + v] else -math.inf)
    out[129] = -math.log(p)
    return out


def _luma(hist):
    hist = np.asarray(hist)
    return hist[..., 0, :, :] if hist.ndim >= 3 and hist.shape[-3] == 3 else hist


def dq_periods(hist) -> np.ndarray:
    """Periods p_k of the 15 luma AC frequencies at zigzag positions 1..15 (1: no period found), int32 (..., 15), from
    histograms shaped like v5ela_jpeg_dct_stats' (..., 3, 64, 129), or the luma part alone (..., 64, 129)."""
    luma = _luma(hist)
    flat = luma.reshape(-1, 64, 129)
    out = np.array([[_dq_period(f[ZIGZAG[z]]) for z in range(1, DQ_FREQS + 1)] for f in flat], np.int32)
    return out.reshape(luma.shape[:-2] + (DQ_FREQS,))


def dq_map(hist, coef) -> np.ndarray:
    """The double-compression map of one file: hist (3, 64, 129) or (64, 129) as v5ela_jpeg_dct_stats returns it, coef
    (ceil(H/8), ceil(W/8), 64) the quantised coefficients of the file's luma blocks in zigzag order (the file's order). float32, per
    block the posterior that it was not aligned-double-compressed; 0.5 everywhere when no frequency has a period."""
    luma = _luma(hist)
    coef = np.asarray(coef)
    idx = np.clip(coef[..., 1:DQ_FREQS + 1].astype(np.int64), -64, 64) + 64
    s = np.zeros(coef.shape[:-1])
    found = False
    for f in range(DQ_FREQS):
        h = luma[ZIGZAG[f + 1]]
        p = _dq_period(h)
        if p > 1:
            t = _dq_lut(h, p)
            s = s + (t[idx[..., f]] - t[129])
            found = True
    if not found:
        return np.full(coef.shape[:-1], 0.5, np.float32)
    with np.errstate(over="ignore"):
        return (1.0 / (1.0 + np.exp(s))).astype(np.float32)


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
