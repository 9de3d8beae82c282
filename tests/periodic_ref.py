"""Exact references for giant periodic frames, from the C oracle run on small ones (test infrastructure).

Every output of the fused kernel is local: a residual pixel depends only on its 16 x 16 MCU (its 8 x 8 luma block and the chroma
samples of the MCU), and a Laplacian value only on its 3 x 3 luma neighbourhood. A frame that repeats a 16 x 16 x 3 tile T, cropped
to H = 16 (a + 2) + r rows by W = 16 (b + 2) + s columns (a, b >= 1, 0 <= r, s < 16), therefore consists of an edge band of 16 rows,
a middle bands that are all alike, and a last band of 16 + r rows (the same across). So:

- every additive record field (histograms and sums) is bilinear in (a, b), and four oracle runs on the tiled
  (32 + r + 16 i) x (32 + s + 16 j) frames, i, j in {1, 2}, give it for any (a, b); the maxima are the maxima over those four;
- the residual map is the (48 + r) x (48 + s) frame's map with its middle band (rows / columns 16..31) repeated a (b) times;
- the JPEG-ghost maps (per-MCU sums of squared residuals) follow the same rule one MCU at a time.

tests/test_periodic_reference.py checks all of this against the oracle on whole frames; tests/test_gpu_limits.py uses it for
frames of up to 2^31 - 65536 pixels, which the oracle cannot run in reasonable time.
"""
from __future__ import annotations

import numpy as np

from oracle import c_oracle, pil_oracle
from oracle.pil_oracle import RECORD_DTYPE

ADDITIVE = ("ela_hist", "ela_sum", "ela_sumsq", "tex_sumabs", "tex_sumsq")


def tiled(tile: np.ndarray, h: int, w: int) -> np.ndarray:
    """The (h, w, 3) frame that repeats `tile` (16 x 16 x 3) from its top-left corner."""
    th, tw = tile.shape[:2]
    return np.ascontiguousarray(np.tile(tile, (h // th + 1, w // tw + 1, 1))[:h, :w])


def _bands(h: int, w: int):
    if h < 48 or w < 48:
        raise ValueError("the band references need h, w >= 48")
    return h // 16 - 2, w // 16 - 2, h % 16, w % 16


def _bilinear(x, a: int, b: int):
    """x[i, j]: the value at (a, b) = (i, j), i, j in {1, 2} (Python ints or object arrays) -> the value at (a, b)."""
    return x[1, 1] + (a - 1) * (x[2, 1] - x[1, 1]) + (b - 1) * (x[1, 2] - x[1, 1]) + \
        (a - 1) * (b - 1) * (x[2, 2] - x[2, 1] - x[1, 2] + x[1, 1])


def _corner_frames(tile, h, w):
    _, _, r, s = _bands(h, w)
    return {(i, j): tiled(tile, 32 + r + 16 * i, 32 + s + 16 * j) for i in (1, 2) for j in (1, 2)}


def expected_record(tile: np.ndarray, h: int, w: int, q: int) -> np.ndarray:
    """The oracle's record (0-d RECORD_DTYPE array) of tiled(tile, h, w) at quality q, from four small frames."""
    a, b, _, _ = _bands(h, w)
    recs = {k: c_oracle.analyze_frame(f, q)["record"] for k, f in _corner_frames(tile, h, w).items()}
    out = np.zeros((), RECORD_DTYPE)
    for f in ADDITIVE:
        v = _bilinear({k: np.asarray(r[f]).astype(object) for k, r in recs.items()}, a, b)
        out[f] = np.asarray(v, dtype=np.uint64) if np.ndim(v) else int(v)
    out["ela_max"] = np.maximum.reduce([r["ela_max"] for r in recs.values()])
    out["tex_maxabs"] = max(int(r["tex_maxabs"]) for r in recs.values())
    return out


def expected_tex_hist(tile: np.ndarray, h: int, w: int) -> np.ndarray:
    """pil_oracle.texture_hist (uint32 [256]) of tiled(tile, h, w)."""
    a, b, _, _ = _bands(h, w)
    hists = {k: pil_oracle.texture_hist(f).astype(object) for k, f in _corner_frames(tile, h, w).items()}
    return np.asarray(_bilinear(hists, a, b), dtype=np.uint32)


def band_index(n: int, unit: int = 1) -> np.ndarray:
    """Index k of the (48 + n % 16)-pixel side from which position k' of an n-pixel side is copied, in units of `unit` pixels
    (1: pixels, 16: MCUs): the first band as it is, the middle band repeated, the rest shifted."""
    a = n // 16 - 2
    m = -(-n // unit)
    k = np.arange(m, dtype=np.int64)
    first, mid = 16 // unit, 16 // unit
    return np.where(k < first, k, np.where(k < first + a * mid, first + (k - first) % mid, k - (a - 1) * mid))


def expected_residual_bands(tile: np.ndarray, h: int, w: int, q: int):
    """-> (small residual map of the (48 + r) x (48 + s) frame, slab(y0, y1) -> rows y0..y1 of the (h, w, 3) residual map)."""
    _bands(h, w)
    small = c_oracle.analyze_frame(tiled(tile, 48 + h % 16, 48 + w % 16), q)["residual"]
    rows, cols = band_index(h), band_index(w)

    def slab(y0: int, y1: int) -> np.ndarray:
        return small[rows[y0:y1]][:, cols]

    return small, slab


def ghost_of(residual: np.ndarray) -> np.ndarray:
    """Per 16 x 16 MCU: sum over its pixels and channels of residual^2 (int64 [ceil(h/16), ceil(w/16)])."""
    h, w, _ = residual.shape
    mh, mw = -(-h // 16), -(-w // 16)
    sq = np.zeros((16 * mh, 16 * mw), np.int64)
    sq[:h, :w] = (residual.astype(np.int64) ** 2).sum(axis=2)
    return sq.reshape(mh, 16, mw, 16).sum(axis=(1, 3))


def expected_ghost(tile: np.ndarray, h: int, w: int, q: int):
    """-> (small ghost map of the (48 + r) x (48 + s) frame, slab(m0, m1) -> MCU rows m0..m1 of the frame's ghost map)."""
    small_res, _ = expected_residual_bands(tile, h, w, q)
    small = ghost_of(small_res)
    rows, cols = band_index(h, 16), band_index(w, 16)

    def slab(m0: int, m1: int) -> np.ndarray:
        return small[rows[m0:m1]][:, cols]

    return small, slab


def tile_of(kind: str, seed: int = 0) -> np.ndarray:
    """16 x 16 x 3 test tiles: 'noise' (uniform), 'smooth' (ramps), 'flat' (one colour) and 'saturated' (0 / 255 stripes)."""
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (16, 16, 3), dtype=np.uint8)
    if kind == "smooth":
        return (np.add.outer(np.arange(16), np.arange(16))[..., None] * np.array([7, 3, 11]) % 256).astype(np.uint8)
    if kind == "flat":
        return np.full((16, 16, 3), [200, 30, 90], np.uint8)
    if kind == "saturated":
        t = np.zeros((16, 16, 3), np.uint8)
        t[..., 0] = 255 * ((np.arange(16)[None, :] // 3) & 1)
        t[..., 2] = 255 * ((np.arange(16)[:, None] // 5) & 1)
        return t
    raise ValueError(kind)
