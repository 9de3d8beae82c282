"""CPU: the band references of tests/periodic_ref.py (records, texture histograms, residual and JPEG-ghost maps of tiled frames,
from small frames) against the C oracle and Pillow / OpenCV run on the whole frame. tests/test_gpu_limits.py checks frames of up to
2^31 - 65536 pixels against these references, so they must be exact for every remainder (h % 16, w % 16), quality and tile."""
import numpy as np
import pytest

from oracle import c_oracle, pil_oracle
from periodic_ref import (band_index, expected_ghost, expected_record, expected_residual_bands, expected_tex_hist, ghost_of, tile_of,
                          tiled)


def check(tile, h, w, q, tex_hist=False):
    full = tiled(tile, h, w)
    o = c_oracle.analyze_frame(full, q)
    want = expected_record(tile, h, w, q)
    assert want.tobytes() == o["record"].tobytes(), (h, w, q)
    _, slab = expected_residual_bands(tile, h, w, q)
    assert np.array_equal(slab(0, h), o["residual"]), (h, w, q)
    _, gslab = expected_ghost(tile, h, w, q)
    assert np.array_equal(gslab(0, -(-h // 16)), ghost_of(o["residual"])), (h, w, q)
    if tex_hist:
        assert np.array_equal(expected_tex_hist(tile, h, w), pil_oracle.texture_hist(full)), (h, w)


def test_band_index():
    assert band_index(48).tolist() == list(range(48))
    idx = band_index(16 * 5 + 3)                                   # a = 3
    assert idx[:16].tolist() == list(range(16))
    assert idx[16:64].tolist() == list(range(16, 32)) * 3
    assert idx[64:].tolist() == list(range(32, 51))
    assert band_index(16 * 5 + 3, 16).tolist() == [0, 1, 1, 1, 2, 3]
    assert band_index(16 * 6, 16).tolist() == [0, 1, 1, 1, 1, 2]


@pytest.mark.parametrize("r", range(16))
def test_every_remainder_pair(r):
    """All 256 (h % 16, w % 16) pairs at q = 90, with a, b = 3, 2 middle bands (the bilinear terms all count)."""
    tile = tile_of("noise", seed=r)
    for s in range(16):
        check(tile, 16 * 5 + r, 16 * 4 + s, 90)


@pytest.mark.parametrize("q", [1, 30, 90, 100])
@pytest.mark.parametrize("kind", ["noise", "smooth", "flat", "saturated"])
def test_qualities_and_tiles(q, kind):
    tile = tile_of(kind, seed=q)
    for h, w in [(16 * 7 + 5, 16 * 4 + 11), (16 * 4, 16 * 6 + 1), (16 * 3 + 15, 16 * 8), (16 * 6 + 8, 16 * 3 + 14)]:
        check(tile, h, w, q, tex_hist=(q == 90))
