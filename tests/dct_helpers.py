"""Shared by the DCT-statistics tests (test infrastructure; may import oracle/): test files of every layout the decoder supports,
and NumPy histograms / luma block grids of the oracle decoder's coefficients, written from the definition in include/v5ela.h."""
import io

import numpy as np
from PIL import Image

from helpers import golden_frame, layout_golden_files, load_json
from oracle import c_oracle

JPEG = load_json("jpeg_golden.json")


def pil_bytes(img, quality, **kw):
    buf = io.BytesIO()
    Image.fromarray(img).save(buf, "JPEG", quality=quality, **kw)
    return buf.getvalue()


def layout_files(max_pixels=300 * 500):
    """[(label, bytes)]: the default 4:2:0 files of jpeg_golden.json's cases, their gray and optimised-Huffman versions, and every
    file of layouts_golden.json (4:4:4, 4:2:2, 4:2:0 with restart intervals, gray with restarts)."""
    out = []
    for c in JPEG["cases"]:
        if c["h"] * c["w"] > max_pixels:
            continue
        rgb = golden_frame(c)
        tag = f"{c['spec'][0]}{c['spec'][1]}_{c['h']}x{c['w']}_q{c['q']}"
        out.append((f"420_{tag}", pil_bytes(rgb, c["q"])))
        out.append((f"gray_{tag}", pil_bytes(np.ascontiguousarray(rgb[..., 1]), c["q"])))
        out.append((f"opt_{tag}", pil_bytes(rgb, c["q"], optimize=True)))
    for case, label, data, _ in layout_golden_files():
        if case["h"] * case["w"] <= max_pixels:
            out.append((f"{label}_{case['h']}x{case['w']}_q{case['q']}", data))
    return out


def odd_size_files(rng, count, max_side=90):
    """[(label, bytes)]: random sizes from 1x1 up, random qualities and layouts (PIL subsampling 0 / 1 / 2, gray)."""
    out = []
    for i in range(count):
        h, w = int(rng.integers(1, max_side)), int(rng.integers(1, max_side))
        q = int(rng.integers(5, 101))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        img = (img.astype(np.int32) // 2 + 64).astype(np.uint8)
        kind = i % 4
        if kind == 3:
            out.append((f"gray_{h}x{w}_q{q}", pil_bytes(np.ascontiguousarray(img[..., 0]), q)))
        else:
            out.append((f"ss{kind}_{h}x{w}_q{q}", pil_bytes(img, q, subsampling=kind)))
    return out


def oracle_blocks(data):
    """-> (coef [blocks, 64] zigzag, DC values at 0, scan order), h, w, ncomp, hs, vs from the oracle decoder."""
    h, w, c = c_oracle.jpeg_info(data)
    hs, vs, _ = c_oracle.jpeg_layout(data)
    if c == 1:
        hs = vs = 1
    coef = c_oracle.jpeg_decode(data, want_coef=True)["coef"]
    return coef, h, w, c, hs, vs


def block_positions(h, w, ncomp, hs, vs):
    """Per scan-order block: (component, bx, by), and whether it covers samples of its component."""
    mcux = (w + 8 * hs - 1) // (8 * hs)
    mcuy = (h + 8 * vs - 1) // (8 * vs)
    pos = []
    for my in range(mcuy):
        for mx in range(mcux):
            if ncomp == 1:
                pos.append((0, mx, my))
                continue
            for r in range(vs):
                for s in range(hs):
                    pos.append((0, hs * mx + s, vs * my + r))
            pos.append((1, mx, my))
            pos.append((2, mx, my))
    real = []
    for comp, bx, by in pos:
        cw = w if comp == 0 else -(-w // hs)
        ch = h if comp == 0 else -(-h // vs)
        real.append(bx < -(-cw // 8) and by < -(-ch // 8))
    return pos, real


def np_hist(data):
    """The histogram of include/v5ela.h, (3, 64, 129) uint32, over the oracle's coefficients."""
    coef, h, w, c, hs, vs = oracle_blocks(data)
    pos, real = block_positions(h, w, c, hs, vs)
    assert len(pos) == coef.shape[0]
    from v5ela.records import ZIGZAG

    nat = np.zeros_like(coef)
    nat[:, ZIGZAG] = coef
    hist = np.zeros((3, 64, 129), np.uint32)
    comps = np.array([p[0] for p in pos])
    real = np.array(real)
    for comp in range(c):
        sel = nat[(comps == comp) & real].astype(np.int64)
        vals = np.clip(sel, -64, 64) + 64
        for k in range(64):
            hist[comp, k] = np.bincount(vals[:, k], minlength=129)
    return hist


def luma_grid(data):
    """The luma blocks' coefficients on their block grid: (ceil(H/8), ceil(W/8), 64), zigzag order."""
    coef, h, w, c, hs, vs = oracle_blocks(data)
    pos, real = block_positions(h, w, c, hs, vs)
    bh, bw = -(-h // 8), -(-w // 8)
    grid = np.zeros((bh, bw, 64), np.int16)
    for g, ((comp, bx, by), ok) in enumerate(zip(pos, real)):
        if comp == 0 and ok:
            grid[by, bx] = coef[g]
    return grid


def qtab_of(data):
    """(3, 64) natural-order DQT tables of the file's components, read from its DQT / SOF segments directly."""
    tables, comp_tq = {}, []
    i = 2
    while i + 4 <= len(data):
        assert data[i] == 0xFF
        m = data[i + 1]
        L = (data[i + 2] << 8) | data[i + 3]
        seg = data[i + 4:i + 2 + L]
        if m == 0xDB:
            k = 0
            while k < len(seg):
                pq, t = seg[k] >> 4, seg[k] & 15
                k += 1
                vals = []
                for _ in range(64):
                    vals.append((seg[k] << 8 | seg[k + 1]) if pq else seg[k])
                    k += 2 if pq else 1
                from v5ela.records import ZIGZAG

                nat = np.zeros(64, np.uint16)
                nat[ZIGZAG] = vals
                tables[t] = nat
        elif m in (0xC0, 0xC1):
            nc = seg[5]
            comp_tq = [seg[8 + 3 * j] & 3 for j in range(nc)]
        elif m == 0xDA:
            break
        i += 2 + L
    out = np.zeros((3, 64), np.uint16)
    for j, t in enumerate(comp_tq):
        out[j] = tables[t]
    return out
