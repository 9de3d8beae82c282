"""Test infrastructure: baseline JPEG files written straight from quantised coefficients, and a NumPy restatement of the inverse
DCT that Pillow and OpenCV run on x86-64 (libjpeg-turbo's SIMD ISLOW path).

A file's coefficients can carry far more than pixels can produce: AC values up to +-1023, DC differences up to +-2047 with the
predictor walking outside int16, 8-bit quantisation entries up to 255 and 16-bit ones (SOF1) up to 65535. An encoder that starts
from pixels never writes such blocks, so the decoder tests build them here."""
from __future__ import annotations

import numpy as np

# zigzag position -> natural (row-major) index, T.81 Figure A.6
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14,
                   21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60,
                   61, 54, 47, 55, 62, 63])

# T.81 Annex K.3 typical tables: (bits[16], vals) for DC luma, DC chroma, AC luma, AC chroma
DC_LUMA = ([0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0], list(range(12)))
DC_CHROMA = ([0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], list(range(12)))
AC_LUMA = ([0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 125], bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738393a"
    "434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5a6a7a8a9"
    "aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa"))
AC_CHROMA = ([0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 119], bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a3536373839"
    "3a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3a4a5a6a7"
    "a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa"))
STANDARD_TABLES = {"dc": (DC_LUMA, DC_CHROMA), "ac": (AC_LUMA, AC_CHROMA)}

# Supplied tables with every symbol a Huffman table may carry beyond baseline's: AC sizes 11..15 at every run, DC sizes up to 15
_WIDE_AC = list(AC_LUMA[1]) + [(r << 4) | s for r in range(16) for s in range(11, 16)]
WIDE_TABLES = {"dc": (([0, 0, 0, 0, 16] + [0] * 11, list(range(16))),) * 2,
               "ac": (([0] * 7 + [len(_WIDE_AC)] + [0] * 8, _WIDE_AC),) * 2}

# layout -> (components, luma hs, luma vs); chroma components are always 1x1
LAYOUTS = {"gray": (1, 1, 1), "420": (3, 2, 2), "422": (3, 2, 1), "444": (3, 1, 1)}


def mcu_grid(h: int, w: int, layout: str):
    """-> (MCUs across, MCUs down, blocks per MCU)."""
    nc, hs, vs = LAYOUTS[layout]
    return (w + 8 * hs - 1) // (8 * hs), (h + 8 * vs - 1) // (8 * vs), (hs * vs + 2 if nc == 3 else 1)


def block_count(h: int, w: int, layout: str) -> int:
    mx, my, bpm = mcu_grid(h, w, layout)
    return mx * my * bpm


def block_components(h: int, w: int, layout: str) -> np.ndarray:
    """Component (0 Y, 1 Cb, 2 Cr) of every block of the scan, in scan order."""
    mx, my, bpm = mcu_grid(h, w, layout)
    per = np.zeros(bpm, np.int64) if bpm == 1 else np.array([0] * (bpm - 2) + [1, 2])
    return np.tile(per, mx * my)


def code_table(spec):
    """(bits, vals) -> {symbol: (code, length)} (T.81 Annex C)."""
    bits, vals = spec
    out, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            out[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return out


class _Bits:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, value: int, length: int):
        self.acc = (self.acc << length) | (value & ((1 << length) - 1))
        self.n += length
        while self.n >= 8:
            self.n -= 8
            byte = (self.acc >> self.n) & 0xFF
            self.out.append(byte)
            if byte == 0xFF:
                self.out.append(0)                # byte stuffing
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)   # pad with one bits


def _magnitude(v: int):
    size = abs(v).bit_length()
    return size, (v if v >= 0 else v + (1 << size) - 1)


def _segment(marker: int, payload: bytes) -> bytes:
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + payload


def write_jpeg(coef, h: int, w: int, layout: str, qt, *, restart: int = 0, tables=None, code_lengths: set | None = None) -> bytes:
    """A complete baseline (or, with a 16-bit table, SOF1) Huffman JPEG file.

    coef  : [blocks, 64] in scan order (what c_oracle.jpeg_decode(..., want_coef=True) returns), zigzag order inside a block;
            column 0 holds the DC value as the decoder's predictor sees it (any int: differences between neighbours of a
            component are what is coded, and a decoder keeps the int16 truncation of the predictor)
    qt    : one table (applied to every component) or [luma, chroma], 64 entries each in natural order; a table with an entry
            above 255 is written with 16-bit precision
    restart: MCUs per restart interval (0 = none)
    tables: {"dc": (luma, chroma), "ac": (luma, chroma)} of (bits, vals); default the Annex K tables
    code_lengths: a set that receives the length of every Huffman code written
    """
    nc, hs, vs = LAYOUTS[layout]
    coef = np.asarray(coef, np.int64)
    assert coef.shape == (block_count(h, w, layout), 64), coef.shape
    qt = np.asarray(qt, np.int64).reshape(-1, 64)
    if nc == 1 or len(qt) == 1:
        qt = qt[:1]
    assert qt.min() >= 1 and qt.max() <= 65535
    tables = tables or STANDARD_TABLES
    ntab = 2 if nc == 3 else 1
    out = bytearray(b"\xff\xd8")
    for t in range(len(qt)):
        wide = int(qt[t].max()) > 255
        zz = qt[t][ZIGZAG]
        out += _segment(0xDB, bytes([(16 if wide else 0) | t]) + b"".join(int(v).to_bytes(2 if wide else 1, "big") for v in zz))
    wide_any = any(int(q.max()) > 255 for q in qt)
    comps = [(1, (hs << 4) | vs, 0)] if nc == 1 else [(1, (hs << 4) | vs, 0), (2, 0x11, min(1, len(qt) - 1)),
                                                      (3, 0x11, min(1, len(qt) - 1))]
    out += _segment(0xC1 if wide_any else 0xC0,
                    bytes([8]) + h.to_bytes(2, "big") + w.to_bytes(2, "big") + bytes([nc]) + b"".join(bytes(c) for c in comps))
    for cls, key in ((0, "dc"), (1, "ac")):
        for t in range(ntab):
            bits, vals = tables[key][t]
            out += _segment(0xC4, bytes([(cls << 4) | t]) + bytes(bits) + bytes(vals))
    if restart:
        out += _segment(0xDD, restart.to_bytes(2, "big"))
    out += _segment(0xDA, bytes([nc]) + b"".join(bytes([i + 1, (0x11 if i else 0) if ntab == 2 else 0]) for i in range(nc)) +
                    bytes([0, 63, 0]))
    dc_codes = [code_table(tables["dc"][t]) for t in range(ntab)]
    ac_codes = [code_table(tables["ac"][t]) for t in range(ntab)]
    mx, my, bpm = mcu_grid(h, w, layout)
    comp_of = block_components(h, w, layout)
    bw = _Bits()
    lengths = set() if code_lengths is None else code_lengths

    def put_code(entry):
        lengths.add(entry[1])
        bw.put(*entry)

    pred = [0, 0, 0]
    for m in range(mx * my):
        if restart and m and m % restart == 0:
            bw.flush()
            bw.out += bytes([0xFF, 0xD0 + (m // restart - 1) % 8])
            pred = [0, 0, 0]
        for b in range(m * bpm, (m + 1) * bpm):
            c = int(comp_of[b])
            t = min(c, ntab - 1)
            blk = coef[b]
            size, bits = _magnitude(int(blk[0]) - pred[c])
            pred[c] = int(blk[0])
            put_code(dc_codes[t][size])
            bw.put(bits, size)
            run = 0
            for k in range(1, 64):
                v = int(blk[k])
                if v == 0:
                    run += 1
                    continue
                while run > 15:
                    put_code(ac_codes[t][0xF0])
                    run -= 16
                size, bits = _magnitude(v)
                put_code(ac_codes[t][(run << 4) | size])
                bw.put(bits, size)
                run = 0
            if run:
                put_code(ac_codes[t][0x00])     # EOB
    bw.flush()
    out += bw.out + b"\xff\xd9"
    return bytes(out)


# ------------------------------------------------------------------------------------------- the x86 SIMD ISLOW inverse DCT
# libjpeg-turbo's SSE2 / AVX2 ISLOW code works on 16-bit lanes: it dequantises with a 16-bit multiply (low half kept), forms
# in0 +- in4 and the two odd-part sums z3 = in3 + in7, z4 = in1 + in5 with 16-bit adds (wrapping), runs every product as a
# 16 x 16 -> 32-bit multiply-add, packs the column-pass outputs to int16 with saturation and the final samples to int8 with
# saturation (+128). A block whose AC rows 1..7 are all zero takes a shortcut in the column pass: the dequantised DC shifted
# left by 2 in 16 bits (wrapping). Within 16-bit inputs no 32-bit sum can overflow. This differs from libjpeg-turbo's C path
# (and from the arithmetic of T.81 A.6 in wide integers) only on blocks no pixel-derived file carries.
C = dict(c0_298=2446, c0_390=3196, c0_541=4433, c0_765=6270, c0_899=7373, c1_175=9633, c1_501=12299, c1_847=15137,
         c1_961=16069, c2_053=16819, c2_562=20995, c3_072=25172)


def _w16(x):
    return ((x + 32768) & 0xFFFF) - 32768


def _pass(v, n: int):
    """One 8-point pass along axis 1 of v [N, 8, 8] (int64), wrapping where the SIMD code wraps -> [N, 8, 8] outputs >> n along
    axis 1, not yet saturated."""
    i = [v[:, k] for k in range(8)]
    t0 = _w16(i[0] + i[4]) << 13
    t1 = _w16(i[0] - i[4]) << 13
    t2 = i[2] * C["c0_541"] + i[6] * (C["c0_541"] - C["c1_847"])
    t3 = i[2] * (C["c0_541"] + C["c0_765"]) + i[6] * C["c0_541"]
    e10, e13, e11, e12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    z3, z4 = _w16(i[7] + i[3]), _w16(i[5] + i[1])
    z3b = z3 * (C["c1_175"] - C["c1_961"]) + z4 * C["c1_175"]
    z4b = z3 * C["c1_175"] + z4 * (C["c1_175"] - C["c0_390"])
    o0 = i[7] * (C["c0_298"] - C["c0_899"]) + i[1] * -C["c0_899"] + z3b
    o3 = i[7] * -C["c0_899"] + i[1] * (C["c1_501"] - C["c0_899"]) + z4b
    o1 = i[5] * (C["c2_053"] - C["c2_562"]) + i[3] * -C["c2_562"] + z4b
    o2 = i[5] * -C["c2_562"] + i[3] * (C["c3_072"] - C["c2_562"]) + z3b
    rnd = 1 << (n - 1)
    out = [e10 + o3, e11 + o2, e12 + o1, e13 + o0, e13 - o0, e12 - o1, e11 - o2, e10 - o3]
    return np.stack([(x + rnd) >> n for x in out], axis=1)


def simd_islow(nat, qt):
    """nat: [N, 8, 8] coefficients in natural order (int16 range), qt: [8, 8] table (any of 1..65535) -> ([N, 8, 8] uint8
    samples, [N, 8, 8] column-pass outputs of the general path before the int16 saturation)."""
    nat = np.asarray(nat, np.int64).reshape(-1, 8, 8)
    q = _w16(np.asarray(qt, np.int64).reshape(8, 8))
    d = _w16(nat * q)                                            # pmullw
    p1 = _pass(d, 11)                                            # column pass: [N, y, x]
    dc_only = ~np.any(nat[:, 1:, :] != 0, axis=(1, 2))
    short = np.broadcast_to(_w16(d[:, 0, :] << 2)[:, None, :], p1.shape)
    ws = np.where(dc_only[:, None, None], short, np.clip(p1, -32768, 32767))
    p2 = _pass(np.swapaxes(ws, 1, 2), 18)                         # row pass: [N, x, y]
    pix = np.clip(np.swapaxes(p2, 1, 2), -128, 127) + 128
    return pix.astype(np.uint8), p1


# ------------------------------------------------------------------------------------------------------ the crafted corpus
DQT_SWEEP = (1, 2, 4, 8, 16, 64, 255, 256, 1000, 32767, 65535)   # the last four need 16-bit tables (SOF1)
SIZES = {"gray": (27, 45), "420": (37, 51), "444": (19, 29), "422": (21, 43)}   # no side a multiple of the MCU


def dc_values(diffs, h: int, w: int, layout: str, restart: int = 0) -> np.ndarray:
    """The DC values a decoder's predictor takes for these coded differences (scan order): running sums per component,
    restarting at 0 with every restart interval."""
    bpm = mcu_grid(h, w, layout)[2]
    comp = block_components(h, w, layout)
    interval = np.arange(len(diffs)) // bpm // restart if restart else np.zeros(len(diffs), np.int64)
    out = np.zeros(len(diffs), np.int64)
    for c in range(3):
        for r in np.unique(interval):
            sel = (comp == c) & (interval == r)
            out[sel] = np.cumsum(np.asarray(diffs, np.int64)[sel])
    return out


def _family_blocks(family: str, h: int, w: int, layout: str, restart: int, rng) -> np.ndarray:
    """[blocks, 64] zigzag coefficients of one family (column 0: the DC predictor values)."""
    n = block_count(h, w, layout)
    z = np.zeros((n, 64), np.int64)
    diffs = rng.integers(-40, 41, n)
    if family == "dc_walk":                     # +-2047 differences in long runs: the predictor leaves int16 and comes back
        diffs = np.where((np.arange(n) // 40) % 2 == 0, 2047, -2047) * np.where(rng.random(n) < 0.1, -1, 1)
        z[:, 1] = rng.integers(-3, 4, n)
    elif family == "ac_single":                 # one +-1023 at each of the 63 positions in turn
        k = 1 + np.arange(n) % 63
        z[np.arange(n), k] = np.where((np.arange(n) // 63) % 2 == 0, 1023, -1023)
    elif family == "no_eob":                    # all 63 AC values non-zero: no EOB
        mag = rng.choice([1, 7, 100, 1023], (n, 63))
        z[:, 1:] = rng.integers(1, mag + 1) * rng.choice([-1, 1], (n, 63))
    elif family == "zrl":                       # ZRL chains ending at position 63
        z[np.arange(n), rng.integers(1, 16, n)] = rng.choice([-1023, -5, 1, 700], n)
        z[:, 63] = rng.choice([-1023, 1023, 1, -1], n)
    elif family == "random":                    # dense random extremes, a fifth of the blocks DC-only
        dens = rng.uniform(0.05, 1.0, (n, 1))
        mag = rng.choice([1023, 200, 30, 5], (n, 1))
        z[:, 1:] = np.where(rng.random((n, 63)) < dens, rng.integers(-mag, mag + 1, (n, 63)), 0)
        z[rng.random(n) < 0.2, 1:] = 0
        diffs = rng.integers(-2047, 2048, n)
    elif family == "wide":                      # WIDE_TABLES: AC values and DC differences up to +-32767
        mag = rng.choice([32767, 5000, 1023, 30], (n, 1))
        z[:, 1:] = np.where(rng.random((n, 63)) < 0.3, rng.integers(-mag, mag + 1, (n, 63)), 0)
        diffs = rng.integers(-32767, 32768, n)
    else:
        raise ValueError(family)
    z[:, 0] = dc_values(diffs, h, w, layout, restart)
    return z


FAMILIES = ("dc_walk", "ac_single", "no_eob", "zrl", "random", "wide")


def corpus():
    """[dict(name, data, coef, h, w, layout, qt, restart, tables)]: every family in every layout, with and without restart
    intervals, at every DQT value of the sweep. coef: what went in (the DC column is the predictor, unbounded); data: the file;
    tables: the supplied Huffman tables (None: Annex K)."""
    out = []
    for fi, family in enumerate(FAMILIES):
        for li, (layout, (h, w)) in enumerate(SIZES.items()):
            for restart in (0, 3):
                rng = np.random.default_rng([fi, li, restart])
                z = _family_blocks(family, h, w, layout, restart, rng)
                tables = WIDE_TABLES if family == "wide" else None
                for q in DQT_SWEEP:
                    qt = np.full(64, q, np.int64)
                    out.append(dict(name=f"{family}_{layout}_r{restart}_q{q}", coef=z, h=h, w=w, layout=layout, qt=qt, restart=restart,
                                    tables=tables, data=write_jpeg(z, h, w, layout, qt, restart=restart, tables=tables)))
    return out


def rewrite_dqt(data: bytes, value: int) -> bytes:
    """A copy of a baseline file with every quantisation table entry set to `value` (16-bit tables and SOF1 above 255); the
    scan and every other segment stay as they are."""
    out = bytearray(data[:2])
    i = 2
    while True:
        m, L = data[i + 1], int.from_bytes(data[i + 2:i + 4], "big")
        seg = data[i:i + 2 + L]
        if m == 0xDB:
            s, k, payload = seg[4:], 0, bytearray()
            while k < len(s):
                pq, t = s[k] >> 4, s[k] & 15
                k += 1 + 64 * (2 if pq else 1)
                wide = value > 255
                payload += bytes([(16 if wide else 0) | t]) + value.to_bytes(2 if wide else 1, "big") * 64
            seg = _segment(0xDB, bytes(payload))
        elif m == 0xC0 and value > 255:
            seg = bytes([0xFF, 0xC1]) + seg[2:]
        out += seg
        i += 2 + L
        if m == 0xDA:
            return bytes(out) + data[i:]


def pillow_rewrites(gray_frame, colour_frame):
    """[(name, file)]: the frames saved by Pillow at quality 100 — the grey one as one component and as 4:4:4 colour, the colour
    one as 4:4:4 and 4:2:0 — each with its quantisation tables rewritten to every value of DQT_SWEEP. The scans are Pillow's."""
    import io

    from PIL import Image

    out = []
    for label, frame, mode, sub in (("grey_L", gray_frame[..., 0], "L", 0), ("grey_444", gray_frame, "RGB", 0),
                                    ("colour_444", colour_frame, "RGB", 0), ("colour_420", colour_frame, "RGB", 2)):
        buf = io.BytesIO()
        Image.fromarray(np.ascontiguousarray(frame), mode).save(buf, "JPEG", quality=100, subsampling=sub)
        out += [(f"{label}_q{q}", rewrite_dqt(buf.getvalue(), q)) for q in DQT_SWEEP]
    return out
