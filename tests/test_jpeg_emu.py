"""CPU: the codec kernels' host/device-shared logic (csrc/v5jpeg_enc.cuh, v5jpeg_dec.cuh), compiled by g++ with the threads of
a CTA emulated between barriers (tests/emu/v5jpeg_emu.cpp), against the oracle and the goldens. A debugging aid for strip /
edge / dummy-block indexing, the bit writer and the self-synchronising Huffman decoder in a container without a GPU; the
-m gpu tests are the real gate."""
import ctypes
import hashlib
import io
import os
import subprocess

import cv2
import numpy as np
import pytest
from PIL import Image

from helpers import check_layout_goldens, HERE, golden_frame, load_json, sha
from oracle import c_oracle

ROOT = os.path.dirname(HERE)
JPEG = load_json("jpeg_golden.json")
SMALL = [c for c in JPEG["cases"] if c["h"] * c["w"] <= 300 * 500]
_id = lambda c: f"{c['spec'][0]}{c['spec'][1]}_{c['h']}x{c['w']}_q{c['q']}"  # noqa: E731


def _build(tag, defs):
    so = os.path.join(HERE, "emu", f"libv5jpeg_emu_{tag}.so")
    src = os.path.join(HERE, "emu", "v5jpeg_emu.cpp")
    csrc = os.path.join(ROOT, "fake-video-detection-engine_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("v5jpeg_enc.cuh", "v5jpeg_dec.cuh", "v5jpeg_common.h", "v5ela_device.cuh", "v5ela_host.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = f"{so}.{os.getpid()}.so"          # written aside, then renamed: parallel test processes never load a half-written file
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", *defs, "-I", os.path.join(ROOT, "include"),
                               "-I", csrc, src, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    u8p, i16p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_int16)
    lib.v5jemu_encode.restype = ctypes.c_int64
    lib.v5jemu_encode.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int, u8p, ctypes.c_int64, i16p]
    lib.v5jemu_decode.argtypes = [u8p, ctypes.c_int64, u8p, u8p, i16p, ctypes.POINTER(ctypes.c_int)]
    lib.v5jemu_info.argtypes = [u8p, ctypes.c_int64] + [ctypes.POINTER(ctypes.c_int)] * 3
    u32p = ctypes.POINTER(ctypes.c_uint32)
    lib.v5jemu_huff_actions.argtypes = [u8p, u8p, ctypes.c_int, ctypes.c_int, u32p, ctypes.c_int, u32p]
    return lib


@pytest.fixture(scope="module", params=["full", "tiny", "full_parts", "tiny_parts"])
def emu(request):
    """'full': the shipped window (1024 subsequences of 1024 bits), the one-launch kernel's flow. 'tiny': 8 subsequences of
    64 bits per window, so that even small files cross many windows and need many synchronisation rounds. 'full_parts' /
    'tiny_parts': the three-launch flow with every file's windows shared out among up to 3 / 5 independent parts (blind
    starts, boundary fix-up walks)."""
    defs = {"full": [], "tiny": ["-DV5J_HUFF_NT=8", "-DV5J_SUB_BITS=64"], "full_parts": ["-DV5J_EMU_PARTS=3"],
            "tiny_parts": ["-DV5J_HUFF_NT=8", "-DV5J_SUB_BITS=64", "-DV5J_EMU_PARTS=5"]}[request.param]
    return _build(request.param, defs)


def _u8(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


def emu_encode(lib, img, q, want_coef=False):
    img = np.ascontiguousarray(img)
    ch = 1 if img.ndim == 2 else 3
    h, w = img.shape[:2]
    cap = 4 * h * w * ch + 4096
    out = np.zeros(cap, np.uint8)
    coef = np.zeros((c_oracle.jpeg_blocks(h, w, ch), 64), np.int16)
    n = lib.v5jemu_encode(_u8(img), h, w, ch, w * ch, q, _u8(out), cap, coef.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    assert 0 < n <= cap
    return (out[:n].tobytes(), coef) if want_coef else out[:n].tobytes()


def emu_decode(lib, data):
    buf = np.frombuffer(data, np.uint8)
    h, w, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rc = lib.v5jemu_info(_u8(buf), len(data), ctypes.byref(h), ctypes.byref(w), ctypes.byref(c))
    if rc:
        raise ValueError(rc)
    rgb = np.zeros((h.value, w.value, 3), np.uint8)
    gray = np.zeros((h.value, w.value), np.uint8)
    hs, vs, _ = c_oracle.jpeg_layout(data)
    mcus = ((h.value + 8 * vs - 1) // (8 * vs)) * ((w.value + 8 * hs - 1) // (8 * hs))
    coef = np.zeros((mcus * (hs * vs + 2 if c.value == 3 else 1), 64), np.int16)
    rounds = ctypes.c_int()
    rc = lib.v5jemu_decode(_u8(buf), len(data), _u8(rgb), _u8(gray), coef.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)),
                           ctypes.byref(rounds))
    if rc:
        raise ValueError(rc)
    return {"rgb": rgb, "gray": gray, "coef": coef, "rounds": rounds.value}


@pytest.mark.parametrize("case", SMALL, ids=_id)
def test_encoder_logic_reproduces_golden_files(emu, case):
    rgb = golden_frame(case)
    data, coef = emu_encode(emu, rgb, case["q"], want_coef=True)
    ref, ref_coef = c_oracle.jpeg_encode(rgb, case["q"], want_coef=True)
    assert np.array_equal(coef, ref_coef)
    assert data == ref
    assert (len(data), hashlib.sha256(data).hexdigest()[:16]) == (case["rgb_file_len"], case["rgb_file_sha"])
    data = emu_encode(emu, np.ascontiguousarray(rgb[..., 1]), case["q"])
    assert (len(data), hashlib.sha256(data).hexdigest()[:16]) == (case["gray_file_len"], case["gray_file_sha"])


@pytest.mark.parametrize("case", SMALL, ids=_id)
def test_decoder_logic_reproduces_golden_pixels(emu, case):
    rgb = golden_frame(case)
    buf = io.BytesIO()
    Image.fromarray(rgb, "RGB").save(buf, "JPEG", quality=case["q"])
    out = emu_decode(emu, buf.getvalue())
    ref = c_oracle.jpeg_decode(buf.getvalue(), want_coef=True)
    assert np.array_equal(out["coef"], ref["coef"])
    assert sha(out["rgb"]) == case["dec_rgb_sha"] and sha(out["gray"]) == case["dec_y_sha"]
    ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(rgb[..., 1]), [cv2.IMWRITE_JPEG_QUALITY, case["q"]])
    out = emu_decode(emu, enc.tobytes())
    assert sha(out["gray"]) == case["dec_gray_file_sha"]


def test_wide_images_cross_strip_boundaries(emu):
    rng = np.random.default_rng(3)
    for h, w in ((20, 300), (9, 520), (40, 771)):
        rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert emu_encode(emu, rgb, 90) == c_oracle.jpeg_encode(rgb, 90)
        gray = np.ascontiguousarray(rgb[..., 0])
        data = emu_encode(emu, gray, 95)
        assert data == c_oracle.jpeg_encode(gray, 95)
        assert np.array_equal(emu_decode(emu, data)["gray"], c_oracle.jpeg_decode(data)["gray"])


def test_decoder_custom_tables_and_noise(emu):
    rng = np.random.default_rng(4)
    rgb = rng.integers(0, 256, (64, 80, 3), dtype=np.uint8)
    for kw in ({"quality": 100}, {"quality": 60, "optimize": True}, {"quality": 5}):
        buf = io.BytesIO()
        Image.fromarray(rgb).save(buf, "JPEG", **kw)
        out = emu_decode(emu, buf.getvalue())
        assert np.array_equal(out["rgb"], np.asarray(Image.open(buf).convert("RGB"))), kw


@pytest.mark.parametrize("subsampling", [0, 1], ids=["444", "422"])
def test_decoder_other_chroma_layouts(emu, subsampling):
    """4:4:4 and 4:2:2 files (PIL subsampling=0 / 1): coefficients as the oracle's, pixels as Pillow's and OpenCV's."""
    rng = np.random.default_rng(40 + subsampling)
    sizes = [(1, 1), (7, 9), (8, 16), (16, 17), (33, 3), (2, 5), (40, 71), (64, 80), (90, 133), (5, 260)]
    for i, (h, w) in enumerate(sizes):
        rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if i % 2 else golden_frame({"spec": ["gen", i, 3], "h": h, "w": w})
        for q in (95, 60):
            buf = io.BytesIO()
            Image.fromarray(rgb).save(buf, "JPEG", quality=q, subsampling=subsampling)
            data = buf.getvalue()
            out = emu_decode(emu, data)
            ref = c_oracle.jpeg_decode(data, want_coef=True)
            assert np.array_equal(out["coef"], ref["coef"]), (h, w, q)
            assert np.array_equal(out["rgb"], np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))), (h, w, q)
            assert np.array_equal(out["gray"], cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_GRAYSCALE)), (h, w, q)


def test_decoder_restart_intervals(emu):
    """Files with restart markers (cv2 IMWRITE_JPEG_RST_INTERVAL, PIL restart_marker_blocks / _rows): every interval is decoded
    from its own known state; all three chroma layouts and one-component files; intervals of 1 MCU up to longer than the file."""
    rng = np.random.default_rng(77)
    for i, (h, w) in enumerate([(40, 48), (1, 1), (17, 130), (64, 64), (100, 37), (33, 260)]):
        rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if i % 2 else golden_frame({"spec": ["gen", i, 4], "h": h, "w": w})
        for ri in (1, 3, 7, 1000):
            ok, enc = cv2.imencode(".jpg", rgb, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_RST_INTERVAL, ri])
            data = enc.tobytes()
            out = emu_decode(emu, data)
            ref = c_oracle.jpeg_decode(data, want_coef=True)
            assert np.array_equal(out["coef"], ref["coef"]), (h, w, ri)
            assert np.array_equal(out["rgb"][..., ::-1], cv2.imdecode(enc, cv2.IMREAD_COLOR)), (h, w, ri)
            assert np.array_equal(out["gray"], cv2.imdecode(enc, cv2.IMREAD_GRAYSCALE)), (h, w, ri)
        for ss in (0, 1, 2):
            buf = io.BytesIO()
            Image.fromarray(rgb).save(buf, "JPEG", quality=75, subsampling=ss, restart_marker_blocks=2 + ss)
            out = emu_decode(emu, buf.getvalue())
            assert np.array_equal(out["rgb"], np.asarray(Image.open(io.BytesIO(buf.getvalue())).convert("RGB"))), (h, w, ss)
        ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(rgb[..., 1]), [cv2.IMWRITE_JPEG_RST_INTERVAL, 4])
        assert np.array_equal(emu_decode(emu, enc.tobytes())["gray"], cv2.imdecode(enc, cv2.IMREAD_GRAYSCALE))
    # a marker that has gone missing: refused, not decoded into something else
    ok, enc = cv2.imencode(".jpg", golden_frame({"spec": ["gen", 1, 2], "h": 64, "w": 64}), [cv2.IMWRITE_JPEG_RST_INTERVAL, 2])
    data = enc.tobytes()
    k = data.index(b"\xff\xd3", data.index(b"\xff\xda"))
    with pytest.raises(ValueError):
        emu_decode(emu, data[:k] + data[k + 2:])


def test_layout_goldens(emu):
    check_layout_goldens(lambda blobs: [emu_decode(emu, b) for b in blobs])


def test_unsupported_files_are_refused(emu):
    rgb = golden_frame({"spec": ["gen", 1, 2], "h": 40, "w": 40})
    for kw in ({"progressive": True},):
        buf = io.BytesIO()
        Image.fromarray(rgb).save(buf, "JPEG", quality=80, **kw)
        with pytest.raises(ValueError):
            emu_decode(emu, buf.getvalue())
    ok, enc = cv2.imencode(".jpg", rgb, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411])
    with pytest.raises(ValueError):
        emu_decode(emu, enc.tobytes())


# ---------------------------------------------------------------------------------------------- header parser robustness
def _segments(data):
    """[(marker, payload bytes)] of the header part, and the rest (entropy data + EOI)."""
    out, i = [], 2
    while True:
        assert data[i] == 0xFF
        m = data[i + 1]
        length = (data[i + 2] << 8) | data[i + 3]
        out.append((m, data[i + 4:i + 2 + length]))
        i += 2 + length
        if m == 0xDA:
            return out, data[i:]


def _assemble(segs, rest):
    b = bytearray(b"\xff\xd8")
    for m, payload in segs:
        b += bytes([0xFF, m]) + (len(payload) + 2).to_bytes(2, "big") + payload
    return bytes(b) + rest


def test_parser_accepts_equivalent_header_layouts(emu):
    """Other writers lay the same baseline stream out differently: all tables in one DHT / DQT segment, 16-bit quantisation
    entries, comment and application segments, fill bytes before markers. Decoded pixels must not change."""
    rgb = golden_frame({"spec": ["gen", 5, 1], "h": 70, "w": 90})
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, "JPEG", quality=85)
    data = buf.getvalue()
    ref = np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))
    segs, rest = _segments(data)
    dht = b"".join(p for m, p in segs if m == 0xC4)
    dqt = b"".join(p for m, p in segs if m == 0xDB)
    merged = [(m, p) for m, p in segs if m not in (0xC4, 0xDB, 0xC0, 0xDA)]
    merged += [(0xFE, b"a comment"), (0xE1, b"Exif\x00\x00" + bytes(40)), (0xDB, dqt), (0xC4, dht)]
    merged += [(m, p) for m, p in segs if m in (0xC0, 0xDA)]
    variant = _assemble(merged, rest)
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(variant)).convert("RGB")), ref)      # Pillow agrees it is the same image
    assert np.array_equal(emu_decode(emu, variant)["rgb"], ref)
    # 16-bit quantisation table entries (Pq = 1)
    wide = bytearray()
    j = 0
    while j < len(dqt):
        wide += bytes([0x10 | dqt[j]]) + b"".join(bytes([0, v]) for v in dqt[j + 1:j + 65])
        j += 65
    v16 = _assemble([(m, bytes(wide) if m == 0xDB else p) for m, p in merged], rest)
    assert np.array_equal(emu_decode(emu, v16)["rgb"], ref)
    # fill bytes (FF FF) before a marker
    i = variant.index(b"\xff\xc0")
    assert np.array_equal(emu_decode(emu, variant[:i] + b"\xff\xff" + variant[i:])["rgb"], ref)
    # trailing garbage after EOI
    assert np.array_equal(emu_decode(emu, data + b"\x00\x01garbage\xff")["rgb"], ref)


def test_parser_refuses_what_the_kernels_do_not_implement(emu):
    rgb = golden_frame({"spec": ["gen", 5, 1], "h": 40, "w": 48})
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, "JPEG", quality=85)
    data = buf.getvalue()
    i = data.index(b"\xff\xc0")
    twelve = bytearray(data)
    twelve[i + 4] = 12                                                   # sample precision
    with pytest.raises(ValueError):
        emu_decode(emu, bytes(twelve))
    cmyk = io.BytesIO()
    Image.fromarray(np.dstack([rgb, rgb[..., 0]]), "CMYK").save(cmyk, "JPEG", quality=85)
    with pytest.raises(ValueError):
        emu_decode(emu, cmyk.getvalue())
    for factor in (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440):   # 4x1 and 1x2 luma sampling
        ok, enc = cv2.imencode(".jpg", rgb, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, factor])
        assert ok
        with pytest.raises(ValueError):
            emu_decode(emu, enc.tobytes())
    for bad in (b"", b"\xff\xd8", data[:20], b"\x89PNG\r\n\x1a\n" + bytes(32), data[:i + 4]):
        with pytest.raises(ValueError):
            emu_decode(emu, bad)


def test_header_that_promises_more_than_the_data_holds_is_refused(emu):
    """A damaged SOF (65535 x 65535) over a few kilobytes of data must be refused before anything is sized by it."""
    rgb = golden_frame({"spec": ["gen", 5, 1], "h": 40, "w": 48})
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, "JPEG", quality=85)
    data = bytearray(buf.getvalue())
    i = data.index(b"\xff\xc0")
    data[i + 5:i + 9] = b"\xff\xff\xff\xff"
    with pytest.raises(ValueError):
        emu_decode(emu, bytes(data))
    with pytest.raises(ValueError):
        emu_decode(emu, buf.getvalue()[:len(buf.getvalue()) // 8 + 700])      # truncated early: too few bits for the blocks


def _canonical(bits, vals):
    """(length, code) -> symbol of the canonical Huffman code of a DHT segment (T.81 Annex C), independently of the C code."""
    out, code, k = {}, 0, 0
    for ln in range(1, 17):
        for _ in range(bits[ln - 1]):
            out[(ln, code)] = vals[k]
            code += 1
            k += 1
        code <<= 1
    return out


def _expected_action(codes, is_dc, win16):
    """What the decoder does with a window whose first 16 bits are win16 (v5jpeg_common.h pack_symbol)."""
    for ln in range(1, 17):
        sym = codes.get((ln, win16 >> (16 - ln)))
        if sym is not None:
            break
    else:
        sym, ln = 0, 16                                    # not a code: symbol 0, 16 bits
    if is_dc:
        size, zinc = min(sym, 15), 1
    else:
        size = sym & 15
        zinc = (sym >> 4) + 1 if size else (16 if (sym >> 4) == 15 else 64)
    return ln | (size << 8) | (zinc << 16) | ((ln + size) << 24)


def _dht_tables(jpeg_bytes):
    """[(is_dc, bits, vals)] of a file's DHT segments."""
    d, i, out = jpeg_bytes, 2, []
    while d[i + 1] != 0xDA:
        seg_len = (d[i + 2] << 8) | d[i + 3]
        if d[i + 1] == 0xC4:
            j = i + 4
            while j < i + 2 + seg_len:
                bits = list(d[j + 1:j + 17])
                n = sum(bits)
                out.append((d[j] >> 4 == 0, bits, list(d[j + 17:j + 17 + n])))
                j += 17 + n
        i += 2 + seg_len
    return out


def test_two_level_huffman_table_equals_canonical_code_for_every_window():
    """The decoder's table (look[] for codes of <= 9 bits, lng[] for the longer ones when they span <= 1024 windows, the
    maxcode walk otherwise) against the canonical code, for ALL 65536 leading 16-bit windows: Annex K tables, the optimised
    tables Pillow writes for several images, and synthetic tables whose long codes span more than 1024 windows (walk)."""
    lib = _build("full", [])
    rng = np.random.default_rng(5)
    tables = []
    for q, kw in ((90, {}), (95, {"optimize": True}), (30, {"optimize": True}), (100, {"optimize": True})):
        buf = io.BytesIO()
        img = rng.integers(0, 256, (96, 128, 3), dtype=np.uint8) if q != 30 else golden_frame(SMALL[0])
        Image.fromarray(img).save(buf, "JPEG", quality=q, **kw)
        tables += _dht_tables(buf.getvalue())
    # synthetic: 2 codes of 2 bits, 1 of 3 bits, then 200 codes of 12 bits (range 65536 - 0xA000 > 1024: walked), and a flat 8-bit code with one free word
    b = [0] * 16
    b[1], b[2], b[11] = 2, 1, 200
    tables.append((False, b, list(range(1, 204))))
    b = [0] * 16
    b[7] = 255                                          # windows 0xFFxx are not codes
    tables.append((False, b, list(range(255))))
    b = [0] * 16
    b[0], b[9], b[15] = 1, 3, 40                        # 1 code of 1 bit, 3 of 10 bits, 40 of 16: long codes start at 0x8000 (walked)
    tables.append((False, b, list(range(16, 60))))
    wins = (np.arange(65536, dtype=np.uint32) << 16) | rng.integers(0, 65536, 65536).astype(np.uint32)
    acts = np.zeros(65536, dtype=np.uint32)
    u32p = ctypes.POINTER(ctypes.c_uint32)
    seen_walk = seen_lng = 0
    for is_dc, bits, vals in tables:
        barr, varr = np.array(bits, dtype=np.uint8), np.array(vals + [0], dtype=np.uint8)
        lb = lib.v5jemu_huff_actions(_u8(barr), _u8(varr), len(vals), int(is_dc), wins.ctypes.data_as(u32p), 65536, acts.ctypes.data_as(u32p))
        assert lb >= 0
        seen_walk += lb == 0x10000 and any(bits[9:])
        seen_lng += lb < 0x10000
        codes = _canonical(bits, vals)
        exp = np.array([_expected_action(codes, is_dc, w) for w in range(65536)], dtype=np.uint32)
        bad = np.nonzero(acts != exp)[0]
        assert bad.size == 0, (is_dc, bits, hex(int(bad[0])), hex(int(acts[bad[0]])), hex(int(exp[bad[0]])))
    assert seen_walk >= 2 and seen_lng >= 8


def test_malformed_huffman_tables_are_refused_by_the_parser():
    """A DHT segment whose code lengths oversubscribe the code space (three codes of one bit) or promise more symbols than it
    carries must make parse_file fail (JPEG_CORRUPT = -1) — the decoder tables are only built later, once per distinct table set,
    and rely on the parser having checked every file's tables."""
    lib = _build("full", [])
    buf = io.BytesIO()
    Image.fromarray(golden_frame(SMALL[0])).save(buf, "JPEG", quality=80)
    good = bytearray(buf.getvalue())
    i = good.index(b"\xff\xc4")                                     # first DHT segment: marker, length (2), Tc/Th (1), 16 counts
    rgb = np.zeros((SMALL[0]["h"], SMALL[0]["w"], 3), np.uint8)

    def rc_of(data):
        arr = np.frombuffer(bytes(data), dtype=np.uint8).copy()
        return lib.v5jemu_decode(_u8(arr), len(arr), _u8(rgb), None, None, None)

    assert rc_of(good) == 0
    bad = bytearray(good)
    bad[i + 5] = 3                                                  # three codes of length 1
    assert rc_of(bad) == -1
    bad = bytearray(good)
    bad[i + 5 + 15] = 200                                           # 200 more codes of length 16 than the segment has symbols for
    assert rc_of(bad) == -1
