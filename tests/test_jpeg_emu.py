"""CPU: the codec kernels' host/device-shared logic (csrc/v5jpeg_enc.cuh, v5jpeg_dec.cuh), compiled by g++ with the threads of
a CTA emulated between barriers (tests/emu/v5jpeg_emu.cpp), against the oracle and the goldens. A debugging aid for strip /
edge / dummy-block indexing, the bit writer and the self-synchronising Huffman decoder in a container without a GPU; the
-m gpu tests are the real gate."""
import collections
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
    deps = [src] + [os.path.join(csrc, f) for f in ("v5jpeg_enc.cuh", "v5jpeg_dec.cuh", "v5jpeg_common.h", "v5jpeg_plan.h", "v5ela_device.cuh", "v5ela_host.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        tmp = f"{so}.{os.getpid()}.so"          # written aside, then renamed: parallel test processes never load a half-written file
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", *defs, "-I", os.path.join(ROOT, "include"),
                               "-I", csrc, src, "-o", tmp])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    u8p, i16p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_int16)
    lib.v5jemu_encode.restype = ctypes.c_int64
    lib.v5jemu_encode.argtypes = [u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int, u8p, ctypes.c_int64, i16p]
    lib.v5jemu_decode.argtypes = [u8p, ctypes.c_int64, u8p, u8p, i16p, ctypes.POINTER(ctypes.c_int), ctypes.c_int]
    vp, ip = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int)
    lib.v5jemu_plan_decode.argtypes = [vp, vp, ctypes.c_int, vp, vp] + [ctypes.c_int] * 6 + [ctypes.c_int64, vp, ctypes.c_int, vp, vp,
                                                                                           ctypes.c_int, ip, ip, ip]
    lib.v5jemu_info.argtypes = [u8p, ctypes.c_int64] + [ctypes.POINTER(ctypes.c_int)] * 3
    u32p = ctypes.POINTER(ctypes.c_uint32)
    lib.v5jemu_huff_actions.argtypes = [u8p, u8p, ctypes.c_int, ctypes.c_int, u32p, ctypes.c_int, u32p]
    return lib


TINY = ["-DV5J_HUFF_NT=8", "-DV5J_SUB_BITS=64"]
Emu = collections.namedtuple("Emu", "lib parts")          # parts: 0 = the one-launch flow, else the three-launch flow's parts


@pytest.fixture(scope="module", params=[("full", 0), ("tiny", 0), ("full", 3), ("tiny", 5)],
                ids=["full", "tiny", "full_parts", "tiny_parts"])
def emu(request):
    """'full': the shipped window (1024 subsequences of 1024 bits), the one-launch kernel's flow. 'tiny': 8 subsequences of
    64 bits per window, so that even small files cross many windows and need many synchronisation rounds. 'full_parts' /
    'tiny_parts': the three-launch flow with every file's windows shared out among up to 3 / 5 independent parts (blind
    starts, boundary fix-up walks)."""
    tag, parts = request.param
    return Emu(_build(tag, TINY if tag == "tiny" else []), parts)


def _u8(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


def emu_encode(emu, img, q, want_coef=False):
    img = np.ascontiguousarray(img)
    ch = 1 if img.ndim == 2 else 3
    h, w = img.shape[:2]
    cap = 4 * h * w * ch + 4096
    out = np.zeros(cap, np.uint8)
    coef = np.zeros((c_oracle.jpeg_blocks(h, w, ch), 64), np.int16)
    n = emu.lib.v5jemu_encode(_u8(img), h, w, ch, w * ch, q, _u8(out), cap, coef.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    assert 0 < n <= cap
    return (out[:n].tobytes(), coef) if want_coef else out[:n].tobytes()


def emu_decode(emu, data):
    buf = np.frombuffer(data, np.uint8)
    h, w, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rc = emu.lib.v5jemu_info(_u8(buf), len(data), ctypes.byref(h), ctypes.byref(w), ctypes.byref(c))
    if rc:
        raise ValueError(rc)
    rgb = np.zeros((h.value, w.value, 3), np.uint8)
    gray = np.zeros((h.value, w.value), np.uint8)
    hs, vs, _ = c_oracle.jpeg_layout(data)
    mcus = ((h.value + 8 * vs - 1) // (8 * vs)) * ((w.value + 8 * hs - 1) // (8 * hs))
    coef = np.zeros((mcus * (hs * vs + 2 if c.value == 3 else 1), 64), np.int16)
    rounds = ctypes.c_int()
    rc = emu.lib.v5jemu_decode(_u8(buf), len(data), _u8(rgb), _u8(gray), coef.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)),
                               ctypes.byref(rounds), emu.parts)
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
        return lib.v5jemu_decode(_u8(arr), len(arr), _u8(rgb), None, None, None, 0)

    assert rc_of(good) == 0
    bad = bytearray(good)
    bad[i + 5] = 3                                                  # three codes of length 1
    assert rc_of(bad) == -1
    bad = bytearray(good)
    bad[i + 5 + 15] = 200                                           # 200 more codes of length 16 than the segment has symbols for
    assert rc_of(bad) == -1


# ---------------------------------------------------------------------------------------------- the decoder's launch plan
# v5j::plan_decode (csrc/v5jpeg_plan.h) through v5jemu_plan_decode: the decisions both decode entry points run, checked without
# a device. A B200 has 148 SMs; the library caps a chunk's workspace at 8 GiB.
PLAN_FIELDS = ("files", "first", "off_tab", "off_q", "off_scan", "stage_bytes", "host_stage_bytes", "runs", "scan_bytes", "stream_bytes",
               "coef_blocks", "plane_bytes", "subs", "rst_entries", "max_windows", "max_intervals", "max_blocks", "max_groups",
               "one_launch", "parts", "launches", "images_hash", "runs_hash")
Plan = collections.namedtuple("Plan", "status bad_file chunks files runs")   # files: (chunk, position, tabset, qt, rgb_off, gray_off,
                                                                            # scan_off, rst_off) per file; runs: (chunk, device
                                                                            # offset, host address - files[0], bytes)


def plan_decode(files, sm_count=148, pinned=False, rgb_offsets=None, gray_offsets=None, want_rgb=True, want_gray=False, path=0, parts=0,
                cap=8 << 30, lib=None):
    """files: bytes or uint8 arrays (views into one buffer for `pinned`); path 1 / 3 and parts force what V5ELA_HUFF_PATH /
    V5ELA_HUFF_PARTS force."""
    lib = lib or _build("full", [])
    keep = [f if isinstance(f, np.ndarray) else np.frombuffer(f, np.uint8) for f in files]
    n = len(keep)
    ptrs = np.array([k.ctypes.data for k in keep], np.uintp)
    lens = np.array([len(k) for k in keep], np.int64)
    offs = [None if o is None else np.ascontiguousarray(o, np.int64) for o in (rgb_offsets, gray_offsets)]
    chunks = np.zeros((n + 1, len(PLAN_FIELDS)), np.int64)
    per_file = np.zeros((n, 8), np.int64)
    runs = np.zeros((n + 1, 4), np.int64)
    nc, nr, bad = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rc = lib.v5jemu_plan_decode(ptrs.ctypes.data, lens.ctypes.data, n, *[None if o is None else o.ctypes.data for o in offs],
                                int(want_rgb), int(want_gray), int(pinned), sm_count, path, parts, cap, chunks.ctypes.data, n + 1,
                                per_file.ctypes.data, runs.ctypes.data, n + 1, ctypes.byref(nc), ctypes.byref(nr), ctypes.byref(bad))
    rows = [dict(zip(PLAN_FIELDS, (int(v) for v in r))) for r in chunks[:nc.value]] if rc == 0 else []
    return Plan(rc, bad.value, rows, per_file, runs[:nr.value])


def carve(blobs, gaps):
    """The files laid out in one buffer (a loader's arena), gaps[i] bytes before file i + 1 -> views in file order."""
    starts = np.cumsum([0] + [len(b) + g for b, g in zip(blobs[:-1], gaps)])
    arena = np.zeros(int(starts[-1]) + len(blobs[-1]), np.uint8)
    views = []
    for b, s in zip(blobs, starts):
        arena[s:s + len(b)] = np.frombuffer(b, np.uint8)
        views.append(arena[s:s + len(b)])
    return views


def scan_range(blob):
    """(first byte, end) of a file's entropy-coded segment: after the SOS header, up to EOI."""
    rest = _segments(blob)[1]
    return len(blob) - len(rest), len(blob) - 2


def small_files(n, seed, h=96, w=128, q=90):
    from v5ela.synth import gen_batch

    return [pil_bytes(f, q) for f in gen_batch(0, n, h, w, seed=seed)]


def pil_bytes(rgb, q, **kw):
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, "JPEG", quality=q, **kw)
    return buf.getvalue()


def hd_files(n=8, q=95):
    """n 1080p q95 files (one picture, written n times: the plan only sees sizes)."""
    return [pil_bytes(golden_frame({"spec": ["gen", 3, 0], "h": 1080, "w": 1920}), q)] * n


def windows(blob, huff_nt=1024, sub_bits=1024):
    """The plan's window count of a file: (subsequences of its scan + 1) over the subsequences per window, rounded up."""
    a, e = scan_range(blob)
    subs = -(-(e - a) * 8 // sub_bits) + 1
    return -(-subs // huff_nt)


def test_plan_picks_the_huffman_path_from_the_batch():
    many = small_files(150, seed=8)
    p = plan_decode(many)
    assert [(c["files"], c["one_launch"], c["launches"]) for c in p.chunks] == [(150, 1, 5)]     # a file per SM: one launch
    hd = hd_files()
    p = plan_decode(hd)
    (c,) = p.chunks
    assert c["max_windows"] == windows(hd[0]) > 1
    assert (c["one_launch"], c["parts"], c["launches"]) == (0, min(16, 148 // 8, c["max_windows"]), 7)
    p = plan_decode(many[:1])                                                   # one file, one window: nothing to share out
    assert (p.chunks[0]["max_windows"], p.chunks[0]["one_launch"], p.chunks[0]["launches"]) == (1, 1, 5)
    rgb = golden_frame({"spec": ["gen", 2, 4], "h": 100, "w": 130})
    for ri in (1, 3, 7):
        ok, enc = cv2.imencode(".jpg", rgb, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_RST_INTERVAL, ri])
        ok, plain = cv2.imencode(".jpg", rgb, [cv2.IMWRITE_JPEG_QUALITY, 90])
        mcus = ((100 + 15) // 16) * ((130 + 15) // 16)
        for batch in ([None], [plain.tobytes(), None] + hd[:2]):            # None: the file with or without restart markers
            with_rst, without = (plan_decode([f or data for f in batch]).chunks[0] for data in (enc.tobytes(), plain.tobytes()))
            assert with_rst["launches"] == without["launches"] + 1 and without["rst_entries"] == 0
            assert with_rst["rst_entries"] == with_rst["max_intervals"] == -(-mcus // ri)
    # forced path and part count
    assert [c["one_launch"] for c in plan_decode(hd, path=1).chunks] == [1]
    assert [(c["one_launch"], c["launches"]) for c in plan_decode(many, path=3).chunks] == [(0, 7)]
    for parts, want in ((3, 3), (16, windows(hd[0])), (17, min(16, 148 // 8, windows(hd[0]))), (0, min(16, 148 // 8, windows(hd[0])))):
        assert plan_decode(hd, parts=parts).chunks[0]["parts"] == want, parts
    assert plan_decode(many[:1], parts=5, path=3).chunks[0]["parts"] == 1                       # clamped to the file's windows


def test_plan_chunks_keep_file_order_under_the_byte_cap():
    blobs = small_files(12, seed=1, h=64, w=80) + hd_files(2) + small_files(9, seed=2, h=130, w=70)
    one = [plan_decode([b]).chunks[0] for b in blobs]
    need = [c["scan_bytes"] * 2 + c["coef_blocks"] * 128 + c["plane_bytes"] + 256 for c in one]
    cap = 3 * max(need[:12])
    p = plan_decode(blobs, cap=cap)
    assert len(p.chunks) > 3
    used = lambda c: c["scan_bytes"] * 2 + c["coef_blocks"] * 128 + c["plane_bytes"]  # noqa: E731
    for k, c in enumerate(p.chunks):
        assert c["first"] == (p.chunks[k - 1]["first"] + p.chunks[k - 1]["files"] if k else 0)
        assert c["files"] == 1 or used(c) <= cap
        if k + 1 < len(p.chunks):
            assert used(c) + need[p.chunks[k + 1]["first"]] > cap                     # split at the first file that crosses
        idx = np.arange(c["first"], c["first"] + c["files"])
        assert (p.files[idx, 0] == k).all() and (p.files[idx, 1] == idx - c["first"]).all()
    assert sum(c["files"] for c in p.chunks) == len(blobs)
    # 65536 entries, one tiny file: no chunk takes more than 65535 files
    p = plan_decode([pil_bytes(np.zeros((8, 8, 3), np.uint8), 50)] * 65536)
    assert [(c["first"], c["files"]) for c in p.chunks] == [(0, 65535), (65535, 1)]


def test_plan_uploads_close_pinned_files_in_one_copy():
    blobs = small_files(4, seed=3)

    def runs_of(views):
        p = plan_decode(views, pinned=True)
        (c,) = p.chunks
        assert c["host_stage_bytes"] == c["off_scan"] < c["stage_bytes"] and c["runs"] == len(p.runs)
        base, dev = views[0].ctypes.data, p.files[:, 6]
        scan = [[v.ctypes.data - base + x for x in scan_range(v.tobytes())] for v in views]   # host addresses - files[0]
        i = 0
        for _, d, src, nbytes in p.runs:                  # files i .. j-1: first scan start .. last scan end, nothing more
            j = i + 1
            while j < len(views) and dev[j] < d + nbytes:
                j += 1
            assert (d, src, nbytes) == (dev[i], scan[i][0], scan[j - 1][1] - scan[i][0])
            assert all(dev[k] - d == scan[k][0] - src for k in range(i, j))    # the host distances, kept on the device
            i = j
        assert i == len(views)
        return len(p.runs)

    assert runs_of(carve(blobs, [0, 4095, 0])) == 1
    assert runs_of(carve(blobs, [0, 4096, 4095])) == 2
    assert runs_of(carve(blobs, [4096, 4096, 4096])) == 4
    assert runs_of(carve(blobs, [0, 0, 0])[::-1]) == 4                 # back to back, but handed over in reverse order
    p = plan_decode(carve(blobs, [0, 0, 0]), pinned=False)
    assert len(p.runs) == 0 and p.chunks[0]["runs"] == 0 and p.chunks[0]["host_stage_bytes"] == p.chunks[0]["stage_bytes"]


def test_plan_tables_and_output_offsets():
    rgb = golden_frame({"spec": ["gen", 4, 1], "h": 40, "w": 56})
    blobs = [pil_bytes(rgb, 90), pil_bytes(rgb, 75), pil_bytes(rgb[:17, :9], 90), pil_bytes(rgb, 60, optimize=True)]
    p = plan_decode(blobs, want_gray=True)
    assert p.files[:, 2].tolist() == [0, 0, 0, 1]                                      # 2 Huffman table sets
    assert p.files[:, 3].tolist() == [0, 1, 0, 2]                                      # 3 quantisation table pairs
    px = np.array([40 * 56, 40 * 56, 17 * 9, 40 * 56])
    packed = np.concatenate([[0], np.cumsum(px)[:-1]])
    assert p.files[:, 4].tolist() == (3 * packed).tolist() and p.files[:, 5].tolist() == packed.tolist()
    assert plan_decode(blobs).files[:, 5].tolist() == [-1] * 4                           # not wanted
    mine = [7, 100000, 0, 3 << 40]
    p = plan_decode(blobs, rgb_offsets=mine, gray_offsets=mine[::-1], want_gray=True)
    assert p.files[:, 4].tolist() == mine and p.files[:, 5].tolist() == mine[::-1]
    for which in ("rgb_offsets", "gray_offsets"):
        p = plan_decode(blobs, want_gray=True, **{which: [0, 10, -1, 20]})
        assert (p.status, p.bad_file, p.chunks) == (-1, 2, [])                         # V5ELA_ERR_INVALID, file 2
    assert plan_decode(blobs[:2] + [b"\xff\xd8\xff\xd9"] + blobs[2:]).status == -1
    assert plan_decode(blobs[:3] + [b""]).bad_file == -1


def _identity_cases():
    """The batches whose plans are pinned in PLANS, keyed by name -> (files, plan_decode keywords)."""
    from helpers import layout_golden_files

    golden = [pil_bytes(golden_frame(c), c["q"]) for c in JPEG["cases"]]
    layouts = [data for _, _, data, _ in layout_golden_files()]
    small = small_files(150, seed=8)
    hd = hd_files()
    rgb = golden_frame({"spec": ["gen", 2, 4], "h": 100, "w": 130})
    rst = [cv2.imencode(".jpg", rgb, [cv2.IMWRITE_JPEG_RST_INTERVAL, ri])[1].tobytes() for ri in (1, 3, 7)]
    gaps = [(0, 4095, 4096, 17)[i % 4] for i in range(len(golden) + len(layouts) - 1)]
    return {
        "golden": (golden, {"want_gray": True}),
        "layouts": (layouts, {}),
        "golden_layouts_pinned": (carve(golden + layouts, gaps), {"pinned": True, "want_gray": True}),
        "golden_small_cap": (golden, {"cap": 3 << 20, "want_rgb": False, "want_gray": True}),
        "golden_one_by_one": (golden[:6] + golden[-6:], {"sm_count": 1}),
        "small": (small, {}),
        "small_three": (small[:20], {"path": 3, "parts": 2}),
        "hd": (hd, {}),
        "hd_pinned_one": (carve(hd, [0] * 7), {"pinned": True, "path": 1}),
        "hd_parts": (hd[:3], {"parts": 5}),
        "restart": (rst + hd[:1] + rst, {"want_gray": True}),
        "offsets": (rst + layouts[:5], {"rgb_offsets": list(range(0, 8 * 1 << 20, 1 << 20)), "gray_offsets": [5] * 8,
                                        "want_gray": True}),
    }


# per case, per chunk: PLAN_FIELDS as the inline planning code of v5ela_jpeg_decode computed them before it became plan_decode
PLANS = {
    "golden": [
        (51, 0, 6944, 33136, 34672, 756096, 756096, 0, 721423, 723056, 83754, 5360256, 5712, 0, 4, 0, 48960, 259200, 0, 2, 7, 2782121060279068821, 7347990519673328018),
    ],
    "layouts": [
        (100, 0, 13600, 65984, 68032, 501184, 501184, 0, 433146, 436352, 71188, 4556032, 3536, 4167, 1, 1020, 6120, 16200, 1, 1, 6, 2978941992027741142, 7347990519673328018),
    ],
    "golden_layouts_pinned": [
        (151, 0, 20544, 72928, 75744, 1453728, 75744, 38, 1377975, 1159408, 154942, 9916288, 9248, 4167, 4, 1020, 48960, 259200, 1, 1, 6, 1983240762508035724, 5955425977745222354),
    ],
    "golden_small_cap": [
        (46, 0, 6256, 32448, 33984, 158320, 158320, 0, 124327, 125808, 12978, 830592, 1041, 0, 1, 0, 3060, 16200, 1, 1, 5, 4761793709795180871, 7347990519673328018),
        (1, 46, 144, 26336, 27872, 209248, 209248, 0, 181368, 181408, 21600, 1382400, 1418, 0, 2, 0, 21600, 115200, 0, 2, 7, 7172847507834886773, 7347990519673328018),
        (1, 47, 144, 26336, 27872, 436576, 436576, 0, 408695, 408736, 48960, 3133440, 3194, 0, 4, 0, 48960, 259200, 0, 4, 7, 1461264457432257590, 7347990519673328018),
        (3, 48, 416, 26608, 28144, 35152, 35152, 0, 7007, 7104, 216, 13824, 59, 0, 1, 0, 72, 360, 1, 1, 5, 4808306941922730919, 7347990519673328018),
    ],
    "golden_one_by_one": [
        (12, 0, 1632, 27824, 29360, 652256, 652256, 0, 622895, 623280, 73872, 4727808, 4885, 0, 4, 0, 48960, 259200, 1, 1, 5, 4034464199807197430, 7347990519673328018),
    ],
    "small": [
        (150, 0, 20400, 46592, 46848, 411280, 411280, 0, 364419, 369232, 43200, 2764800, 3043, 0, 1, 0, 288, 1536, 1, 1, 5, 7415665858578630172, 7347990519673328018),
    ],
    "small_three": [
        (20, 0, 2720, 28912, 29168, 77808, 77808, 0, 48626, 49280, 5760, 368640, 407, 0, 1, 0, 288, 1536, 0, 1, 7, 486575828909855675, 7347990519673328018),
    ],
    "hd": [
        (8, 0, 1088, 27280, 27536, 5543056, 5543056, 0, 5515514, 5515776, 391680, 25067520, 43104, 0, 6, 0, 48960, 259200, 0, 6, 7, 4892082029303608587, 7347990519673328018),
    ],
    "hd_pinned_one": [
        (8, 0, 1088, 27280, 27536, 5547392, 27536, 1, 5519847, 5515776, 391680, 25067520, 43104, 0, 6, 0, 48960, 259200, 1, 6, 5, 5975986920465846770, 1283703292144602290),
    ],
    "hd_parts": [
        (3, 0, 416, 26608, 26864, 2095184, 2095184, 0, 2068314, 2068416, 146880, 9400320, 16164, 0, 6, 0, 48960, 259200, 0, 5, 7, 8965784193501919565, 7347990519673328018),
    ],
    "restart": [
        (7, 0, 960, 27152, 27408, 746032, 746032, 0, 718620, 718848, 51228, 3278592, 5624, 186, 6, 63, 48960, 259200, 0, 6, 8, 8047436379921102236, 7347990519673328018),
    ],
    "offsets": [
        (8, 0, 1088, 27280, 27536, 42208, 42208, 0, 14661, 14928, 1151, 73664, 128, 96, 1, 63, 378, 1700, 1, 1, 6, 1962567815962931798, 7347990519673328018),
    ],
}


def test_plans_equal_the_pinned_table():
    cases = _identity_cases()
    assert set(cases) == set(PLANS)
    for name, (files, kw) in cases.items():
        p = plan_decode(files, **kw)
        assert p.status == 0, name
        assert [tuple(c[f] for f in PLAN_FIELDS) for c in p.chunks] == PLANS[name], name


@pytest.mark.parametrize("tag", ["full", "tiny"])
def test_emulator_decodes_with_the_parts_the_plan_picks(tag):
    """Each golden file as a batch of its own (the node's one-crop call): the path and part count its plan picks, pixels as Pillow's.
    The 'tiny' window (8 subsequences of 64 bits) gives every file many windows, and so the three-launch flow with up to 16 parts."""
    lib = _build(tag, TINY if tag == "tiny" else [])
    picked = set()
    for case in SMALL:
        data = pil_bytes(golden_frame(case), case["q"])
        (c,) = plan_decode([data], lib=lib).chunks
        parts = 0 if c["one_launch"] else c["parts"]
        picked.add(parts)
        out = emu_decode(Emu(lib, parts), data)
        assert np.array_equal(out["rgb"], np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))), _id(case)
    assert picked == {0} if tag == "full" else {0, 2, 3, 16} <= picked
