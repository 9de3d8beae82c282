"""CPU: the JPEG decoder's block stage on coefficients at the limits of what a baseline file can carry (tests/jpeg_craft.py):
AC values of +-1023 everywhere, DC differences of +-2047 walking the predictor outside int16, no-EOB blocks, ZRL chains, the
longest Annex K codes, quantisation entries 1..255 and 16-bit ones up to 65535 (SOF1), and supplied Huffman tables with the
non-baseline symbols (AC sizes 11..15, DC sizes up to 15). The reference is the decode Pillow and
OpenCV give on x86-64 (libjpeg-turbo's SIMD ISLOW path); the emulated device code (tests/emu/v5jpeg_emu.cpp) and the oracle must
both reproduce it bit for bit."""
import io
import platform

import cv2
import numpy as np
import pytest
from PIL import Image

import jpeg_craft as jc
from helpers import adversarial_blocks_frame
from oracle import c_oracle
from test_jpeg_emu import _build, Emu, emu_decode, TINY

CORPUS = jc.corpus()
REWRITES = jc.pillow_rewrites(*adversarial_blocks_frame())
FILES = [(e["name"], e["data"]) for e in CORPUS] + REWRITES


def reference(data):
    """Pillow's RGB and OpenCV's IMREAD_GRAYSCALE decode, or None where Pillow and OpenCV (IMREAD_COLOR) disagree."""
    rgb = np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))
    buf = np.frombuffer(data, np.uint8)
    if not np.array_equal(rgb, cv2.imdecode(buf, cv2.IMREAD_COLOR)[..., ::-1]):
        return None
    return {"rgb": rgb, "gray": cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE)}


@pytest.fixture(scope="module")
def refs():
    if platform.machine().lower() not in ("x86_64", "amd64"):
        pytest.skip(f"the reference is libjpeg-turbo's x86 SIMD inverse DCT; Pillow / OpenCV on {platform.machine()} run other code")
    out = [reference(data) for _, data in FILES]
    bad = [name for (name, _), r in zip(FILES, out) if r is None]
    if bad:
        pytest.skip(f"Pillow and OpenCV decode {len(bad)} crafted files differently (first: {bad[0]}): no single reference")
    return out


def test_writer_round_trips_through_the_oracle_and_pillow_opens_every_file():
    for e in CORPUS:
        got = c_oracle.jpeg_decode(e["data"], want_coef=True)["coef"]
        assert np.array_equal(got, e["coef"].astype(np.int16)), e["name"]        # the DC column: the int16 truncation
        im = Image.open(io.BytesIO(e["data"]))
        assert im.size == (e["w"], e["h"]) and im.mode == ("L" if e["layout"] == "gray" else "RGB"), e["name"]
        im.load()


def test_corpus_reaches_the_extremes():
    """What the corpus is for: column-pass values past int16, DC predictors outside int16, blocks without EOB, 16-bit codes,
    16-bit tables, restart intervals, sides that are not multiples of the MCU."""
    peak, dc_out, no_eob, lengths = 0, False, 0, set()
    for e in CORPUS:
        coef16 = e["coef"].astype(np.int16)
        nat = np.zeros((len(coef16), 64), np.int64)
        nat[:, jc.ZIGZAG] = coef16
        _, p1 = jc.simd_islow(nat.reshape(-1, 8, 8), e["qt"].reshape(8, 8))
        peak = max(peak, int(np.abs(p1).max()))
        dc_out |= bool((np.abs(e["coef"][:, 0]) > 32767).any())
        no_eob += int((e["coef"][:, 63] != 0).sum())
        if e["name"].endswith("_q1"):
            jc.write_jpeg(e["coef"], e["h"], e["w"], e["layout"], e["qt"], restart=e["restart"], tables=e["tables"], code_lengths=lengths)
    assert peak > 32767 and dc_out and no_eob > 0 and 16 in lengths
    assert any(e["qt"].max() > 255 for e in CORPUS) and any(b"\xff\xdd" in e["data"] for e in CORPUS)
    assert max(int(np.abs(e["coef"][:, 1:]).max()) for e in CORPUS) > 16383                # AC size 15
    assert all(e["h"] % (8 * jc.LAYOUTS[e["layout"]][2]) and e["w"] % (8 * jc.LAYOUTS[e["layout"]][1]) for e in CORPUS)


def test_numpy_model_is_the_reference_on_one_component_files(refs):
    """jpeg_craft.simd_islow (the model the kernels restate) gives Pillow's samples on every one-component crafted file."""
    for e, r in zip(CORPUS, refs):
        if e["layout"] != "gray":
            continue
        nat = np.zeros((len(e["coef"]), 64), np.int64)
        nat[:, jc.ZIGZAG] = e["coef"].astype(np.int16)
        pix, _ = jc.simd_islow(nat.reshape(-1, 8, 8), e["qt"].reshape(8, 8))
        mx, my, _ = jc.mcu_grid(e["h"], e["w"], "gray")
        plane = pix.reshape(my, mx, 8, 8).transpose(0, 2, 1, 3).reshape(8 * my, 8 * mx)
        assert np.array_equal(plane[:e["h"], :e["w"]], r["gray"]), e["name"]


def test_oracle_equals_pillow_and_opencv(refs):
    for (name, data), r in zip(FILES, refs):
        o = c_oracle.jpeg_decode(data)
        assert np.array_equal(o["rgb"], r["rgb"]), name
        assert np.array_equal(o["gray"], r["gray"]), name


@pytest.mark.parametrize("build,parts", [("full", 0), ("tiny", 0), ("full", 3), ("tiny", 5)],
                         ids=["full", "tiny", "full_parts", "tiny_parts"])
def test_emulated_decoder_equals_pillow_and_opencv(refs, build, parts):
    """Both builds of the emulator (the shipped window and 8 x 64-bit windows) and both Huffman flows (one launch per file,
    and the three-launch flow with the windows shared out among parts)."""
    emu = Emu(_build(build, TINY if build == "tiny" else []), parts)
    for (name, data), r in zip(FILES, refs):
        out = emu_decode(emu, data)
        assert np.array_equal(out["rgb"], r["rgb"]), name
        assert np.array_equal(out["gray"], r["gray"]), name
