"""Drop-in replacement for the reference node ``nodes/V_nodes/v5_texture_ela.py`` (same module path, same ``run``).

Behaviour contract kept from the reference (line numbers: /root/reference/nodes/V_nodes/v5_texture_ela.py):
  * ``run(state) -> state``; inputs ``face_detections``, ``debug``, ``data_dir`` (:16-18), env ``OPENAI_API_KEY`` (:49);
    outputs ``texture_ela_score`` / ``texture_ela_details`` with the three reason strings (:22-23, :29-30, :176-177);
  * at most three faces, ranked by confidence * w * h of ``faces[0]`` (:33-42); artefacts ``ela_analysis/ela_{i}.jpg`` and
    ``fft_{i}.jpg`` numbered by rank (:80, :90); the GPT-4o request — model, prompts, three base64 JPEGs, JSON response
    format, 30 s timeout (:102-125); mean of ``fake_probability`` (:147-165); ``V5_debug.json`` keys (:166-173);
    any per-face failure is printed and skipped, never raised (:140-144).
What runs on the B200 instead of Pillow/OpenCV/NumPy:
  * decoding the crop file, both as RGB (:64) and as its luma plane (:83), through ``v5ela_jpeg_decode_host`` — pixel-identical;
  * the error-level analysis (:66-78) through ``v5ela_analyze_host`` — bit-exact;
  * the FFT log-magnitude image (:84-88) of every crop through one ``v5ela_spectrum_ragged_host`` call (within one grey level of
    NumPy; identical on every golden crop);
  * JPEG-encoding the three files the reference leaves in ``ela_analysis/`` — the scratch file ``temp_ela_{i}.jpg`` (:66-67,
    quality 90), ``ela_{i}.jpg`` (:80-81, quality 75) and ``fft_{i}.jpg`` (:90-91, quality 95, one component) — through
    ``v5ela_jpeg_encode_host``; the files equal the reference's byte for byte.
  There is no CPU fallback for any of it: a missing library or GPU — or a crop outside the GPU decoder's set (not a JPEG,
  progressive, CMYK, 12-bit: nothing V1 writes) — surfaces as that face's error, like any other analysis failure
  (reference :140-144). Reading and writing the files with Pillow/OpenCV instead is an explicit choice of the caller
  (``v5_gpu_codec = False``), never something the node decides on its own.
Optional state keys (defaults = the reference's literals): ``v5_quality`` 90, ``v5_max_faces`` 3, ``v5_device`` 0,
  ``v5_gpu_fft`` True (False: the reference's NumPy spectrum), ``v5_gpu_codec`` True (False: Pillow/OpenCV read and write the
  files), ``v5_keep_temp_jpeg`` True (the reference always leaves its scratch file behind, :66-67; nothing reads it, so a
  caller that does not want it may switch it off). The
  V5F v1 statistics of every analysed face are attached as ``ela_features`` to ``texture_ela_details`` entries and
  ``V5_debug.json`` (lr_node reads only ``avg_score``).
Host side, unchanged: the OpenAI call.
"""
import base64
import json
import os
import traceback

import cv2
import numpy as np
from dotenv import load_dotenv
from openai import OpenAI
from PIL import Image

from nodes import dump_node_debug

load_dotenv()

_SYSTEM_PROMPT = (
    "You are a forensic image analyst specializing in deepfake detection. "
    "You MUST return a JSON object (nothing else) with keys 'fake_probability' "
    "and 'reasoning'."
)
_USER_PROMPT = "Analyze this face for manipulation. Return JSON."


def _finish(state, score, details):
    state["texture_ela_score"] = score
    state["texture_ela_details"] = details
    return state


def _rank_faces(detections, limit):
    """Detections that carry a crop, best first by confidence x bbox area of their first face."""
    with_crops = [d for d in detections if d.get("faces")]

    def weight(det):
        face = det["faces"][0]
        return face["confidence"] * face["bbox"]["w"] * face["bbox"]["h"]

    return with_crops, sorted(with_crops, key=weight, reverse=True)[:limit]


def _read_crop(crop_path, device, gpu_codec):
    """The crop as RGB (reference :64) and as its luma plane (:83)."""
    if not gpu_codec:
        return np.asarray(Image.open(crop_path).convert("RGB")), cv2.imread(crop_path, cv2.IMREAD_GRAYSCALE)
    from v5ela import jpeg

    with open(crop_path, "rb") as fh:
        data = fh.read()
    planes = jpeg.decode_host([data], want_rgb=True, want_gray=True, device=device)[0]   # raises for unsupported files
    return planes["rgb"], planes["gray"]


def _write_jpeg(path, image, quality, device, gpu_codec):
    """``Image.save(path, 'JPEG', quality=q)`` / ``cv2.imwrite(path, gray)`` — the same bytes either way."""
    if gpu_codec:
        from v5ela import jpeg

        with open(path, "wb") as fh:
            fh.write(jpeg.encode_host(image[None], quality, device=device)[0])
    elif image.ndim == 3:
        Image.fromarray(image, "RGB").save(path, "JPEG", quality=quality)
    else:
        cv2.imwrite(path, image, [cv2.IMWRITE_JPEG_QUALITY, quality])


def _gpu_artefacts(crops, ela_dir, state):
    """ELA + spectrum artefacts of the selected crops. ``crops``: list of (rank, crop_path). All crops — whatever their sizes — go
    through ONE ragged analysis call (one upload, one launch sequence, one download: ``v5ela_analyze_ragged_host``) and ONE ragged
    spectrum call (``v5ela_spectrum_ragged_host``); a crop that cannot be read is reported and left out, like any per-face failure
    of the reference (:140-144).
    Returns {rank: (feature dict, ela path, fft path)}."""
    from v5ela import host as v5host
    from v5ela.records import features

    quality = int(state.get("v5_quality", 90))
    device = int(state.get("v5_device", 0))
    gpu_codec = bool(state.get("v5_gpu_codec", True))
    debug = state.get("debug", False)
    loaded = []
    for rank, crop_path in crops:
        try:
            rgb, gray = _read_crop(crop_path, device, gpu_codec)
            loaded.append((rank, rgb, gray))
        except Exception as e:
            print(f"Error analyzing face {rank}: {e}")
            if debug:
                traceback.print_exc()
    out = {}
    if not loaded:
        return out
    records, _, enhanced = v5host.analyze_ragged_host([rgb for _, rgb, _ in loaded], quality=quality, want_enhanced=True, device=device)
    gpu_fft = state.get("v5_gpu_fft", True)
    spectra = v5host.spectrum_ragged_host([gray for _, _, gray in loaded], device=device) if gpu_fft else None
    for j, (rank, rgb, gray) in enumerate(loaded):
        try:
            if state.get("v5_keep_temp_jpeg", True):
                _write_jpeg(os.path.join(ela_dir, f"temp_ela_{rank}.jpg"), rgb, quality, device, gpu_codec)
            feats = features(records[j], rgb.shape[0] * rgb.shape[1])
            feats["rank"] = rank
            ela_path = os.path.join(ela_dir, f"ela_{rank}.jpg")
            _write_jpeg(ela_path, enhanced[j], 75, device, gpu_codec)      # PIL's default quality (reference :81)
            if gpu_fft:
                spectrum = spectra[j]
            else:
                log_mag = 20 * np.log(np.abs(np.fft.fftshift(np.fft.fft2(gray))) + 1)
                spectrum = cv2.normalize(log_mag, None, 0, 255, cv2.NORM_MINMAX, dtype=cv2.CV_8U)
            fft_path = os.path.join(ela_dir, f"fft_{rank}.jpg")
            _write_jpeg(fft_path, spectrum, 95, device, gpu_codec)          # OpenCV's default quality (reference :91)
            out[rank] = (feats, ela_path, fft_path)
        except Exception as e:
            print(f"Error analyzing face {rank}: {e}")
            if debug:
                traceback.print_exc()
    return out


def _ask_model(client, image_paths):
    """One chat completion over (crop, ELA image, spectrum image); returns the raw message content."""
    parts = [{"type": "text", "text": _USER_PROMPT}]
    for path in image_paths:
        with open(path, "rb") as fh:
            b64 = base64.b64encode(fh.read()).decode("utf-8")
        parts.append({"type": "image_url", "image_url": {"url": f"data:image/jpeg;base64,{b64}"}})
    response = client.chat.completions.create(
        model="gpt-4o",
        messages=[{"role": "system", "content": _SYSTEM_PROMPT}, {"role": "user", "content": parts}],
        response_format={"type": "json_object"},
        timeout=30.0,
    )
    return response.choices[0].message.content


def _probabilities(results):
    out = []
    for item in results:
        value = item.get("fake_probability") if isinstance(item, dict) else item
        try:
            out.append(float(value))
        except Exception:
            pass
    return out


def run(state: dict) -> dict:
    print("Node V5: Running Texture & ELA Analysis...")
    detections = state.get("face_detections", [])
    debug = state.get("debug", False)

    if not detections:
        print("Node V5: No faces detected to analyze.")
        return _finish(state, 0.0, {"reason": "No faces found"})
    with_crops, chosen = _rank_faces(detections, int(state.get("v5_max_faces", 3)))
    if not with_crops:
        print("Node V5: Face detections present but no crops were generated.")
        return _finish(state, 0.0, {"reason": "No face crops available"})

    ela_dir = os.path.join(state.get("data_dir"), "ela_analysis")
    os.makedirs(ela_dir, exist_ok=True)

    api_key = os.getenv("OPENAI_API_KEY")
    client = OpenAI(api_key=api_key) if api_key else None
    if client is None:
        print("Node V5: OPENAI_API_KEY not found. Skipping OpenAI analysis.")

    # the GPU work of all selected crops in one batch (the reference decodes, re-encodes and transforms them one by one, :56-91)
    present = []
    for rank, detection in enumerate(chosen):
        try:
            crop_path = detection["faces"][0]["crop_path"]
            if os.path.exists(crop_path):
                present.append((rank, crop_path))
        except Exception as e:
            print(f"Error analyzing face {rank}: {e}")
    try:
        artefacts = _gpu_artefacts(present, ela_dir, state)
    except Exception as e:                                      # no library / no GPU: every face fails the way one would (:140-144)
        artefacts = {}
        for rank, _ in present:
            print(f"Error analyzing face {rank}: {e}")
        if debug:
            traceback.print_exc()

    verdicts, per_face = [], []
    for rank, crop_path in present:
        try:
            if rank not in artefacts:
                continue
            feats, ela_path, fft_path = artefacts[rank]
            per_face.append(feats)
            if client is None:
                continue
            content = _ask_model(client, (crop_path, ela_path, fft_path))
            if not content:
                if debug:
                    print(f"[DEBUG] V5: Empty response content for face {rank}, skipping.")
                continue
            try:
                verdict = json.loads(content)
            except Exception as parse_err:
                print(f"Error parsing OpenAI response for face {rank}: {parse_err}")
                if debug:
                    print(f"[DEBUG] V5: Raw content: {content}")
                continue
            if isinstance(verdict, dict):
                verdict.setdefault("ela_features", feats)
            verdicts.append(verdict)
        except Exception as e:
            print(f"Error analyzing face {rank}: {e}")
            if debug:
                traceback.print_exc()

    scores = _probabilities(verdicts)
    if not scores:
        print("Node V5: No analysis results generated.")
        details = {"reason": "Analysis failed or no keys"}
        if per_face:
            details["ela_features"] = per_face
        return _finish(state, 0.0, details)

    avg_score = sum(scores) / len(scores)
    print(f"Node V5: Analysis complete. Score: {avg_score:.2f}")
    _finish(state, avg_score, verdicts)
    dump_node_debug(state, "V5", {"faces_analyzed": len(verdicts), "avg_score": avg_score, "ela_features": per_face})
    return state
