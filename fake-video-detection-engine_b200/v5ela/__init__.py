"""v5ela — B200-native ELA + texture features for fake-video-detection-engine's V5 node.

Public surface:
  analyze_batch(frames_u8[N,H,W,3] on cuda) -> {"records", ["residual"], ["enhanced"]}   (v5ela.batch)
  analyze_ragged([frames_u8[H_i,W_i,3] ...]) -> the same for frames of different sizes, one launch (v5ela.batch)
  analyze_sweep(frames, qualities, want_ghost) -> records at many JPEG qualities in one launch, + JPEG-ghost maps (v5ela.batch)
  reduce_records(records, group)                                                           (v5ela.batch)
  spectrum_batch(gray_u8[N,H,W]) / spectrum_ragged([gray_u8[H_i,W_i] ...])  (FFT log-magnitude images) (v5ela.batch)
  as_records / features / combine / ghost_curve                                            (v5ela.records)
  gen_frame / gen_batch / gen_batch_torch  (synthetic keyframes, SURVEY Appendix B)        (v5ela.synth)
  shard_range / analyze_sharded            (multi-GPU, one process per GPU, NCCL gather)   (v5ela.shard)
  jpeg.encode_* / jpeg.decode_*            (baseline JPEG codec on the GPU, SURVEY §8f-2/3)  (v5ela.jpeg)
  analyze_jpeg_files(files)                (JPEG bytes in, records out: decode + analyse)   (v5ela.batch)
  handoff.face_detections_on_device        (V1 crop rule on device-resident frames, §8f-4)  (v5ela.handoff)
The drop-in node lives in ``nodes/V_nodes/v5_texture_ela.py`` next to this package.
"""
from .records import RECORD_BYTES, RECORD_DTYPE, as_records, combine, features, ghost_curve  # noqa: F401
from .synth import gen_batch, gen_batch_torch, gen_frame  # noqa: F401


def __getattr__(name):  # lazy: importing the package must not require the CUDA library (CPU-only tooling, tests)
    if name in ("analyze_batch", "analyze_ragged", "analyze_sweep", "reduce_records", "get_handle", "spectrum_batch", "spectrum_ragged", "analyze_jpeg_files"):
        from . import batch

        return getattr(batch, name)
    if name in ("shard_range", "analyze_sharded", "gather_records"):
        from . import shard

        return getattr(shard, name)
    raise AttributeError(name)
