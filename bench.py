#!/usr/bin/env python
"""bench.py — keyframes/s of the V5 ELA+texture hot path on N B200s (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C]     # N=1: plain python; N>1: launched under torchrun
    python bench.py --impl reference [...]                                # the reference's CPU path on the host cores
    python bench.py [...] --dump-outputs DIR                              # also write the last timed step's records as .npy

--config selects one of BASELINE.json's five configurations (default 2, the one the metric is quoted on):
  1  16 x 1280x720, q=90, per GPU (the reference's own CPU-runnable case)                          weak
  2  256 x 1920x1080, q=90, per GPU                                                                  weak
  3  1024 x 3840x2160, q=90, sharded over the N GPUs                                                 strong
  4  64 videos x 32 keyframes of 1080p, whole videos per rank, per-video records gathered by NCCL   strong
  5  512 x 1080p at q in {75, 85, 90, 95} (four passes per step), sharded over the N GPUs           strong
A step = one pass of the hot path over the configuration's batch, records-only mode, followed for N>1 by the NCCL gather of the
per-frame (config 4: per-video) records to rank 0.
  value     : whole-job frames/s with inputs resident in HBM (CUDA events, max over ranks). The timed region is --steps steps;
              with --min-seconds S > 0 steps are added until it lasts at least S: `steps` is what was timed, `timed_region_s`
              its length.
  e2e       : the same metric through the reference-facing C-ABI call with HOST (pinned) buffers — the H2D copy of every frame and
              the D2H copy of the records are inside the timed region; `ceiling_frames_s` = what a bare pinned cudaMemcpyAsync of
              the same bytes reaches on this rank at the same moment (all ranks copying concurrently), `per_rank_ms` every rank's time.
  roofline  : fused kernel only — algorithmic bytes (3*H*W + 3144 per frame) / its CUDA-event duration against the measured HBM
              copy bandwidth in MEASURED_PEAKS.json; `int_issue_frac` = the issue-slot utilisation ncu measured (the resource that
              binds the kernel), tagged with the hash of the sources it was profiled on.
  parity    : untimed spot-check of the timed call's records against the C oracle (oracle/ is only ever the checker).
  e2e_from_jpeg_files : (config 2) the same work starting from JPEG files in host memory — GPU decode + analyse.
  cpu_baseline : (N=1) the oracle port of the reference's ELA core (Pillow/libjpeg-turbo + NumPy/OpenCV statistics) on all host
              cores, on a bounded sample of the same frames. Reported, not the target.
--dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned to its caller — the records of every
              quality, after the per-video reduction (config 4) and the gather to rank 0 — one float64 file per record field,
              DIR/<field>.npy of shape (qualities, records, ...), and DIR/record_index.npy naming the records written: all of them
              up to 64 MB in all, beyond that a sample drawn with a fixed seed. The frames come from fixed seeds, so two builds run
              with the same arguments can be compared file for file.
--impl reference runs min(--steps, 8) steps of CPU work (each takes seconds) and reports that number as `steps`.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import time

# stdout must carry exactly one JSON line. Native libraries write there too (NCCL prints its version banner to stdout at the
# VERSION and WARN debug levels), so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to a
# duplicate of the original stdout (emit()).
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "fake-video-detection-engine_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

UNIT = "frames/s"
RECORD_BYTES = 3144

# name -> (frames, H, W, qualities, scaling, group, description); `frames` is per GPU for weak configurations, total for strong ones
CONFIGS = {
    1: dict(frames=16, h=720, w=1280, q=(90,), scaling="weak", group=0, metric="720p_keyframes_per_sec_v5_ela_texture",
            what="16 synthetic 1280x720 RGB keyframes per GPU, JPEG q=90 — BASELINE.json configs[0]"),
    2: dict(frames=256, h=1080, w=1920, q=(90,), scaling="weak", group=0, metric="1080p_keyframes_per_sec_v5_ela_texture",
            what="256 synthetic 1920x1080 RGB keyframes per GPU, JPEG q=90 — BASELINE.json configs[1]"),
    3: dict(frames=1024, h=2160, w=3840, q=(90,), scaling="strong", group=0, metric="4k_keyframes_per_sec_v5_ela_texture",
            what="1024 synthetic 3840x2160 RGB keyframes sharded over the GPUs, JPEG q=90 — BASELINE.json configs[2]"),
    4: dict(frames=2048, h=1080, w=1920, q=(90,), scaling="strong", group=32, metric="1080p_keyframes_per_sec_v5_ela_texture",
            what="64 synthetic 1080p videos x 32 keyframes (video v frame k = gen_frame(32v+k, seed=v)), whole videos per GPU, per-video "
                 "records reduced on the device and gathered by NCCL — BASELINE.json configs[3]"),
    5: dict(frames=512, h=1080, w=1920, q=(75, 85, 90, 95), scaling="strong", group=0, metric="1080p_keyframes_per_sec_v5_ela_texture",
            what="512 synthetic 1920x1080 RGB keyframes sharded over the GPUs, analysed at JPEG q in {75, 85, 90, 95} (four passes per "
                 "step; value counts frame-analyses) — BASELINE.json configs[4]"),
}


def local_range(cfg: dict, rank: int, world: int):
    """[lo, hi) of the configuration's frames this rank owns."""
    from v5ela.shard import shard_range, shard_videos

    if cfg["scaling"] == "weak":
        return rank * cfg["frames"], (rank + 1) * cfg["frames"]
    if cfg["group"]:
        return shard_videos(cfg["frames"] // cfg["group"], cfg["group"], rank, world)
    return shard_range(cfg["frames"], rank, world)


def workload_config(cid: int, n_gpus: int) -> dict:
    cfg = CONFIGS[cid]
    total = cfg["frames"] * (n_gpus if cfg["scaling"] == "weak" else 1)
    per_gpu_bytes = 3 * cfg["h"] * cfg["w"] * (cfg["frames"] if cfg["scaling"] == "weak" else math.ceil(cfg["frames"] / n_gpus))
    return {
        "workload": cfg["what"] + " (gen_frame, SURVEY App. B), records-only",
        "baseline_config": cid, "height": cfg["h"], "width": cfg["w"], "quality": list(cfg["q"]) if len(cfg["q"]) > 1 else cfg["q"][0],
        "global_frames": total, "frame_analyses_per_step": total * len(cfg["q"]), "group_size": cfg["group"],
        "l2": f"inputs ({per_gpu_bytes / 1e9:.2f} GB per GPU) " + ("are larger than the 126 MB L2; no flush needed" if per_gpu_bytes > 126e6 * 2
                                                                  else "fit the 126 MB L2: a 256 MB buffer is overwritten between timed steps"),
        "sharding": ("by frame, contiguous per rank" if not cfg["group"] else "by video, contiguous per rank") +
                    ("; one NCCL gather of 3144-byte records to rank 0 per step" if n_gpus > 1 else "; single GPU"),
    }


def source_hash() -> str:
    """Hash over the CUDA sources the library is built from, comments and white space removed (profiles/source_hash.py): what a
    profile has to match to describe this build."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("v5_source_hash", os.path.join(ROOT, "profiles", "source_hash.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.source_hash(os.path.join(PKG, "csrc"))


# ------------------------------------------------------------------------------------------------- CPU reference arm
_CPU_FRAMES = None


def _cpu_init(frames):
    global _CPU_FRAMES
    _CPU_FRAMES = frames
    try:
        import cv2

        cv2.setNumThreads(1)
    except Exception:
        pass


def _cpu_work(job):
    from oracle import pil_oracle

    i, q = job
    rec = pil_oracle.ela_core(_CPU_FRAMES[i % len(_CPU_FRAMES)], q)
    return int(rec["ela_sum"][0])


def cpu_reference_rate(cid: int, frames_per_step: int, repeats: int = 1, warmup: int = 0, distinct: int = 8):
    """Frame-analyses/s of the reference's CPU ELA core (+ §8a statistics) with one process per host core."""
    import multiprocessing as mp

    from oracle import pil_oracle
    from v5ela.synth import gen_frame

    cfg = CONFIGS[cid]
    cores = os.cpu_count() or 1
    pics = [gen_frame(i, cfg["h"], cfg["w"], 0) for i in range(min(distinct, frames_per_step))]
    jobs = [(i, q) for q in cfg["q"] for i in range(frames_per_step)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(pics,)) as pool:
        pool.map(_cpu_work, [(i, cfg["q"][0]) for i in range(cores)])           # spin the workers up
        for _ in range(warmup):
            pool.map(_cpu_work, jobs, chunksize=1)
        times = []
        for _ in range(max(1, repeats)):
            t0 = time.perf_counter()
            pool.map(_cpu_work, jobs, chunksize=1)
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return len(jobs) * len(times) / total, cores, total / len(times), pil_oracle.versions()


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = CONFIGS[args.config]
    # one step = the configuration's per-GPU batch, as in the native arm, bounded to ~256 frames of 1080p worth of CPU work
    budget_px = 256 * 1080 * 1920
    per_step = max(16, min(cfg["frames"], budget_px // (cfg["h"] * cfg["w"] * len(cfg["q"]))))
    steps = max(1, min(args.steps, 8))                          # ~2 s of CPU work per step on 16 cores: the arm ends within minutes
    fps, cores, step_s, versions = cpu_reference_rate(args.config, per_step, repeats=steps, warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": min(args.warmup, 1), "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": workload_config(args.config, args.gpus),
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{per_step} frames of {cfg['w']}x{cfg['h']} per step x {len(cfg['q'])} qualities x {steps} steps "
                                   "(8 distinct gen_frame pictures cycled)"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference arm: the reference's own operations (v5_texture_ela.py:66-73: PIL save q -> open -> ImageChops.difference -> "
                "getextrema) + NumPy/OpenCV record statistics, one process per host core; the reference module itself is pure Python "
                "over Pillow and is not present on the GPU box",
        "libraries": versions,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------------ clock sampling
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, power, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in out.strip().splitlines():
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
                power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower() == "active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [c for c, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir: str, per_quality: list) -> dict:
    """--dump-outputs: every field of the records (padding excluded) as float64 — exact for all of them — stacked over the
    qualities, DIR/<field>.npy of shape (qualities, records, ...), and DIR/record_index.npy, which records they are: all of them,
    or, where that would pass DUMP_LIMIT_BYTES (~6 kB per record and quality), a sample drawn with a fixed seed."""
    import numpy as np

    from v5ela.records import RECORD_DTYPE

    fields = [f for f in RECORD_DTYPE.names if f != "pad"]
    n = len(per_quality[0])
    per_record = 8 * len(per_quality) * (1 + sum(int(np.prod(RECORD_DTYPE[f].shape)) for f in fields))
    keep = min(n, DUMP_LIMIT_BYTES // per_record)
    index = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    arrays = {f: np.stack([r[f][index] for r in per_quality]).astype(np.float64) for f in fields}
    arrays["record_index"] = index.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "files": sorted(name + ".npy" for name in arrays), "bytes": sum(a.nbytes for a in arrays.values()),
            "records": n, "records_written": keep}


def load_profile_json(name: str):
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            return json.load(f)
    except Exception:
        return None


def load_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def set_affinity(local_rank: int) -> dict:
    """Run (and first-touch the pinned host buffers) on the CPU cores next to this rank's GPU: matters for `e2e` at N > 1."""
    try:
        import pynvml

        pynvml.nvmlInit()
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
        return {"ok": True, "cpus_before": before, "cpus_after": len(os.sched_getaffinity(0))}
    except Exception as e:  # reported, not hidden: the e2e figure at N > 1 depends on it
        return {"ok": False, "error": repr(e)[:200], "cpus": len(os.sched_getaffinity(0))}


# ---------------------------------------------------------------------------------------------------------- GPU arm
def run_native_arm(args):
    import torch
    import torch.distributed as dist

    import v5ela
    from v5ela import _abi
    from v5ela.batch import analyze_batch, get_handle, reduce_records
    from v5ela.records import as_records, combine
    from v5ela.shard import gather_records

    cid = args.config
    cfg = CONFIGS[cid]
    H, W, quals, group = cfg["h"], cfg["w"], cfg["q"], cfg["group"]
    bytes_per_frame = 3 * H * W + RECORD_BYTES                  # algorithmic bytes, SURVEY.md §8d
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cpu_baseline = None
    if world == 1 and not args.no_cpu:                          # before CUDA is initialised: the pool forks
        sample = max(16, min(8 * (os.cpu_count() or 1), (128 * 1080 * 1920) // (H * W)))
        fps, cores, _, versions = cpu_reference_rate(cid, sample, repeats=1)
        cpu_baseline = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{sample} frames of {W}x{H} (gen_frame) x {len(quals)} qualities, oracle/pil_oracle.ela_core = the "
                                  "reference's v5_texture_ela.py:66-73 calls + record statistics, one process per core",
                        "libraries": versions}
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU implementation (use --impl reference)")
    _abi.load()
    affinity = set_affinity(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime

        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))
    lo, hi = local_range(cfg, rank, world)
    n_local = hi - lo
    total = cfg["frames"] * (world if cfg["scaling"] == "weak" else 1)
    total_records = total // group if group else total

    if group:                                                   # config 4: video v frame k = gen_frame(32 v + k, seed = v)
        frames = torch.cat([v5ela.gen_batch_torch(group * v, group, H, W, seed=v, device=dev) for v in range(lo // group, hi // group)]) \
            if n_local else torch.empty((0, H, W, 3), dtype=torch.uint8, device=dev)
    else:
        frames = v5ela.gen_batch_torch(lo, n_local, H, W, seed=0, device=dev)
    records = torch.empty((len(quals), n_local, RECORD_BYTES), dtype=torch.uint8, device=dev)
    handle = get_handle(local_rank)
    if args.block_stage:
        handle.block_stage = args.block_stage
    small = n_local * 3 * H * W < 2 * 126e6
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None
    local_out = [None] * len(quals)                             # this rank's records of the latest step, per quality

    def step():
        for qi, q in enumerate(quals):
            analyze_batch(frames, quality=q, records_out=records[qi], handle=handle)
            local_out[qi] = reduce_records(records[qi], group, handle=handle) if group else records[qi]
            if world > 1:
                gather_records(local_out[qi], total_records)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()

    # ---- number of timed steps: --steps, or more when --min-seconds asks for a longer timed region
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    K = args.steps
    if args.min_seconds > 0:
        e0.record()
        step()
        e1.record()
        barrier()
        est = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(est, op=dist.ReduceOp.MAX)
        # (+5 %: a single step timed alone runs a little slower than the steps of the timed region, and the region must not end up short)
        K_min = int(math.ceil(1.05 * args.min_seconds * 1e3 / max(float(est.item()), 1e-3)))
        K = max(K, min(K_min, 200000 if not small else 4000))   # L2-sized inputs: one event pair and one flush per step

    # ---- device-resident throughput (value) + fused-kernel duration (roofline), clocks sampled during the region
    sampler = ClockSampler(local_rank) if rank == 0 else None
    handle.profile_enable(True)
    handle.profile_read(reset=True)
    launches0 = handle.launch_count
    barrier()
    if flush is None:
        e0.record()
        for _ in range(K):
            step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
    else:                                                       # inputs fit the L2: evict them between timed steps, time each step
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for a, b in evs:
            flush.fill_(1)
            a.record()
            step()
            b.record()
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = handle.launch_count - launches0
    fused_ms, fused_n = handle.profile_read(reset=True)
    handle.profile_enable(False)
    inst = handle.last_instantiation
    dumped = []
    if args.dump_outputs:
        # the gather returns a view of a receive block that the next gather overwrites, so each quality's result is gathered
        # again here (untimed, every rank takes part) from the records this rank computed in the last timed step, and copied
        for r in local_out:
            r = gather_records(r, total_records) if world > 1 else r
            if rank == 0:
                dumped.append(as_records(r))
    # keep the GPU busy a little longer so that slow nvidia-smi polling still sees the load (local work only)
    t_end = time.perf_counter() + 0.4
    while time.perf_counter() < t_end and n_local:
        analyze_batch(frames, quality=quals[0], records_out=records[0], handle=handle)
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())

    # ---- untimed parity spot-check of what was just timed, against the C oracle (rank 0)
    parity = None
    if rank == 0 and not args.no_parity and n_local:
        from oracle import c_oracle

        # `records` still holds what the last timed step wrote; nothing here may issue a collective (only rank 0 is in this branch)
        torch.cuda.synchronize()
        ok, checked = True, 0
        if group:                                               # video 0: device aggregate == combine(oracle records of its frames)
            host = frames[:group].cpu().numpy()
            orecs, _ = c_oracle.analyze(host, quals[0])
            agg = as_records(reduce_records(records[0][:group], group, handle=handle))
            ok = agg[0].tobytes() == combine(orecs).tobytes() and as_records(records[0][:group]).tobytes() == orecs.tobytes()
            checked = group
        else:
            picks = sorted({0, n_local // 3, (2 * n_local) // 3, n_local - 1})[: (2 if H * W > 4e6 else 4)]
            for qi, q in enumerate(quals):
                got = as_records(records[qi][picks])
                for j, i in enumerate(picks):
                    o = c_oracle.analyze_frame(frames[i].cpu().numpy(), q)
                    ok = ok and got[j].tobytes() == o["record"].tobytes()
                    checked += 1
        parity = {"frames": checked, "vs": "c_oracle", "ok": bool(ok), "instantiation": inst, "block_stage": handle.block_stage}

    # ---- end to end through the host-buffer C-ABI entry point (pinned host memory), on a bounded part of the local shard
    n_e2e = max(1, min(n_local, (4 << 30) // (3 * H * W)))
    host_frames = torch.empty((n_e2e, H, W, 3), dtype=torch.uint8, pin_memory=True)
    host_frames.copy_(frames[:n_e2e])
    host_records = torch.empty((n_e2e, RECORD_BYTES), dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream(dev).cuda_stream
    handle.set_quality(quals[0])

    def e2e_step():
        handle.analyze_host(host_frames.data_ptr(), n_e2e, H, W, host_records.data_ptr(), None, None, stream)
        if world > 1:
            gather_records(host_records.to(dev, non_blocking=True), n_e2e * world)   # every rank holds n_e2e records

    for _ in range(2):
        e2e_step()
    barrier()
    e0.record()
    e2e_step()
    e1.record()
    barrier()
    est_e = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:                                               # every rank must run the same number of steps: they end in a collective
        dist.all_reduce(est_e, op=dist.ReduceOp.MAX)
    Ke = max(2, min(50, int(math.ceil(1e3 / max(float(est_e.item()), 1e-3)))))            # about 1 s, at most 50 steps
    barrier()
    e0.record()
    for _ in range(Ke):
        e2e_step()
    e1.record()
    barrier()
    e2e_local_ms = e0.elapsed_time(e1)
    ok_e2e = bool(torch.equal(host_records, records[0][:n_e2e].cpu()))
    # the ceiling of that path: the same bytes through a bare pinned copy, every rank at the same time
    dst = torch.empty_like(host_frames, device=dev)
    dst.copy_(host_frames, non_blocking=True)
    barrier()
    e0.record()
    for _ in range(3):
        dst.copy_(host_frames, non_blocking=True)
    e1.record()
    barrier()
    h2d_ms = e0.elapsed_time(e1) / 3
    del dst
    per_rank = torch.tensor([e2e_local_ms, h2d_ms], dtype=torch.float64, device=dev)
    if world > 1:
        allr = [torch.empty_like(per_rank) for _ in range(world)]
        dist.all_gather(allr, per_rank)
    else:
        allr = [per_rank]
    e2e_ms = max(float(x[0]) for x in allr)
    h2d_ms_max = max(float(x[1]) for x in allr)

    # ---- the same work starting from JPEG FILES in host memory, the form V1 hands keyframes/crops over in
    # (cv2.imwrite default quality 95, v1_keyframes_facetrack.py:112,166): only compressed bytes cross PCIe; the GPU
    # decodes (SURVEY §8f-2), analyses, and the records come back. Config 2 only.
    files_leg = None
    if cid == 2 and not args.no_files:
        dt_local, Kf = -1.0, max(3, min(K, 12))                 # no collective inside the try: a failure on one rank must not hang the others
        try:
            from v5ela import jpeg
            from v5ela.batch import analyze_jpeg_files

            os.environ.setdefault("V5ELA_HOST_THREADS", str(max(1, (os.cpu_count() or 1) // world)))
            enc, enc_sizes = jpeg.encode_batch(frames, 95)                  # warm-up (workspace allocation), then timed once
            torch.cuda.synchronize()
            del enc, enc_sizes                                              # let the timed call reuse the 1.6 GB output block
            e0.record()
            enc, enc_sizes = jpeg.encode_batch(frames, 95)
            e1.record()
            torch.cuda.synchronize()
            encode_fps = n_local / (e0.elapsed_time(e1) * 1e-3)
            enc, enc_sizes = enc.cpu().numpy(), enc_sizes.cpu().numpy()
            # the files sit back to back in one page-locked arena (what a loader that reads files for the GPU would use)
            offs = [0]
            for i in range(n_local):
                offs.append(offs[-1] + (int(enc_sizes[i]) + 63) // 64 * 64)
            arena = torch.empty(offs[-1], dtype=torch.uint8, pin_memory=True)
            arena_np = arena.numpy()
            blobs = []
            for i in range(n_local):
                arena_np[offs[i]:offs[i] + enc_sizes[i]] = enc[i, :enc_sizes[i]]
                blobs.append(arena_np[offs[i]:offs[i] + int(enc_sizes[i])])
            del enc
            host_recs_f = torch.empty((n_local, RECORD_BYTES), dtype=torch.uint8, pin_memory=True)
            out = None
            for _ in range(2):
                out = analyze_jpeg_files(blobs, quality=quals[0], device=dev)
                host_recs_f.copy_(out["records"], non_blocking=True)
            torch.cuda.synchronize()
            same = bool(torch.equal(analyze_batch(out["rgb"], quality=quals[0])["records"].cpu(), host_recs_f))
            t0 = time.perf_counter()
            for _ in range(Kf):
                out = analyze_jpeg_files(blobs, quality=quals[0], device=dev)
                host_recs_f.copy_(out["records"], non_blocking=True)
            torch.cuda.synchronize()
            dt_local = time.perf_counter() - t0
            files_leg = {"value": None, "unit": UNIT, "steps": Kf,
                         "h2d_bytes_per_step": int(sum(len(b) for b in blobs)), "d2h_bytes_per_step": n_local * RECORD_BYTES,
                         "input": f"{n_local} JPEG files per GPU (4:2:0, quality 95, mean {sum(len(b) for b in blobs) / n_local / 1e3:.0f} kB) "
                                  "in one pinned host arena; header parsing on the host, wall clock, max over ranks",
                         "decode_status_ok": bool((out["status"] == 0).all().item()), "records_match_decoded_frames": same,
                         "files_written_by": "v5ela_jpeg_encode on the GPU (== cv2.imwrite's bytes), device-resident frames in, "
                                             f"{encode_fps:.0f} files/s (not part of the timed region)",
                         "api": "v5ela_jpeg_decode + v5ela_analyze (C ABI)"}
            del out
        except Exception as e:  # an extra figure must not take the headline down with it
            files_leg = {"error": repr(e)}
            dt_local = -1.0
        tt = torch.tensor([dt_local, -dt_local], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if float(tt[1]) > 0:                                    # some rank failed (its dt is -1)
            files_leg = files_leg if "error" in files_leg else {"error": "the files leg failed on another rank"}
        else:
            files_leg["value"] = n_local * world * Kf / float(tt[0])

    if rank == 0:
        peak, peak_src = load_peak()
        analyses = total * len(quals)
        value = analyses * K / (ms_max * 1e-3)
        kernel_ms = fused_ms / max(fused_n, 1)
        achieved = n_local * bytes_per_frame / (kernel_ms * 1e-3) / 1e9 if n_local else 0.0
        issue = load_profile_json("fused_kernel_issue.json") or {}
        dram = load_profile_json("fused_kernel_dram.json") or {}
        cur_hash = source_hash()
        traffic = None
        if dram.get("dram_bytes_per_frame") and (dram.get("height"), dram.get("width")) == (H, W):
            traffic = float(dram["dram_bytes_per_frame"]) * n_local
        e2e_frames = n_e2e * world
        line = {
            "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "steps_requested": args.steps,
            "warmup": warm, "ms_per_step": ms_max / K, "timed_region_s": ms_max * 1e-3, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": workload_config(cid, world),
            "e2e": {"value": e2e_frames * Ke / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": n_e2e * 3 * H * W, "d2h_bytes_per_step": n_e2e * RECORD_BYTES,
                    "frames_per_step_per_gpu": n_e2e, "steps": Ke, "records_match_device_path": ok_e2e,
                    "ceiling_frames_s": e2e_frames / (h2d_ms_max * 1e-3),
                    "ceiling": "bare pinned cudaMemcpyAsync of the same frames, all ranks concurrently, max over ranks "
                               f"({n_e2e * 3 * H * W / h2d_ms_max / 1e6:.1f} GB/s per GPU on the slowest rank)",
                    "per_rank_ms": [round(float(x[0]) / Ke, 3) for x in allr],
                    "per_rank_h2d_gbs": [round(n_e2e * 3 * H * W / float(x[1]) / 1e6, 1) for x in allr],
                    "affinity": affinity,
                    "api": "v5ela_analyze_host (C ABI, pinned host buffers, chunked copy/compute overlap)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": "ela_fused_kernel", "kernel_ms": kernel_ms,
                         "kernel_launches_timed": int(fused_n), "bytes_per_launch": n_local * bytes_per_frame,
                         "peak_source": peak_src,
                         "kernel_instantiation": f"ela_fused_kernel<{inst}> ({'width % 16 == 0, aligned, records only' if inst == 'fast' else inst}), "
                                                 f"block stage '{handle.block_stage}'",
                         "int_issue_frac": (issue.get("issue_slots_busy_pct") or 0) / 100.0 or None,
                         "int_issue": issue,
                         "profile_source_hash": issue.get("source_hash"), "build_source_hash": cur_hash,
                         "profile_matches_build": issue.get("source_hash") == cur_hash,
                         "note": "integer-issue / latency bound, not HBM bound: ~%d exact int32 thread-instructions per pixel (DESIGN.md 4.4); "
                                 "traffic, int_issue_frac and int_issue are ncu figures of the committed profile (profiles/), valid for this "
                                 "build only if profile_matches_build" % round(32 * (issue.get("warp_instructions_per_pixel") or 3.67))},
        }
        if parity is not None:
            line["parity"] = parity
        if files_leg is not None:
            line["e2e_from_jpeg_files"] = files_leg
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if args.dump_outputs:
            line["outputs"] = write_outputs(args.dump_outputs, dumped)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json configuration 1..5 (default 2)")
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="minimum length of the timed region: steps are added to --steps to reach it (default 0: exactly --steps)")
    ap.add_argument("--impl", choices=("native", "reference"), default="native")
    ap.add_argument("--block-stage", choices=("smem", "mma"), default=None, help="build of the fused kernel's block stage (default: library's)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed oracle spot-check")
    ap.add_argument("--no-files", action="store_true", help="skip the JPEG-files leg of config 2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the records of the last timed step to DIR/<field>.npy (float64); native arm only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs is for the native arm")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_native_arm(args)


if __name__ == "__main__":
    sys.exit(main())
