"""bench.py's command-line contract. CPU: the arm that runs without a GPU (--impl reference) prints exactly one JSON line on
stdout with the keys a caller reads; the native arm refuses to run without a CUDA device instead of falling back. GPU: the native
arm times exactly --steps steps and --dump-outputs writes what they computed."""
import json
import os
import subprocess
import sys

import pytest
from helpers import HERE

ROOT = os.path.dirname(HERE)


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "1080p_keyframes_per_sec_v5_ela_texture" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("256 synthetic 1920x1080")


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_native_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and p.stdout.strip() == ""
    assert "no CUDA device" in p.stderr


def test_bad_step_count_and_reference_dump_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120)
        assert p.returncode == 2 and p.stdout.strip() == "", extra


def test_dump_larger_than_the_limit_is_a_seeded_sample(tmp_path):
    """Past the size limit, --dump-outputs writes the same fixed sample of records every time, and says which ones."""
    code = f"""
import sys; sys.argv = ["bench.py"]; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, "fake-video-detection-engine_b200")!r}]
import numpy as np, bench
from oracle import c_oracle
from v5ela.synth import gen_batch
recs, _ = c_oracle.analyze(gen_batch(0, 40, 24, 40, seed=0), 90)
bench.DUMP_LIMIT_BYTES = 15 * 2 * 8 * 781                       # room for 15 of the 40 records at two qualities
for d in ("a", "b"):
    bench.write_outputs({str(tmp_path)!r} + "/" + d, [recs, recs[::-1]])
"""
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    import numpy as np

    from oracle import c_oracle
    from v5ela.synth import gen_batch

    recs, _ = c_oracle.analyze(gen_batch(0, 40, 24, 40, seed=0), 90)
    idx = np.load(tmp_path / "a" / "record_index.npy")
    assert len(idx) == 15 and len(set(idx)) == 15 and np.all(np.diff(idx) > 0)
    assert np.array_equal(idx, np.load(tmp_path / "b" / "record_index.npy"))
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= 15 * 2 * 8 * 781 + 16 * 128                 # + the .npy headers
    hist = np.load(tmp_path / "a" / "ela_hist.npy")
    assert hist.shape == (2, 15, 3, 256)
    assert np.array_equal(hist[0], recs["ela_hist"][idx.astype(int)]) and np.array_equal(hist[1], recs["ela_hist"][::-1][idx.astype(int)])


@pytest.mark.gpu
def test_native_arm_times_the_steps_asked_for_and_dumps_what_they_computed(tmp_path):
    """`steps` is exactly --steps; --dump-outputs writes the last timed step's records, one float64 file per field, identical from
    run to run and equal to the oracle's records of the same seeded frames."""
    import numpy as np

    from oracle import c_oracle
    from v5ela.records import RECORD_DTYPE
    from v5ela.synth import gen_frame

    fields = [f for f in RECORD_DTYPE.names if f != "pad"]
    dumps = []
    for run in range(2):
        out = tmp_path / f"run{run}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", "3", "--warmup", "1", "--no-cpu",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads(p.stdout)
        assert d["steps"] == 3 and d["parity"]["ok"]
        assert sorted(os.listdir(out)) == sorted(f + ".npy" for f in fields + ["record_index"]) == d["outputs"]["files"]
        assert np.array_equal(np.load(out / "record_index.npy"), np.arange(16.0)) and d["outputs"]["records_written"] == 16
        dumps.append({f: np.load(out / (f + ".npy")) for f in fields})
    for i in (0, 15):
        want = c_oracle.analyze_frame(gen_frame(i, 720, 1280, 0), 90)["record"]
        for f in fields:
            a = dumps[0][f]
            assert a.dtype == np.float64 and a.shape == (1, 16) + RECORD_DTYPE[f].shape, f
            assert np.array_equal(a, dumps[1][f]), f
            assert np.array_equal(a[0, i], want[f].astype(np.float64)), (i, f)


def test_profile_source_hash_ignores_comments_and_matches_the_committed_profile():
    """bench.py says whether the ncu figures it quotes (roofline.traffic, int_issue) describe the build it timed by comparing a
    hash of csrc/ with the one stamped into profiles/fused_kernel_*.json. The hash ignores comments and white space, changes with
    any token, and the committed profiles carry the hash of the committed sources."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("v5_source_hash", os.path.join(ROOT, "profiles", "source_hash.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    a = 'int f(int x) { return x /* not a comment in "s" */ + 1; }  // tail\nconst char *s = "a // b /* c */";\n'
    b = 'int f(int x)\n{\n    return x + 1;\n}\nconst char *s = "a // b /* c */";'
    assert mod.strip_code(a).strip() == mod.strip_code(b).strip()
    assert mod.strip_code(a) != mod.strip_code(a.replace("+ 1", "+ 2"))
    assert mod.strip_code(a) != mod.strip_code(a.replace('"a // b', '"a / b'))
    h = mod.source_hash(os.path.join(ROOT, "fake-video-detection-engine_b200", "csrc"))
    for name in ("fused_kernel_dram.json", "fused_kernel_issue.json"):
        with open(os.path.join(ROOT, "profiles", name)) as f:
            assert json.load(f)["source_hash"] == h, f"{name}: re-capture (profiles/final_run_r02.sh) and profiles/derive_fused_json.py after a kernel change"
