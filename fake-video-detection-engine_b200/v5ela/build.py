"""In-tree build of libv5ela.so with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(_HERE), "csrc")
LIB_PATH = os.path.join(_HERE, "libv5ela.so")


def build_library(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, f) for f in ("v5ela.cu", "v5ela_mma.cu", "v5jpeg.cu", "v5ela_device.cuh", "v5ela_dctmma.cuh", "v5ela_launch.cuh", "v5ela_workitem.cuh", "v5ela_host.h",
                                            "v5ela_fft.cuh", "v5ela_spec_plan.h", "v5ela_handle.h", "v5jpeg_common.h", "v5jpeg_enc.cuh", "v5jpeg_dec.cuh", "v5jpeg_dct.cuh", "v5jpeg_plan.h")]
    srcs.append(os.path.join(os.path.dirname(os.path.dirname(_HERE)), "include", "v5ela.h"))
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return LIB_PATH
    cmd = ["make", "-C", CSRC, "-B"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("building libv5ela.so failed (nvcc -gencode arch=compute_100a,code=sm_100a)")
    return LIB_PATH
