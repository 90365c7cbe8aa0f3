"""Build libquadx_b200.so (the C-ABI of include/quadx_b200.h) for sm_100a, in-tree.

    python fpv-drone-rl-agent_b200/csrc/build.py [--force]

nvcc cross-compiles without a GPU; the .so travels to the GPU box with the
repo snapshot (it is git-ignored, not gpurun-ignored)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
LIB = os.environ.get("QX_LIB_OUT") or os.path.join(HERE, "libquadx_b200.so")  # QX_LIB_OUT: tuning builds (QX_NVCC_EXTRA) next to the product library
SOURCES = ["qx_kernels.cu", "ppo_kernels.cu", "ppo_update_kernels.cu", "sac_kernels.cu"]
HEADERS = ["qx_model.cuh", "qx_lanes.cuh", "qx_ref_constants.cuh", "qx_internal.h", "tc05.cuh", os.path.join(ROOT, "include", "quadx_b200.h"), os.path.join(ROOT, "include", "ppo_b200.h"),
           os.path.join(ROOT, "include", "sac_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "--use_fast_math",  # FTZ + approximate div/sqrt in the once-per-step epilogue; parity tests hold
    "-fmad=false",  # no implicit contraction: every fused multiply-add is written as one (fmaf / __ffma2_rn), so that the same source gives the
                    # same roundings in every kernel instantiation (generic / specialised / paired kernels are compared bit for bit)
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
    "--threads", "0",  # the translation units compile in parallel
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
    deps.append(os.path.abspath(__file__))
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs = [os.path.join(HERE, s) for s in SOURCES if os.path.exists(os.path.join(HERE, s))]
    extra = os.environ.get("QX_NVCC_EXTRA", "").split()  # e.g. -DQX_MIN_BLOCKS=5 for tuning runs
    cmd = [nvcc, *NVCC_FLAGS, *extra, "-I", os.path.join(ROOT, "include"), "-o", LIB, *srcs]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    log_path = os.path.join(HERE, "build.log") if not os.environ.get("QX_LIB_OUT") else LIB + ".log"  # a tuning build keeps the product's log intact
    with open(log_path, "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log)
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
