"""In-tree build of libmdn_loss.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m mdn_sfm_b200.build [--force] [--verbose]

The library lands in mdn_sfm_b200/_lib/libmdn_loss.so: git-ignored, but shipped to the GPU box by gpurun.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "csrc", "mdn_loss.cu")
DEPS = [SRC, os.path.join(HERE, "csrc", "mdn_common.cuh"), os.path.join(HERE, "csrc", "mdn_fused.cuh"), os.path.join(HERE, "csrc", "mdn_resize.cuh"), os.path.join(HERE, "csrc", "mdn_metrics.cuh"), os.path.join(HERE, "csrc", "mdn_flow_eval.cuh"), os.path.join(ROOT, "include", "mdn_loss.h")]
OUT_DIR = os.path.join(HERE, "_lib")
OUT = os.path.join(OUT_DIR, "libmdn_loss.so")


def nvcc_path():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def up_to_date():
    return os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS)


def build(force=False, verbose=False):
    if up_to_date() and not force:
        return OUT
    os.makedirs(OUT_DIR, exist_ok=True)
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
           "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v",
           "--expt-relaxed-constexpr", "-I", os.path.join(ROOT, "include"), "-o", OUT, SRC]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed (exit %d)" % r.returncode)
    with open(os.path.join(OUT_DIR, "ptxas.log"), "w") as f:
        f.write(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
