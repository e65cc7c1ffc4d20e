"""Build libtip.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m trigenicinteractionpredictor_b200.build [--force] [--verbose]

The shared library lands next to this file (git-ignored, but it travels to the GPU box with the
tree).  There is no other backend: if the library is missing the package refuses to run.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
OBJ_DIR = os.path.join(HERE, "csrc", "_obj")
LIB_PATH = os.path.join(HERE, "libtip.so")

SOURCES = ["tip_api.cu", "tip_em.cu", "tip_generic.cu", "tip_mstep.cu", "tip_rows.cu", "tip_metrics.cu", "tip_peer.cu",
           "tip_reduce.cu", "tip_seg3.cu", "tip_pairs.cu", "tip_predict.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v",
    "--expt-relaxed-constexpr", "-I", INCLUDE, "-I", CSRC,
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libtip.so cannot be built and there is no fallback path")


def _digest() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(CSRC, name), "rb") as fh:
                h.update(name.encode() + b"\0" + fh.read())
    with open(os.path.join(INCLUDE, "tip.h"), "rb") as fh:
        h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile(nvcc: str, src: str, verbose: bool) -> str:
    obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
    cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = os.path.join(OBJ_DIR, src.replace(".cu", ".ptxas.log"))
    with open(log, "w") as fh:
        fh.write(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (src, res.stderr[-6000:]))
    if verbose:
        print(res.stderr)
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    stamp = os.path.join(OBJ_DIR, "stamp.sha256")
    want = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read().strip() == want:
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(lambda s: _compile(nvcc, s, verbose), SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fPIC", "-lcudart"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stderr[-4000:])
    with open(stamp, "w") as fh:
        fh.write(want)
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
