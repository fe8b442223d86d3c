"""In-tree nvcc build of libb200ppf.so (sm_100a only).

The library is built next to the sources (yolo_ppf_pose_estimation_b200/_build/) so that it
travels with the repository snapshot to the GPU box; nothing is installed into site-packages.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
BUILD_DIR = os.path.join(_HERE, "_build")
LIB_PATH = os.path.join(BUILD_DIR, "libb200ppf.so")

SOURCES = ["capi.cu", "sort_scan.cu", "k1_features.cu", "k2_table.cu", "k3_vote.cu", "scene_grid.cu", "k4_cluster.cu", "verify.cu",
           "k5_transform.cu", "k6_icp.cu", "prep.cu", "microbench.cu", "group.cu", "k7_cvppf.cu"]
HEADERS = ["ppf_common.cuh", "ppf_math.cuh", os.path.join("..", "..", "include", "b200ppf.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    # the path's float arithmetic must round like PCL's un-fused x86 build (oracle: -ffp-contract=off)
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libb200ppf.so cannot be built (there is no CPU fallback)")


def _host_cxx() -> str:
    for cand in ("/usr/bin/g++", shutil.which("g++")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("g++ not found")


def _fingerprint() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    h.update(os.environ.get("B200PPF_NVCC_EXTRA", "").encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a and link libb200ppf.so. Returns its path."""
    os.makedirs(BUILD_DIR, exist_ok=True)
    stamp = os.path.join(BUILD_DIR, "fingerprint.txt")
    fp = _fingerprint()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == fp:
        return LIB_PATH
    nvcc, cxx = _nvcc(), _host_cxx()
    extra = os.environ.get("B200PPF_NVCC_EXTRA", "").split()  # tuning experiments, e.g. -DB200PPF_VOTE_THREADS=256
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(BUILD_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, "-ccbin", cxx] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + \
              ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- nvcc {src}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    link = [nvcc, "-ccbin", cxx, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs + \
           ["-cudart", "shared"]
    subprocess.run(link, check=True)
    with open(stamp, "w") as fh:
        fh.write(fp)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
