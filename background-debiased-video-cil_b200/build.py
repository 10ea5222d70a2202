"""Builds libbgdebias_b200.so (C ABI, include/bgdebias.h) from csrc/*.cu with nvcc for sm_100a.

In-tree build: objects under csrc/_obj/, the library next to this file.  nvcc cross-compiles
without a GPU, so this runs in the build container; the resulting .so travels to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import pathlib
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = pathlib.Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
OBJ = CSRC / ("_obj" + ("_" + os.environ["BGD_BUILD_OUT"].replace(".", "_") if os.environ.get("BGD_BUILD_OUT") else ""))
LIB = PKG / os.environ.get("BGD_BUILD_OUT", "libbgdebias_b200.so")
EXTRA_DEFINES = [d for d in os.environ.get("BGD_BUILD_DEFINES", "").split() if d]
SOURCES = ["api.cu", "median_swar.cu", "median_bitsliced.cu", "median_tma_planner.cu", "median_colplane_c1.cu",
           "median_colplane_c2.cu", "median_colplane_c4.cu", "median_ldsm_q0.cu", "median_ldsm_q1.cu",
           "median_ldsm_q2.cu", "median_ldsm_q3.cu", "median_ldsm_q4.cu", "median_ldsm_q5.cu", "bgmix.cu", "raggedmix.cu", "nanreduce.cu", "cutmix.cu", "resize.cu",
           "resized_crop.cu", "shardpack.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-O2,-Wall",
    "-I", str(ROOT / "include"), "-I", str(CSRC),
    # no --use_fast_math: the blend must round every fp32 operation like the reference
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; cannot build libbgdebias_b200.so")
    return exe


def _stamp() -> str:
    h = hashlib.sha256()
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [ROOT / "include" / "bgdebias.h"]):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS + EXTRA_DEFINES).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> pathlib.Path:
    stamp_file = OBJ / "stamp"
    stamp = _stamp()
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    OBJ.mkdir(parents=True, exist_ok=True)
    nvcc = _nvcc()
    extra = ["-Xptxas", "-v"] if verbose else []

    def compile_one(src: str) -> None:
        cmd = [nvcc, *NVCC_FLAGS, *EXTRA_DEFINES, *extra, "-c", str(CSRC / src), "-o", str(OBJ / (src + ".o"))]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError(f"nvcc failed on {src}")

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        list(ex.map(compile_one, SOURCES))
    link = [nvcc, "-shared", "--cudart", "shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB),
            *[str(OBJ / (s + ".o")) for s in SOURCES]]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    stamp_file.write_text(stamp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
