"""Builds ``libvqae_b200.so`` (the C-ABI library of include/vqae_b200.h) with nvcc for sm_100a.

In-tree, explicit ``nvcc -shared``: the .so sits next to the Python package so it travels to
the GPU box with the repository snapshot.  No torch headers are involved -- the boundary is a
plain C ABI loaded with ctypes (see ``vqae_b200/_lib.py``).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from pathlib import Path

CSRC = Path(__file__).resolve().parent
PKG = CSRC.parent
REPO = PKG.parent.parent
LIB_PATH = PKG / "libvqae_b200.so"
STAMP = PKG / ".libvqae_b200.stamp"

SOURCES = ["abi.cu", "conv_f32.cu", "stems.cu", "quantize.cu", "quantize_tc.cu", "tc_kernels.cu",
           "tc_down.cu", "tc_chain.cu", "tc_resident.cu", "up_tail.cu", "up_head.cu", "pack.cu",
           "mma_same.cu", "mma_down.cu", "mma_up.cu", "tc_split.cu", "mma_front.cu", "mma_stem.cu", "tc_down128.cu", "mma_same_split.cu", "ema.cu", "mbconv.cu",
           "quality.cu", "codemap_pack.cu"]
# test / measurement aids: a separate library that links against the product library
AID_SOURCES = ["testaids.cu", "tc_bench.cu"]
AIDS_PATH = PKG / "libvqae_b200_testaids.so"
HEADERS = ["common.cuh", "kernels.cuh", "tc_common.cuh", "mma_common.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]
OBJ_DIR = CSRC / "build"            # git-ignored ("build/"); objects are rebuilt per file


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise FileNotFoundError("nvcc not found; cannot build libvqae_b200.so")


def _headers_digest() -> str:
    h = hashlib.sha256()
    for f in [CSRC / s for s in HEADERS] + [REPO / "include" / "vqae_b200.h",
                                            REPO / "include" / "vqae_b200_testaids.h"]:
        h.update(f.name.encode())
        h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _digest() -> str:
    h = hashlib.sha256(_headers_digest().encode())
    for s in SOURCES + AID_SOURCES:
        h.update(s.encode())
        h.update((CSRC / s).read_bytes())
    return h.hexdigest()


def build_library(force: bool = False, verbose: bool = False) -> Path:
    """Compile if sources changed since the last build; return the library path.  One nvcc -c per
    changed .cu (in parallel), then one link."""
    from concurrent.futures import ThreadPoolExecutor
    digest = _digest()
    if not force and LIB_PATH.exists() and AIDS_PATH.exists() and STAMP.exists() \
            and STAMP.read_text() == digest:
        return LIB_PATH
    nvcc = _nvcc()
    OBJ_DIR.mkdir(exist_ok=True)
    hd = _headers_digest()
    logs = []

    def compile_one(src: str):
        obj = OBJ_DIR / (src + ".o")
        tag = OBJ_DIR / (src + ".sha")
        want = hashlib.sha256(hd.encode() + (CSRC / src).read_bytes()).hexdigest()
        if not force and obj.exists() and tag.exists() and tag.read_text() == want:
            return obj, 0, ""
        cmd = [nvcc, *NVCC_FLAGS, "-I", str(REPO / "include"), "-I", str(CSRC), "-c",
               str(CSRC / src), "-o", str(obj)]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode == 0:
            tag.write_text(want)
        return obj, proc.returncode, " ".join(cmd) + "\n" + proc.stdout + proc.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES + AID_SOURCES), os.cpu_count() or 4)) as ex:
        results = list(ex.map(compile_one, SOURCES + AID_SOURCES))
    logs = [r[2] for r in results if r[2]]
    failed = [r for r in results if r[1] != 0]
    if not failed:
        main_objs = [str(r[0]) for r in results[:len(SOURCES)]]
        aid_objs = [str(r[0]) for r in results[len(SOURCES):]]
        for cmd in (
            [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", str(LIB_PATH),
             *main_objs],
            [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", str(AIDS_PATH),
             *aid_objs, "-L", str(PKG), "-l:libvqae_b200.so", "-Xlinker", "-rpath=$ORIGIN"],
        ):
            proc = subprocess.run(cmd, capture_output=True, text=True)
            logs.append(" ".join(cmd) + "\n" + proc.stdout + proc.stderr)
            if proc.returncode != 0:
                failed = [(None, proc.returncode, logs[-1])]
                break
    log = "\n".join(logs)
    (PKG / "build.log").write_text(log)
    if failed:
        sys.stderr.write("\n".join(r[2] for r in failed))
        raise RuntimeError("nvcc failed building libvqae_b200.so (see output above)")
    if verbose:
        print(log)
    STAMP.write_text(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
