"""Build csrc/*.cu into csrc/libpixelnerf_b200.so with plain nvcc for sm_100a (no torch headers).

nvcc cross-compiles without a GPU, so this runs in the CPU-only build container; the resulting .so is
git-ignored but travels to the GPU box with the repository snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(CSRC, "libpixelnerf_b200.so")
SOURCES = ["api.cu", "ray_tile.cu", "gather_pe.cu", "mlp_fp32.cu", "mlp_dispatch.cu", "mlp_umma_pair.cu", "field_bwd.cu", "encode_rays.cu", "train_umma.cu"]
HEADERS = ["pnr_common.cuh", "umma.cuh", "pnr_lab.h", "train_umma.cuh", os.path.join("..", "..", "include", "pixelnerf_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc() -> str:
    path = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(path):
        raise RuntimeError("nvcc not found: cannot build libpixelnerf_b200.so")
    return path


def _stamp() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    force = force or bool(os.environ.get("PNR_FORCE_BUILD"))
    stamp_file = os.path.join(CSRC, "build", "stamp")
    stamp = _stamp()
    if not force and os.path.exists(OUT) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        print(f"build: {os.path.basename(OUT)} is current (sha256 of sources + flags {stamp[:16]}); PNR_FORCE_BUILD=1 recompiles")
        return OUT
    print(f"build: compiling {len(SOURCES)} CUDA sources for sm_100a (stamp {stamp[:16]})")
    os.makedirs(os.path.join(CSRC, "build"), exist_ok=True)
    for stale in os.listdir(os.path.join(CSRC, "build")):          # objects of sources that no longer exist
        if stale.endswith(".o") and stale[:-2] + ".cu" not in SOURCES:
            os.remove(os.path.join(CSRC, "build", stale))
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(CSRC, "build", src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        with open(obj + ".log", "w") as fh:
            fh.write(r.stderr)
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp_file, "w") as fh:
        fh.write(stamp)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
