"""Build the CUDA extension (sm_100a) in-tree with nvcc.

The product is ONE shared library, rtabmap_b200/lib/liblcd_b200.so, exporting the C ABI of
include/lcd_b200.h.  It is compiled with
``-gencode arch=compute_100a,code=sm_100a -lineinfo`` (cross-compiles without a GPU) and is
git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "csrc"
LIB = ROOT / "lib" / "liblcd_b200.so"
SOURCES = ["engine.cu"]
HEADERS = ["common.cuh", "nn_hamming.cuh", "nn_tensor.cuh", "l2_path.cuh", "nn_tensor_f32.cuh", "resolve.cuh", "score.cuh", "bayes.cuh", "verify.cuh", "match_bf.cuh", "pnp_device.cuh", "orb.cuh", "gftt.cuh", "orb_pattern.h", "../../include/lcd_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "--fmad=false",  # fp64 PnP code must round like the host oracle; the integer kernels do not care
    "-shared", "-Xcompiler", "-fPIC",
    "-diag-suppress", "1886",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; the CUDA extension cannot be built")


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = [CSRC / s for s in SOURCES] + [(CSRC / h).resolve() for h in HEADERS]
    return any(d.exists() and d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile liblcd_b200.so if it is missing or older than its sources."""
    if not force and not needs_build():
        return LIB
    LIB.parent.mkdir(parents=True, exist_ok=True)
    tmp = LIB.with_name(f".{LIB.name}.{os.getpid()}.tmp")  # written beside the target and renamed: readers never see a partial file
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", str(tmp), *[str(CSRC / s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=str(CSRC))
    if res.returncode != 0:
        tmp.unlink(missing_ok=True)
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    os.replace(tmp, LIB)
    if verbose:
        print(res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
