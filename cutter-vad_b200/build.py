"""Build recipe for libcvad_b200.so (nvcc, sm_100a only, in-tree)."""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
SRC = HERE / "csrc" / "cvad_capi.cu"
OUT = HERE / "libcvad_b200.so"
DEV_SRC = HERE / "csrc" / "cvad_dev.cu"            # development probes: a separate library, never loaded by the product
DEV_OUT = HERE / "libcvad_b200_dev.so"
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def sources():
    return sorted((HERE / "csrc").glob("*.cu")) + sorted((HERE / "csrc").glob("*.cuh")) + \
        [HERE.parent / "include" / "cutter_vad_b200.h"]


def _fresh(out: Path) -> bool:
    return out.exists() and all(out.stat().st_mtime >= s.stat().st_mtime for s in sources())


def build(force: bool = False, verbose: bool = False) -> Path:
    nvcc = os.environ.get("NVCC", "nvcc")
    extra = os.environ.get("CVAD_NVCC_EXTRA", "").split()          # extra nvcc flags for experimental builds
    for src, out in ((SRC, OUT), (DEV_SRC, DEV_OUT)):
        if not force and _fresh(out):
            continue
        cmd = [nvcc, *NVCC_FLAGS, *extra, *(["-Xptxas", "-v"] if verbose else []), "-o", str(out), str(src)]
        subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force=True, verbose=True))
