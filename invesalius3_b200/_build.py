"""In-tree build recipes: libb2v.so (CUDA, sm_100a) and the CPU oracle.

nvcc cross-compiles without a GPU; the resulting .so files are git-ignored but travel
to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "libb2v.so"
OBJ = PKG / "csrc" / "_obj"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",              # reference arithmetic (Rust, NumPy) never contracts to FMA
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found; libb2v.so cannot be built")


def _newer(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def build_cuda(force: bool = False, verbose: bool = False) -> Path:
    """Compile every csrc/*.cu for sm_100a and link libb2v.so next to the package."""
    srcs = sorted(CSRC.glob("*.cu"))
    hdrs = sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) + sorted((ROOT / "include").glob("*.h"))
    OBJ.mkdir(exist_ok=True)
    nvcc = _nvcc()
    jobs = []
    for s in srcs:
        o = OBJ / (s.stem + ".o")
        if force or _newer(o, [s, *hdrs]):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(s), "-o", str(o)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        (OBJ / (s.stem + ".ptxas.txt")).write_text(r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s.name}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return o

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            list(ex.map(compile_one, jobs))
    objs = [OBJ / (s.stem + ".o") for s in srcs]
    if force or jobs or _newer(LIB, objs):
        cmd = [nvcc, "-shared", "-o", str(LIB), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a",
               "-Xcompiler", "-fPIC"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link of libb2v.so failed:\n{r.stdout}\n{r.stderr}")
    return LIB


def build_oracle(force: bool = False) -> Path:
    """Compile the CPU oracle (test infrastructure only) via oracle/Makefile, and the 3-D mask
    editor's restatement via oracle/mask_edit.mk."""
    for recipe in ([], ["-f", "mask_edit.mk"]):
        r = subprocess.run(["make", "-C", str(ROOT / "oracle"), *recipe, *(["-B"] if force else [])],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"oracle build failed:\n{r.stdout}\n{r.stderr}")
    return ROOT / "oracle" / "liboracle.so"


if __name__ == "__main__":
    force = "--force" in sys.argv
    print(build_cuda(force=force, verbose="-v" in sys.argv))
    print(build_oracle(force=force))
