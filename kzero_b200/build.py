"""In-tree build of libkzb200.so with nvcc for sm_100a (B200).  No torch involvement: the product is a
plain C-ABI shared library.  `python -m kzero_b200.build` or `__graft_entry__.build()`.

The .so is written next to this file (kzero_b200/libkzb200.so), is git-ignored, and travels to the GPU
box with the snapshot.  nvcc cross-compiles here without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OBJ = PKG / "_obj"
LIB = PKG / "libkzb200.so"

SOURCES = ["onnx_reader.cpp", "net_spec.cpp", "api.cpp", "executor.cu", "encode.cu", "conv_fp32.cu", "conv_i2c.cu", "tower8k.cu", "heads.cu", "heads8.cu", "selfplay/selfplay.cpp"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
              "-Xcompiler", "-fPIC,-fvisibility=hidden,-Wall,-Wno-unknown-pragmas", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in [os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"]:
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found")


def _newest_dep() -> float:
    deps = [p for p in CSRC.rglob("*") if p.is_file()] + [PKG.parent / "include" / "kzb200.h", Path(__file__)]
    return max(p.stat().st_mtime for p in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and LIB.exists() and LIB.stat().st_mtime >= _newest_dep():
        return LIB
    nvcc = _nvcc()
    OBJ.mkdir(exist_ok=True)

    def compile_one(src: str):
        obj = OBJ / (src.replace("/", "_") + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-x", "cu", "-c", str(CSRC / src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=8) as ex:
        results = list(ex.map(compile_one, SOURCES))
    logs = []
    for src, obj, r in results:
        logs.append(f"== {src}\n{r.stderr}")
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    (OBJ / "ptxas.log").write_text("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    cmd = [nvcc, "-shared", "-o", str(LIB), *[str(o) for _, o, _ in results], "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
