"""Builds libbmx.so (the CUDA kernels + C ABI) in-tree for sm_100a with nvcc.

The built library lives next to this file so that it travels to the GPU box with the source
snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libbmx.so"
REFMAIN_PATH = PKG_DIR / "bmx_refmain"

SOURCES = ["bmx_scan.cu", "bmx_abi.cu", "bmx_host.cu", "bmx_multi.cu", "bmx_multipat.cu", "bmx_exchange.cu", "bmx_ranges.cu", "bmx_dict.cu", "bmx_tables.cpp", "bmx_partition.cpp"]
HEADERS = ["bmx_internal.h", "bmx_scanner.h", "bmx_ctx.h", "../../include/bmx.h"]
NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC,-Wall,-pthread",
]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libbmx.so cannot be built (there is no CPU fallback)")
    return nvcc


def _stale(target: Path, deps: list[Path]) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile libbmx.so (and the bmx_refmain demo) if missing or older than its sources.
    One object per source (compiled in parallel, only the stale ones), then one link."""
    from concurrent.futures import ThreadPoolExecutor

    headers = [CSRC / h for h in HEADERS]
    objdir = CSRC / "build"
    objdir.mkdir(exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> Path:
        obj = objdir / (src.rsplit(".", 1)[0] + ".o")
        if force or _stale(obj, [CSRC / src, *headers]):
            cmd = [nvcc, *NVCC_FLAGS, "-c", "-o", str(obj), str(CSRC / src)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            subprocess.run(cmd, check=True, cwd=CSRC)
        return obj

    with ThreadPoolExecutor(len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB_PATH, objs):
        subprocess.run([nvcc, *NVCC_FLAGS, "-shared", "-o", str(LIB_PATH), *[str(o) for o in objs]], check=True, cwd=CSRC)
    refmain_src = CSRC / "bmx_refmain.cpp"
    if refmain_src.exists() and (force or _stale(REFMAIN_PATH, [refmain_src, LIB_PATH])):
        cmd = ["g++", "-O2", "-std=c++17", "-o", str(REFMAIN_PATH), str(refmain_src),
               f"-I{PKG_DIR.parent / 'include'}", f"-L{PKG_DIR}", "-lbmx", f"-Wl,-rpath,{PKG_DIR}",
               "-Wl,-rpath,$ORIGIN"]
        subprocess.run(cmd, check=True, cwd=CSRC)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
