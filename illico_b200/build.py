"""Builds ``libillico_b200.so`` in-tree with nvcc for sm_100a (no GPU needed to compile)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libillico_b200.so")
SOURCES = ["api.cu", "stage.cu", "stage_dense_tma.cu", "fused.cu", "rank_ovr.cu", "rank_ovo.cu", "extras.cu", "counts.cu", "ttest.cu", "repart.cu", "recode.cu", "hostpack.c"]
HEADERS = ["common.cuh", "sort.cuh", "epilogue.cuh", "tma.cuh", os.path.join("..", "..", "include", "illico_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",            # strict f64 epilogue: no contraction (reference compute_pval is fastmath=False)
    "-Xcompiler", "-fPIC",
    "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compiles every source to an object (in parallel, only the stale ones) and links the shared library."""
    from concurrent.futures import ThreadPoolExecutor

    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdr_time = max(os.path.getmtime(os.path.normpath(os.path.join(CSRC, h))) for h in HEADERS)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o").replace(".c", ".o"))
        path = os.path.join(CSRC, src)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(path), hdr_time):
            return obj, ""
        if src.endswith(".c"):      # host-only code (the packed upload's squeeze loop): plain gcc
            cmd = [shutil.which("gcc") or "gcc", "-O3", "-fPIC", "-c", path, "-o", obj]
        else:
            cmd = [_nvcc()] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("compiler failed:\n" + res.stdout + res.stderr)
        return obj, res.stderr

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        done = list(ex.map(compile_one, SOURCES))
    res = subprocess.run([_nvcc(), "-shared", "-o", LIB] + [o for o, _ in done], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    if verbose:
        print("".join(log for _, log in done))
    return LIB


if __name__ == "__main__":
    import sys

    print(build(force=True, verbose="-v" in sys.argv))
