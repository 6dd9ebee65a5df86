"""In-tree nvcc build of libsknnr_b200.so (sm_100a only).

Used by ``__graft_entry__.build()`` and by ``python -m sknnr_b200._build``.  The product
never builds lazily at import time: a missing library is a loud error (``_lib.py``).
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIBNAME = "libsknnr_b200.so"
SOURCES = ["api.cu", "search_simt.cu", "search_tc.cu", "refine.cu", "project.cu", "hamming.cu", "forest.cu", "raster.cu", "misc.cu"]
HEADERS = ["common.cuh", "kernels.h", "tc_common.cuh", os.path.join("..", "..", "include", "sknnr_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas=-v", *os.environ.get("SK_NVCC_EXTRA", "").split(),
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libsknnr_b200.so")


def lib_path() -> str:
    # SKNNR_B200_LIB: load another build of the same library (A/B timing of kernel variants)
    return os.environ.get("SKNNR_B200_LIB") or os.path.join(LIBDIR, LIBNAME)


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False, variant: str = "", extra_flags=()) -> str:
    """``variant``: build into lib/libsknnr_b200_<variant>.so with ``extra_flags`` (e.g. -DSK_CHECKS)."""
    nvcc = nvcc_path()
    objdir = os.path.join(HERE, "build" + ("_" + variant if variant else ""))
    os.makedirs(objdir, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    logs = {}

    def compile_one(src: str) -> str:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s, *hdrs, os.path.abspath(__file__)]):
            cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            logs[src] = r.stderr
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return o

    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    out = os.path.join(LIBDIR, LIBNAME.replace(".so", f"_{variant}.so")) if variant else os.path.join(LIBDIR, LIBNAME)
    if force or _stale(out, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, *objs]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        for src, log in logs.items():
            print(f"==== {src}\n{log}")
    with open(os.path.join(objdir, "ptxas.log"), "a") as f:
        for src, log in logs.items():
            f.write(f"==== {src}\n{log}\n")
    return out


if __name__ == "__main__":
    var = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")]
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv, variant=var[0] if var else "",
                extra_flags=[a for a in sys.argv[1:] if a.startswith("-D")]))
