"""Builds csrc/*.cu into ONE in-tree shared library, libtome_b200.so, for sm_100a (nvcc cross-compiles without a GPU).

The library has a plain C ABI (include/tome_b200.h) and links only cudart; there is no torch in its signatures.
Objects are cached by source mtime under csrc/_build/ so an edit to one kernel recompiles one file.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "_build")
LIB = os.path.join(HERE, "libtome_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
         "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _deps_mtime():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hdrs.append(os.path.join(HERE, "..", "include", "tome_b200.h"))
    return max(os.path.getmtime(h) for h in hdrs)


def _compile(src: str, verbose: bool) -> str:
    obj = os.path.join(BUILD, src[:-3] + ".o")
    sp = os.path.join(CSRC, src)
    if os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(sp), _deps_mtime()):
        return obj
    cmd = [NVCC, *FLAGS, "-c", sp, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    with open(obj[:-2] + ".ptxas.log", "w") as f:
        f.write(log)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{log}")
    if verbose:
        for line in log.splitlines():
            if "spill" in line and "0 bytes spill stores, 0 bytes spill loads" not in line:
                print(f"[build] {src}: {line.strip()}")
    return obj


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(BUILD, exist_ok=True)
    if force:
        for f in os.listdir(BUILD):
            os.remove(os.path.join(BUILD, f))
    srcs = _sources()
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), srcs))
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(o) for o in objs):
        cmd = [NVCC, "-shared", "-o", LIB, *objs, "-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(verbose=True, force="--force" in sys.argv))
