"""Build libmogstn.so (sm_100a only) in-tree with nvcc.  `python -m mog_asr_b200.build [--force]`."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
# MOG_SO: build (and, in _lib.py, load) another copy of the library, e.g. to compare two builds in one session
# (tools/kbench.py, tools/dbg_bwd.py)
SO = os.environ.get("MOG_SO") or os.path.join(PKG, "libmogstn.so")
SOURCES = ["mog_stn.cu", "mog_asr.cu", "mog_bce.cu", "mog_air.cu", "mog_air_head.cu", "mog_detection.cu", "mog_synth.cu"]
HEADERS = [os.path.join(CSRC, "mog_common.cuh"), os.path.join(CSRC, "mog_stn_warp.cuh"), os.path.join(CSRC, "mog_stn_bwd_col.cuh"), os.path.join(ROOT, "include", "mogstn.h")]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC or install CUDA 12.9+ under /usr/local/cuda)")


def flags(verbose: bool = False) -> list[str]:
    f = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
         "-ccbin", "/usr/bin/g++"]
    if verbose:
        f += ["-Xptxas", "-v"]
    return f


def stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return SO
    cmd = [nvcc_path()] + flags(verbose) + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", SO]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libmogstn.so (exit %d)" % res.returncode)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
