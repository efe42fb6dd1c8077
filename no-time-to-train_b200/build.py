"""Build libnttt_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m no-time-to-train_b200.build      (or)      python no-time-to-train_b200/build.py

The library has no torch dependency: plain CUDA runtime (linked statically) behind the C-ABI declared in
include/nttt_b200.h.  Objects go to no-time-to-train_b200/csrc/_obj/ (git-ignored).
"""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB_PATH = os.path.join(PKG_DIR, "libnttt_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "--expt-relaxed-constexpr",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    # NTTT_BUILD_ABLATE=1: measurement build for tools/ablate.py (-DNTTT_ABLATE compiles the NTTT_STOP_AFTER switch
    # in).  The flavour is recorded next to the objects so that switching it rebuilds.
    ablate = os.environ.get("NTTT_BUILD_ABLATE", "0") not in ("", "0")
    flavour_file = os.path.join(OBJ, "flavour")
    flavour = "ablate" if ablate else "product"
    extra = ["-DNTTT_ABLATE"] if ablate else []
    extra += os.environ.get("NTTT_EXTRA_NVCC_FLAGS", "").split()  # A/B experiments (recorded in the flavour)
    flavour += " " + " ".join(extra)
    if not os.path.exists(flavour_file) or open(flavour_file).read() != flavour:
        force = True
        with open(flavour_file, "w") as f:
            f.write(flavour)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(PKG_DIR), "include", "nttt_b200.h"))
    headers.append(os.path.abspath(__file__))
    cc = nvcc()
    jobs = []
    objs = []
    for src in sources():
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + headers):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [cc, *NVCC_FLAGS, *extra, "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, r

    if jobs:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for src, r in ex.map(compile_one, jobs):
                log = os.path.join(OBJ, os.path.basename(src)[:-3] + ".ptxas.log")
                with open(log, "w") as f:
                    f.write(r.stderr)
                if verbose:
                    sys.stderr.write(r.stderr)
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    if jobs or force or _stale(LIB_PATH, objs):
        cmd = [cc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", *objs, "-o", LIB_PATH]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
