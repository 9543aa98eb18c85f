"""Build libclimsr_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Every translation unit is compiled to an object file in parallel (build/ is git-ignored), then linked into
climsr_b200/libclimsr_b200.so.  ``python build.py --force`` rebuilds everything, ``-v`` adds ptxas resource usage,
``CSR_BUILD_TRACE=1`` compiles the per-role clock stamps of tools/trace_conv.py in.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
OUT = os.path.join(HERE, "climsr_b200", "libclimsr_b200.so")
SOURCES = sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CFLAGS = ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _defines():
    d = []
    if os.environ.get("CSR_BUILD_TRACE") == "1":
        d.append("-DCSR_ENABLE_TRACE")          # per-role clock stamps (tools/trace_conv.py)
    return d


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    return hdrs + [os.path.join(HERE, "..", "include", "climsr_b200.h"), __file__]


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def needs_build() -> bool:
    return _stale(OUT, [os.path.join(CSRC, s) for s in SOURCES] + _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    defs = _defines()
    tag = hashlib.md5(" ".join(defs).encode()).hexdigest()[:6]
    jobs = []
    for src in SOURCES:
        obj = os.path.join(OBJ, f"{src[:-3]}.{tag}.o")
        if force or _stale(obj, [os.path.join(CSRC, src)] + _deps()):
            jobs.append((src, [nvcc] + CFLAGS + defs + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]))

    def run(job):
        return job[0], subprocess.run(job[1], capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for src, r in ex.map(run, jobs):
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError(f"nvcc failed compiling {src}")
            if verbose:
                print(r.stdout + r.stderr)
    objs = [os.path.join(OBJ, f"{src[:-3]}.{tag}.o") for src in SOURCES]
    r = subprocess.run([nvcc] + ARCH + ["-shared", "-cudart", "static", "-o", OUT] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed linking libclimsr_b200.so")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
