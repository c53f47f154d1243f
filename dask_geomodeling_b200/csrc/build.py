"""Build libgeokernels.so in-tree with nvcc for sm_100a.

Usage: python -m dask_geomodeling_b200.csrc.build [--force] [--verbose]

Each .cu is compiled to an object (in parallel, skipped when up to date) and
linked into dask_geomodeling_b200/libgeokernels.so with a static cudart, so the
library has no dependency on torch or on a CUDA toolkit at run time.
"""
import os
import re
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
LIB = os.path.join(PKG, "libgeokernels.so")
BUILD = os.path.join(HERE, "build")

NVCC_FLAGS = [
    "-std=c++17",
    "-O3",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    # bit-exactness with the NumPy/SciPy CPU path: no FMA contraction, IEEE div/sqrt
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def sources():
    return sorted(f for f in os.listdir(HERE) if f.endswith(".cu"))


def _deps_mtime():
    hdrs = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cuh", ".h"))]
    include = os.path.join(os.path.dirname(PKG), "include")
    hdrs += [os.path.join(include, f) for f in os.listdir(include) if f.endswith(".h")]
    return max(os.path.getmtime(h) for h in hdrs)


_INCLUDE = re.compile(r'^#include "([^"]+)"[ \t]*$', re.M)


def _spliced(path, seen):
    """The text of `path` with every `#include "..."` replaced by the included file (found
    relative to the including one), itself spliced; a file already spliced is left out."""
    def include(m):
        inc = os.path.normpath(os.path.join(os.path.dirname(path), m.group(1)))
        if inc in seen:
            return ""
        seen.add(inc)
        return _spliced(inc, seen)
    return _INCLUDE.sub(include, open(path).read())


def _embed_prelude():
    """gm_jit_prelude.cuh, with the headers it includes spliced in -> build/gm_jit_prelude.inc
    (a C++ raw string literal that gm_jit.cu includes; NVRTC compiles it at run time, with no
    include path)."""
    src = os.path.join(HERE, "gm_jit_prelude.cuh")
    dst = os.path.join(BUILD, "gm_jit_prelude.inc")
    text = 'R"GMJIT(' + _spliced(src, {src}) + ')GMJIT"\n'
    if not os.path.exists(dst) or open(dst).read() != text:
        with open(dst, "w") as f:
            f.write(text)


def build(force=False, verbose=False):
    os.makedirs(BUILD, exist_ok=True)
    _embed_prelude()
    nvcc = _nvcc()
    hdr_time = _deps_mtime()
    jobs = []
    objs = []
    for src in sources():
        path = os.path.join(HERE, src)
        obj = os.path.join(BUILD, src[:-3] + ".o")
        objs.append(obj)
        stale = (
            force
            or not os.path.exists(obj)
            or os.path.getmtime(obj) < max(os.path.getmtime(path), hdr_time)
        )
        if stale:
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            jobs.append(cmd)

    def run(cmd):
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed: {}\n{}\n{}".format(" ".join(cmd), res.stdout, res.stderr))
        if verbose:
            sys.stderr.write(res.stderr)
        return 0

    if jobs:
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as pool:
            list(pool.map(run, jobs))
    stale_lib = not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs)
    if jobs or stale_lib or force:
        link = [nvcc, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
                "-Xcompiler", "-fPIC", "-o", LIB] + objs + ["-ldl"]
        run(link)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
