"""What the specialiser makes of a program, without a GPU: generate the fused kernel through
``gm_jit_source``, compile it with NVRTC for sm_100a (the options of ``gm_jit.cu``), disassemble it
with ``cuobjdump -sass`` and report for the hot loop (the loop over full chunks of U groups).  In the
two-set loop (programs whose two chunks of input fit ``kTwoSetWords`` of gm_jit.cu) one pass of it
evaluates two chunks, c from one register set and c + 1 from the other; the single-set loop evaluates
one chunk per pass:

  * instructions per pixel (loop instructions / (chunks per pass * U * V) pixels),
  * the opcode mix,
  * for each chunk of the pass (two-set loop: each half, up to its stores), the position of each
    LDG in it and whether all of them come before its first compare (the first ISETP / FSETP /
    DSETP: evaluation has started).  In the two-set loop the LDGs of a half load the NEXT chunk, so
    "all before" means chunk c + 1 is in flight while chunk c is evaluated,
  * registers and spills (ptxas).

The baked variant (``gm_jit_baked_source``) has the program's constants as literals: the kernel
``jit_launch`` builds when a program's constants repeat on large rasters; the unbaked variant is
what runs under ``GM_JIT_NO_BAKE`` or on the first launches of a program.

    python tools/jit_sass.py [--shapes cfg2,cfg1,reclass200] [--dump DIR]
"""
import argparse
import collections
import ctypes
import glob
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from dask_geomodeling_b200 import _native, workloads  # noqa: E402
from dask_geomodeling_b200.raster import _program  # noqa: E402
from dask_geomodeling_b200.raster._program import Leaf, Node  # noqa: E402

CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
# the options of nvrtc_compile in gm_jit.cu, plus -v for the register / spill report
NVRTC_OPTS = ["--gpu-architecture=sm_100a", "-std=c++17", "-fmad=false", "-prec-div=true",
              "-prec-sqrt=true", "-ftz=false", "-lineinfo", "-default-device", "-Xptxas=-v"]
F4 = (np.dtype("f4"), workloads.F32_MAX)


def shapes():
    """name -> (expression, leaf types)."""
    r = Node("reclassify", [Leaf(0)], dtype="int64", fillvalue=np.iinfo("i8").max,
             data=workloads.CFG2_PAIRS, select=True)
    st = Node("step", [Node("clip", [Leaf(1), r])], left=0, right=1, value=50.0, at=0.5)
    cfg1 = Node("maskbelow", [Node("multiply", [Node("add", [Leaf(0), Leaf(1)], dtype="float32",
                                                     fillvalue=workloads.F32_MAX), 0.5],
                                   dtype="float32", fillvalue=workloads.F32_MAX)], value=40.0)
    big = Node("reclassify", [Leaf(0)], dtype="int64", fillvalue=np.iinfo("i8").max,
               data=[(k, 1) for k in range(0, 400, 2)], select=False)
    big = Node("isdata", [Node("clip", [Leaf(1), big])])
    def add_chain(n, dtype):
        t = (np.dtype(dtype), np.finfo(dtype).max)
        node = Leaf(0)
        for i in range(1, n):
            node = Node("add", [node, Leaf(i)], dtype=dtype, fillvalue=t[1])
        return node, [t] * n
    return {
        "cfg2": (Node("isdata", [st]), [(np.dtype("i2"), 32767), F4]),
        "add4_f4": add_chain(4, "f4"),
        "add8_f4": add_chain(8, "f4"),
        "cfg1": (cfg1, [F4, F4]),
        "reclass200": (big, [(np.dtype("i2"), 32767), F4]),
    }


def generate(node, leaf_types):
    """(unbaked source, baked source) of the program of `node`, from the library."""
    prog, _, results = _program.compile_expression([node], leaf_types)
    ins = (ctypes.c_int32 * max(len(leaf_types), 1))(*[_native.dtype_code(d) for d, _ in leaf_types])
    outs = (ctypes.c_int32 * len(results))(*[_native.dtype_code(t.dtype) for t in results])
    lib = _native.load_library()
    sources = []
    for fn in (lib.gm_jit_source, lib.gm_jit_baked_source):
        length = ctypes.c_int64()
        if fn(ctypes.byref(prog), ins, outs, None, 0, ctypes.byref(length)):
            raise RuntimeError(lib.gm_last_error().decode())
        buf = ctypes.create_string_buffer(length.value + 1)
        fn(ctypes.byref(prog), ins, outs, buf, length.value + 1, ctypes.byref(length))
        sources.append(buf.value.decode())
    return sources


def nvrtc_compile(src):
    libs = sorted(glob.glob(os.path.join(CUDA, "lib64", "libnvrtc.so*")))
    if not libs:
        raise RuntimeError("libnvrtc not found under " + CUDA)
    lib = ctypes.CDLL(libs[-1])
    prog = ctypes.c_void_p()
    if lib.nvrtcCreateProgram(ctypes.byref(prog), src.encode(), b"gm_fused.cu", 0, None, None):
        raise RuntimeError("nvrtcCreateProgram failed")
    opts = (ctypes.c_char_p * len(NVRTC_OPTS))(*[o.encode() for o in NVRTC_OPTS])
    rc = lib.nvrtcCompileProgram(prog, len(NVRTC_OPTS), opts)
    n = ctypes.c_size_t()
    lib.nvrtcGetProgramLogSize(prog, ctypes.byref(n))
    log = ctypes.create_string_buffer(n.value)
    lib.nvrtcGetProgramLog(prog, log)
    if rc:
        raise RuntimeError("NVRTC failed:\n" + log.value.decode())
    lib.nvrtcGetCUBINSize(prog, ctypes.byref(n))
    cubin = ctypes.create_string_buffer(n.value)
    lib.nvrtcGetCUBIN(prog, cubin)
    lib.nvrtcDestroyProgram(ctypes.byref(prog))
    return cubin.raw, log.value.decode()


INSTR = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_.]+)([^;]*);")


def sass(cubin):
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "k.cubin")
        with open(path, "wb") as f:
            f.write(cubin)
        text = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", path], check=True,
                              capture_output=True, text=True).stdout
    return [(int(m.group(1), 16), m.group(3), m.group(4).strip()) for m in INSTR.finditer(text)], text


def hot_loop(instrs):
    """The loop over full chunks: the first loop (backward branch) that stores to global memory
    (the loop before it, if any, copies tables into shared memory)."""
    for i, (addr, op, args) in enumerate(instrs):
        if op.split(".")[0] == "BRA":
            target = int(args.split(",")[-1].strip(), 16)
            if target < addr:
                start = next(j for j, ins in enumerate(instrs) if ins[0] == target)
                if any(o.startswith("STG") for _, o, _ in instrs[start:i + 1]):
                    return instrs[start:i + 1]
    raise RuntimeError("no loop found")


def analyse(src):
    """Hot-loop facts of a generated source: a dict with two_sets, pixels (per loop pass), loop (its
    instructions), halves (per chunk of the pass: LDG positions and the first compare, relative to
    it), registers, spills (bytes stored and loaded) and the ptxas log."""
    m_v, m_u = re.search(r"p\.n / (\d+);", src), re.search(r"chunk = 256LL \* (\d+);", src)
    cubin, log = nvrtc_compile(src)
    instrs, text = sass(cubin)
    loop = hot_loop(instrs)
    ops = [op.split(".")[0] for _, op, _ in loop]
    two_sets = "p.chunks_per_block" in src
    stg = [i for i, op in enumerate(ops) if op == "STG"]
    cut = stg[len(stg) // 2 - 1] + 1          # after the stores of the first chunk
    halves = []
    for lo, hi in (((0, cut), (cut, len(ops))) if two_sets else ((0, len(ops)),)):
        part = ops[lo:hi]
        halves.append({"ldg": [i for i, op in enumerate(part) if op == "LDG"],
                       "first_compare": next((i for i, op in enumerate(part) if op in ("ISETP", "FSETP", "DSETP")),
                                             len(part))})
    regs = re.search(r"Used (\d+) registers", log)
    spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", log)
    return {"two_sets": two_sets, "pixels": (2 if two_sets else 1) * int(m_v.group(1)) * int(m_u.group(1)), "loop": loop, "ops": ops, "halves": halves,
            "registers": int(regs.group(1)) if regs else None,
            "spills": int(spill.group(1)) + int(spill.group(2)) if spill else None, "log": log, "text": text}


def report(name, src):
    a = analyse(src)
    ops, pixels = a["ops"], a["pixels"]
    mix = collections.Counter(ops).most_common()
    print("{}: {} instructions per {} pixels = {:.2f} per pixel; {} registers, spills {} bytes".format(
        name, len(ops), pixels, len(ops) / pixels, a["registers"], a["spills"]))
    for h, half in enumerate(a["halves"]):
        ldg = half["ldg"]
        print("  {}: LDG at {}; first compare at {}; all LDGs before it: {}".format(
            "half {} (next chunk's loads)".format(h) if a["two_sets"] else "chunk", ldg, half["first_compare"],
            bool(ldg) and max(ldg) < half["first_compare"]))
    print("  LDS {}, S2R {}".format(ops.count("LDS"), ops.count("S2R")))
    print("  mix: " + ", ".join("{} {}".format(c, op) for op, c in mix))
    return a["text"]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--shapes", default="cfg2,cfg1,reclass200")
    ap.add_argument("--dump", metavar="DIR", help="write <shape>[_baked].cu / .sass there")
    args = ap.parse_args()
    table = shapes()
    for shape in args.shapes.split(","):
        src, baked = generate(*table[shape])
        for label, text in ((shape + "_baked", baked), (shape, src)):
            listing = report(label, text)
            if args.dump:
                os.makedirs(args.dump, exist_ok=True)
                with open(os.path.join(args.dump, label + ".cu"), "w") as f:
                    f.write(text)
                with open(os.path.join(args.dump, label + ".sass"), "w") as f:
                    f.write(listing)


if __name__ == "__main__":
    main()
