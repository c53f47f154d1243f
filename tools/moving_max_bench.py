"""MovingMax by size on one GPU: gm_moving_max on a 16384^2 float32 / float64 output plus its
size//2 halo, resident in HBM (1.1 to 2.4 GB per source, beyond the 126 MB L2), 5 % no data.

Sizes 11 (the compile-time kernels, the anchor), 17 (radius 8: the tiled kernel for float32,
the chord kernel for float64) and 33, 65, 67, 101, 201, 401 and 1025 (the chord kernel).  Per
size: kernel time from CUDA events over back-to-back calls (warmed up, at least 0.5 s of calls),
Gpx/s, and the shared-memory load bound the kernel's design implies: the
shared-memory load wavefronts per pixel (one per warp-wide load of up to 128 bytes; an SM serves
one per clock) over 148 SMs at the card's maximum SM clock, with the fraction of it reached.

With --parent LIB (a libgeokernels.so built from an earlier commit): sizes 17, 33 and 65 run on
both libraries, alternating in this one process, three times each, and the outputs are compared.
With --tiled-vs-chord: every (dtype, size) up to radius 8 without a compile-time kernel runs on
the tiled and on the chord kernel (GM_MOVING_MAX_KERNEL=tiled / chord), alternating, on a 16384^2
output: the measurement behind the choice between the two in run_moving_max.

Prints one JSON line; the GPU name, power limit and maximum SM clock are read in the same run.

Usage: python tools/moving_max_bench.py [--parent LIB] [--tiled-vs-chord] [--side 16384] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SIZES = (11, 17, 33, 65, 67, 101, 201, 401, 1025)
OLD_VS_NEW = (17, 33, 65)
# moving_max_chord_kernel's tile (csrc/gm_stencil.cu: MMC_TX, MMC_GROUPS * MMC_ROWS)
CHORD_TX, CHORD_ROWS = 256, 32


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    line = out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else ""
    parts = [p.strip() for p in line.split(",")]
    if len(parts) != 3:
        raise RuntimeError("nvidia-smi gave no GPU description: " + repr(out.stdout + out.stderr))
    return {"name": parts[0], "power_limit": parts[1], "sm_clock_max": parts[2]}


def kernel_of(size, dtype):
    """The kernel gm_moving_max selects (csrc/gm_stencil.cu: try_moving_max_fixed, run_moving_max)."""
    if size <= 15 and dtype in ("u1", "i2", "i4", "f4", "f8"):
        return "moving_max_block_kernel" if np.dtype(dtype).itemsize == 4 else "moving_max_fixed_kernel"
    if size <= 17 and not (np.dtype(dtype).itemsize == 8 and size >= 15):   # radius <= 8, 8-byte cells < 7
        return "moving_max_tiled_kernel"
    return "moving_max_chord_kernel"


def wavefronts_per_pixel(size, itemsize):
    """Shared-memory load wavefronts per output pixel that the kernel's design implies."""
    r = size // 2
    per_warp_load = max(1, 32 * itemsize // 128)     # wavefronts of one warp-wide scalar load
    if size <= 15 and itemsize == 4:
        # moving_max_block_kernel: a thread owns 4 columns x 8 rows and reads (8 + 2r) rows of
        # NQ 16-byte quads (4 wavefronts per warp-wide LDS.128)
        nq = (4 + 2 * r + 3) // 4
        return (8 + 2 * r) * nq * 4 / (32 * 32)
    if size <= 15 or (size == 17 and itemsize < 8):
        # moving_max_fixed_kernel / moving_max_tiled_kernel: per tile row and column 2 wmax chord
        # loads, then 2r + 1 plane loads per pixel, over a 64 x 32 tile
        chord = (32 + 2 * r) / 32 * 2 * r
        return (chord + 2 * r + 1) / 32 * per_warp_load
    levels = int(np.floor(np.log2(2 * r + 1))) + 1
    staged = (CHORD_TX + 2 * r) * (CHORD_ROWS + 2 * r) / (CHORD_TX * CHORD_ROWS)
    loads = 2 * (2 * r + 1) + 2 * (levels - 1) * staged     # chords, then the table build
    return loads / 32 * per_warp_load


def timed(fn, min_seconds=0.5):
    import torch

    fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    iters = max(3, int(np.ceil(min_seconds * 1000 / max(start.elapsed_time(stop), 1e-3))))
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / iters


def parent_library(path):
    from dask_geomodeling_b200 import _native

    lib = ctypes.CDLL(os.path.abspath(path))
    for name in ("gm_init", "gm_last_error", "gm_moving_max"):
        restype, argtypes = _native.SYMBOLS[name]
        getattr(lib, name).restype = restype
        getattr(lib, name).argtypes = argtypes
    if lib.gm_init(0) != 0:
        raise RuntimeError(lib.gm_last_error().decode())
    return lib


ANCHOR_NOTE = ("size 11 float32 is moving_max_block_kernel on a window padded to a 16-byte row pitch "
               "(pitch_pad columns), the form MovingMax requests; README.md's 513 Gpx/s for the same kernel "
               "is bench.py's stencil leg at 32768^2")
# (dtype, size) up to radius 8 without a compile-time kernel: radius 1...8 for int8, uint16,
# uint32 and int64, radius 8 for the others
TILED_WORKLOADS = ([(d, s) for d in ("i1", "u2", "u4", "i8") for s in (3, 7, 11, 15, 17)] +
                   [(d, 17) for d in ("u1", "i2", "i4", "f4", "f8")])


def random_device(shape, dtype, seed):
    """Device values of `dtype` with 5 % no data (the dtype maximum); integer cells are random bytes."""
    import torch

    gen = torch.Generator(device="cuda").manual_seed(seed)
    d = np.dtype(dtype)
    if d.kind == "f":
        t = torch.randn(shape, dtype=torch.float32 if d.itemsize == 4 else torch.float64, device="cuda",
                        generator=gen) * 100
        t[torch.rand(shape, device="cuda", generator=gen) < 0.05] = float(np.finfo(d).max)
        return t
    count = int(np.prod(shape))
    t = torch.randint(0, 256, (count * d.itemsize,), dtype=torch.uint8, device="cuda", generator=gen)
    return t


def tiled_vs_chord(lib, call, n):
    """The tiled against the chord kernel (GM_MOVING_MAX_KERNEL), alternated twice per workload,
    with the outputs compared."""
    import torch
    from dask_geomodeling_b200 import _native

    rows = []
    for dtype, size in TILED_WORKLOADS:
        r = size // 2
        d = np.dtype(dtype)
        holder, nodata_ptr = _native.scalar_ptr(np.finfo(d).max if d.kind == "f" else np.iinfo(d).max, d)
        src_t = random_device((1, n + 2 * r, n + 2 * r), dtype, size)
        src = _native.DeviceArray((1, n + 2 * r, n + 2 * r), d, ptr=src_t.data_ptr(), owner=src_t)
        outs = [torch.empty(n * n * d.itemsize, dtype=torch.uint8, device="cuda") for _ in range(2)]
        dsts = [_native.DeviceArray((1, n, n), d, ptr=o.data_ptr(), owner=o) for o in outs]
        tiled, chord = [], []
        for _ in range(2):
            try:
                os.environ["GM_MOVING_MAX_KERNEL"] = "tiled"
                tiled.append(round(timed(lambda: call(lib, src, dsts[0], nodata_ptr, size), 0.3), 4))
                os.environ["GM_MOVING_MAX_KERNEL"] = "chord"
                chord.append(round(timed(lambda: call(lib, src, dsts[1], nodata_ptr, size), 0.3), 4))
            finally:
                del os.environ["GM_MOVING_MAX_KERNEL"]
        torch.cuda.synchronize()
        rows.append({"dtype": dtype, "size": size, "selected": kernel_of(size, dtype),
                     "tiled_ms": tiled, "chord_ms": chord, "identical_bytes": bool(torch.equal(*outs))})
        print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
        del src, src_t, dsts, outs
    return rows


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--side", type=int, default=16384)
    parser.add_argument("--parent", default=None, help="libgeokernels.so of an earlier commit")
    parser.add_argument("--sizes", default=",".join(str(s) for s in SIZES))
    parser.add_argument("--tiled-vs-chord", action="store_true",
                        help="time the tiled kernel against the chord kernel where the tiled one is selected")
    parser.add_argument("--out", default=None)
    args = parser.parse_args()

    import torch
    from dask_geomodeling_b200 import _native

    info = gpu_info()
    props = torch.cuda.get_device_properties(0)
    sms = props.multi_processor_count
    clock_ghz = float(info["sm_clock_max"].split()[0]) / 1000.0
    lib = _native.lib()
    parent = parent_library(args.parent) if args.parent else None
    side = torch.cuda.Stream()
    stream = side.cuda_stream
    n = args.side
    results = {"gpu": info, "sms": sms, "side": n, "rows": [], "old_vs_new": [], "tiled_vs_chord": [],
               "notes": ANCHOR_NOTE}

    def call(library, src, dst, nodata_ptr, size):
        rc = library.gm_moving_max(ctypes.byref(_native.as_gm_array(src)), ctypes.byref(_native.as_gm_array(dst)),
                                   nodata_ptr, 1, size, stream)
        if rc != 0:
            raise RuntimeError(library.gm_last_error().decode())

    with torch.cuda.stream(side):
        for dtype in ("f4", "f8"):
            tdtype = torch.float32 if dtype == "f4" else torch.float64
            nodata = float(np.finfo(dtype).max)
            holder, nodata_ptr = _native.scalar_ptr(nodata, dtype)
            dst_t = torch.empty((1, n, n), dtype=tdtype, device="cuda")
            dst = _native.DeviceArray((1, n, n), dtype, ptr=dst_t.data_ptr(), owner=dst_t)
            for size in (int(s) for s in args.sizes.split(",")):
                r = size // 2
                gen = torch.Generator(device="cuda").manual_seed(size)
                # float32 up to size 15: the window padded to a 16-byte row pitch, as
                # MovingMax.get_sources_and_requests asks its store for it (TMA tile staging)
                pad = (-(n + 2 * r)) % 4 if dtype == "f4" and size <= 15 else 0
                src_t = torch.randn((1, n + 2 * r, n + 2 * r + pad), dtype=tdtype, device="cuda",
                                    generator=gen) * 100
                src_t[torch.rand(src_t.shape, device="cuda", generator=gen) < 0.05] = nodata
                src = _native.DeviceArray(src_t.shape, dtype, ptr=src_t.data_ptr(), owner=src_t)
                ms = timed(lambda: call(lib, src, dst, nodata_ptr, size))
                itemsize = np.dtype(dtype).itemsize
                wf = wavefronts_per_pixel(size, itemsize)
                bound_ms = n * n * wf / (sms * clock_ghz * 1e9) * 1e3
                results["rows"].append({
                    "dtype": dtype, "size": size, "kernel": kernel_of(size, dtype), "pitch_pad": pad, "ms": round(ms, 4),
                    "gpx_s": round(n * n / ms / 1e6, 2), "ns_per_px_per_sm": round(ms * 1e6 * sms / (n * n), 4),
                    "smem_wavefronts_per_px": round(wf, 3), "smem_bound_ms": round(bound_ms, 4),
                    "fraction_of_bound": round(bound_ms / ms, 3)})
                print(json.dumps(results["rows"][-1]), file=sys.stderr, flush=True)
                if parent is not None and size in OLD_VS_NEW:
                    new, old = [], []
                    for _ in range(3):
                        new.append(round(timed(lambda: call(lib, src, dst, nodata_ptr, size)), 4))
                        old.append(round(timed(lambda: call(parent, src, dst, nodata_ptr, size)), 4))
                    ref_t = torch.empty_like(dst_t)
                    call(parent, src, _native.DeviceArray((1, n, n), dtype, ptr=ref_t.data_ptr(), owner=ref_t),
                         nodata_ptr, size)
                    call(lib, src, dst, nodata_ptr, size)
                    torch.cuda.synchronize()
                    identical = bool(torch.equal(dst_t.view(torch.int32 if dtype == "f4" else torch.int64),
                                                 ref_t.view(torch.int32 if dtype == "f4" else torch.int64)))
                    results["old_vs_new"].append({"dtype": dtype, "size": size, "new_ms": new, "old_ms": old,
                                                  "identical_bytes": identical})
                    print(json.dumps(results["old_vs_new"][-1]), file=sys.stderr, flush=True)
                del src, src_t
        if args.tiled_vs_chord:
            results["tiled_vs_chord"] = tiled_vs_chord(lib, call, n)
    line = json.dumps(results)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
