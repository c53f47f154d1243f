"""Reprojection throughput on one GPU: a 16384^2 float32 request in EPSG:3857 from a resident
16384^2 source in EPSG:4326 (separable warp) and from one in UTM zone 31N (per-cell transverse
Mercator), plus the same requests through ``get_data``.

Reports, per case: gm_warp_nn time from CUDA events over back-to-back calls, Gpx/s, the algorithmic
bytes (one read + one write of the itemsize per cell and band) over time as a fraction of the HBM
bandwidth measured by a device-to-device copy in the same run, and ``get_data`` end to end (the
result copied back to host memory).  For the UTM kernel it also counts the FP64 instructions in its
SASS.  Prints one JSON line; the GPU name and power limit are read in the same run.

Usage: python tools/reproject_bench.py [--size 16384] [--iters 20] [--out FILE]
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def fp64_sass_count(kernel_pattern="warp_cells_kernelIfE"):
    """FP64 instructions in the SASS of the float32 per-cell warp kernel (static count: every
    instruction of the kernel, including the rarely taken slow paths of the libm functions)."""
    from dask_geomodeling_b200 import _native

    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        return None
    sass = subprocess.run([tool, "-sass", _native.LIB_PATH], capture_output=True, text=True).stdout
    counts, inside = {}, False
    for line in sass.splitlines():
        if "Function :" in line:
            inside = kernel_pattern in line
            continue
        if inside:
            m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9]*)", line)
            if m and m.group(1) in ("DADD", "DMUL", "DFMA", "DSETP", "DMNMX", "F2F", "DRCP", "MUFU",
                                    "F2I", "I2F", "DSQRT"):
                op = m.group(1)
                if op in ("F2F", "F2I", "I2F", "MUFU") and ".F64" not in line:
                    continue
                counts[op] = counts.get(op, 0) + 1
    return {"total": sum(counts.values()), "by_opcode": counts}


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--size", type=int, default=16384)
    parser.add_argument("--iters", type=int, default=20)
    parser.add_argument("--out", default=None)
    args = parser.parse_args()

    import torch

    from dask_geomodeling_b200 import _native, utils
    from dask_geomodeling_b200._compat import config
    from dask_geomodeling_b200.raster import MemorySource, sources

    if not torch.cuda.is_available():
        raise SystemExit("reproject_bench needs a CUDA device")
    n = args.size
    # a stream of our own: torch's default stream has handle 0, which the library reads as "its
    # own stream", and events recorded on it would then not bracket the warp
    stream = torch.cuda.Stream()
    result = {"gpu": gpu_info(), "size": n, "dtype": "float32", "iters": args.iters}

    # HBM bandwidth of a 2 GiB device-to-device copy (read + write), same run
    a = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(10):
        b.copy_(a)
    stop.record()
    torch.cuda.synchronize()
    hbm = 2 * a.numel() * 4 * 10 / (start.elapsed_time(stop) / 1e3)
    result["measured_hbm_GBps"] = round(hbm / 1e9, 1)
    del a, b

    rng = np.random.default_rng(0)
    data = rng.random((1, n, n), dtype=np.float32)
    request_box = (1.2, 40.2, 4.8, 43.8)
    bbox = utils.Extent(request_box, "EPSG:4326").transformed("EPSG:3857").bbox
    cases = {}
    with config.set({"geomodeling.device-cache-bytes": 8 << 30}), torch.cuda.stream(stream), \
            _native.use_stream(stream.cuda_stream):
        for name, projection in (("4326_to_3857", "EPSG:4326"), ("utm31n_to_3857", "EPSG:32631")):
            x1, y1, x2, y2 = utils.Extent((1.0, 40.0, 5.0, 44.0), "EPSG:4326").transformed(projection).bbox
            source = MemorySource(data, -1.0, projection, pixel_size=((x2 - x1) / n, (y2 - y1) / n),
                                  pixel_origin=(x1, y2))
            resident = sources.resident_copy(source.data)
            gt = tuple(source.geo_transform)

            def call():
                return sources._warp_call(resident, (0, 0), (n, n), gt, projection, -1.0, bbox, n, n,
                                          "EPSG:3857", count_misses=False)[0]

            for _ in range(3):
                out = call()
            torch.cuda.synchronize()
            start.record(stream)
            for _ in range(args.iters):
                out = call()
            stop.record(stream)
            torch.cuda.synchronize()
            seconds = start.elapsed_time(stop) / 1e3 / args.iters
            cells = n * n
            algorithmic = 2 * cells * 4
            request = dict(mode="vals", projection="EPSG:3857", bbox=bbox, width=n, height=n)
            source.get_data(**request)
            torch.cuda.synchronize()
            e2e = []
            for _ in range(3):
                t0 = time.perf_counter()
                values = source.get_data(**request)["values"]
                torch.cuda.synchronize()
                e2e.append(time.perf_counter() - t0)
            assert values.shape == (1, n, n)
            cases[name] = {
                "kernel_ms": round(seconds * 1e3, 3),
                "gpx_per_s": round(cells / seconds / 1e9, 2),
                "algorithmic_GBps": round(algorithmic / seconds / 1e9, 1),
                "fraction_of_measured_hbm": round(algorithmic / seconds / hbm, 3),
                "get_data_ms_median": round(sorted(e2e)[1] * 1e3, 1),
                "no_data_cells": int(np.count_nonzero(np.asarray(values) == -1.0)),
            }
            del out, values
    sass = fp64_sass_count()
    if sass is not None:
        cases["utm31n_to_3857"]["fp64_sass_instructions_static"] = sass
    result["cases"] = cases
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
