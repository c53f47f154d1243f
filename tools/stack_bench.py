"""Stacks on one GPU: gm_reduce_stack over N float32 8192^2 rasters (N = 4, 8, 16, 64; max, sum,
last) and one int16 stack, the evaluator's kernel (program compiled once) against gm_reduce_stack
at N = 8 (time and bytes), and
gm_place of a 256^2 float32 source at N = 8, 1 000 and 100 000 coordinates into 16384^2 (last,
max, sum), against the former copy-and-reduce path at N = 8.

With --stats: mean, var, std and argmax (gm_reduce_stack_stat) over N = 4, 16, 64 float32 8192^2
rasters next to sum (gm_reduce_stack) in the same run, and Place of the 256^2 source at 1 000
coordinates into 16384^2 for sum, mean and argmax (gm_place_stat).

Times are CUDA events around back-to-back calls on resident inputs (8192^2 float32 inputs are
268 MB each, beyond the 126 MB L2).  Algorithmic bytes: one read of every input cell and one write
of every output cell (var and std read their stack twice in the kernel, but need it once); for
Place one write of the output (the source stays in L2).  The share of HBM is taken against
6451.5 GB/s, the device-to-device copy rate measured on this project's B200 (DESIGN §3).  Prints
one JSON line; the GPU name and power limit are read in the same run.

Usage: python tools/stack_bench.py [--stats] [--iters 10] [--out FILE]
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

HBM_GBS = 6451.5


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def timed(fn, iters):
    import torch

    fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / iters


def main():
    parser = argparse.ArgumentParser()
    parser.add_argument("--iters", type=int, default=10)
    parser.add_argument("--size", type=int, default=8192)
    parser.add_argument("--place-size", type=int, default=16384)
    parser.add_argument("--stats", action="store_true", help="mean / var / std / argmax instead")
    parser.add_argument("--out", default=None)
    args = parser.parse_args()
    results = stats_bench(args) if args.stats else stack_bench(args)
    line = json.dumps(results)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


def device_stack(rng, n, size, dtype, nodata):
    from dask_geomodeling_b200 import _native

    out = []
    for k in range(n):
        if np.dtype(dtype).kind == "f":
            v = rng.standard_normal((1, size, size), dtype=np.float32).astype(dtype)
        else:
            v = rng.integers(-1000, 1000, (1, size, size)).astype(dtype)
        v[0, :: 7 + k % 5] = nodata
        out.append((_native.DeviceArray.from_host(v), nodata))
    return out


def rate(nbytes, ms):
    return {"ms": round(ms, 4), "gbs": round(nbytes / ms / 1e6, 1), "hbm_share": round(nbytes / ms / 1e6 / HBM_GBS, 3)}


def stats_bench(args):
    import torch
    from dask_geomodeling_b200 import _native, _state
    from dask_geomodeling_b200.raster import _program, spatial

    side = torch.cuda.Stream()
    results = {"gpu": gpu_info(), "hbm_gbs": HBM_GBS, "reduce": [], "place": []}
    size, rng = args.size, np.random.default_rng(0)
    with torch.cuda.stream(side), _native.use_stream(side.cuda_stream), _state.device_resident():
        f32 = device_stack(rng, 64, size, "f4", np.float32(-9999.0))
        for n in (4, 16, 64):
            stack = f32[:n]
            nbytes = (n + 1) * size * size * 4
            for statistic in ("sum", "mean", "var", "std", "argmax"):
                run = _program.run_stack if statistic == "sum" else _program.run_stack_stat
                ms = timed(lambda: run(statistic, stack, np.dtype("f4"), -9999.0, True), args.iters)
                results["reduce"].append(dict({"n": n, "dtype": "float32", "statistic": statistic},
                                              **rate(nbytes, ms)))
        del f32
        psize = args.place_size
        src = rng.uniform(1, 100, (1, 256, 256)).astype("f4")
        src[src < 10] = -9999.0
        payload = {"values": _native.DeviceArray.from_host(src), "no_data_value": -9999.0}
        coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(0, psize, 1000), rng.uniform(0, psize, 1000))]
        for statistic in ("sum", "mean", "argmax"):
            kwargs = {"mode": "warp", "anchor": (0.0, 256.0), "coordinates": coordinates,
                      "src_bbox": (0.0, 0.0, 256.0, 256.0), "dst_bbox": (0.0, 0.0, float(psize), float(psize)),
                      "cellsize": (1.0, 1.0), "statistic": statistic}
            ms = timed(lambda: spatial.Place.process(kwargs, payload), max(2, args.iters // 2))
            results["place"].append(dict({"n": 1000, "statistic": statistic}, **rate(psize * psize * 4, ms)))
    return results


def stack_bench(args):

    import torch
    from dask_geomodeling_b200 import _native, _state
    from dask_geomodeling_b200.raster import _program, spatial
    from dask_geomodeling_b200.raster.reduction import reduce_rasters

    lib = _native.lib()
    # a stream of its own: the library's calls and the timing events must share one stream
    side = torch.cuda.Stream()
    results = {"gpu": gpu_info(), "hbm_gbs": HBM_GBS, "reduce": [], "place": []}
    size = args.size
    rng = np.random.default_rng(0)

    with torch.cuda.stream(side), _native.use_stream(side.cuda_stream), _state.device_resident():
        f32 = device_stack(rng, 64, size, "f4", np.float32(-9999.0))
        for n in (4, 8, 16, 64):
            for statistic in ("max", "sum", "last"):
                stack = f32[:n]
                ms = timed(lambda: _program.run_stack(statistic, stack, np.dtype("f4"), -9999.0, True), args.iters)
                nbytes = (n + 1) * size * size * 4
                row = {"n": n, "dtype": "float32", "statistic": statistic, "ms": round(ms, 4),
                       "gbs": round(nbytes / ms / 1e6, 1), "hbm_share": round(nbytes / ms / 1e6 / HBM_GBS, 3)}
                if n == 8:
                    # the evaluator's kernel alone: the program compiled once, launched on the same inputs
                    node = _program.Node("reduce", [_program.Leaf(i) for i in range(n)], statistic=statistic,
                                         dtype="float32", fillvalue=-9999.0)
                    compiled = _program.CompiledProgram([node], [(np.dtype("f4"), nd) for _, nd in stack])
                    evaluated = _native.DeviceArray((1, size, size), "f4")
                    inputs = [v for v, _ in stack]
                    ev_ms = timed(lambda: compiled.launch(inputs, [evaluated]), args.iters)
                    b = _program.run_stack(statistic, stack, np.dtype("f4"), -9999.0, True).to_host()
                    row.update(evaluator_ms=round(ev_ms, 4),
                               identical_bytes=evaluated.to_host().tobytes() == b.tobytes())
                results["reduce"].append(row)
        del f32
        i16 = device_stack(rng, 16, size, "i2", -32768)
        ms = timed(lambda: _program.run_stack("max", i16, np.dtype("i2"), -32768, True), args.iters)
        nbytes = 17 * size * size * 2
        results["reduce"].append({"n": 16, "dtype": "int16", "statistic": "max", "ms": round(ms, 4),
                                  "gbs": round(nbytes / ms / 1e6, 1),
                                  "hbm_share": round(nbytes / ms / 1e6 / HBM_GBS, 3)})
        del i16

        psize = args.place_size
        src = rng.uniform(1, 100, (1, 256, 256)).astype("f4")
        src[src < 10] = -9999.0
        payload = {"values": _native.DeviceArray.from_host(src), "no_data_value": -9999.0}
        for n in (8, 1000, 100000):
            coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(0, psize, n), rng.uniform(0, psize, n))]
            for statistic in ("last", "max", "sum"):
                kwargs = {"mode": "warp", "anchor": (0.0, 256.0), "coordinates": coordinates,
                          "src_bbox": (0.0, 0.0, 256.0, 256.0), "dst_bbox": (0.0, 0.0, float(psize), float(psize)),
                          "cellsize": (1.0, 1.0), "statistic": statistic}
                ms = timed(lambda: spatial.Place.process(kwargs, payload), max(2, args.iters // 2))
                nbytes = psize * psize * 4
                row = {"n": n, "statistic": statistic, "ms": round(ms, 4), "gbs": round(nbytes / ms / 1e6, 1),
                       "hbm_share": round(nbytes / ms / 1e6 / HBM_GBS, 3)}
                if n == 8:
                    old_ms = timed(lambda: old_place(_native, lib, reduce_rasters, src, payload, kwargs),
                                   max(2, args.iters // 2))
                    a = spatial.Place.process(kwargs, payload)["values"].to_host()
                    b = old_place(_native, lib, reduce_rasters, src, payload, kwargs)["values"].to_host()
                    row.update(old_ms=round(old_ms, 4), identical_bytes=a.tobytes() == b.tobytes())
                results["place"].append(row)
    return results


def old_place(_native, lib, reduce_rasters, src, payload, kwargs):
    """The former warp mode: one request-sized gm_resample_nn copy per coordinate, then
    reduce_rasters over the copies."""
    psize = round(kwargs["dst_bbox"][2])
    holder, nodata_ptr = _native.scalar_ptr(-9999.0, src.dtype)
    stack = []
    for cx, cy in kwargs["coordinates"]:
        di, dj = round(cx), psize - 256 - round(cy - 256.0)
        if di <= -256 or di >= psize or dj <= -256 or dj >= psize:
            continue
        placed = _native.DeviceArray((1, psize, psize), src.dtype)
        _native.check(lib.gm_resample_nn(ctypes.byref(_native.as_gm_array(payload["values"])),
                                         ctypes.byref(_native.as_gm_array(placed)), nodata_ptr,
                                         float(-di), 1.0, float(-dj), 1.0, _native.current_stream()))
        stack.append({"values": placed, "no_data_value": -9999.0})
    return reduce_rasters(stack, kwargs["statistic"])


if __name__ == "__main__":
    main()
