"""Temporal kernels of this tree against another build of libgeokernels.so, alternated in one
process on the same inputs and the same stream.

Cases: sum, std and Cumulative sum over 64 frames of an odd 8191 x 8191 float32 plane (no whole
16-byte pixel groups, so the one-pixel-per-thread VEC = 1 forms), the int16 sum over 365 frames of
8192 x 8192 (16-byte loads), and the median of one 600-frame bin of a 2048 x 2048 int32 stack
(float64 working dtype, 1024 sort slots per pixel).  Every case is timed `--reps` times per build,
the builds alternating, so that the spread of one build's repetitions is the run-to-run noise
against which the difference between builds is read.  Outputs of the two builds are compared.

Usage: python tools/temporal_vec1_bench.py --baseline-lib OTHER/libgeokernels.so [--out FILE.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STATS = {"sum": 0, "median": 5, "std": 6}


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # the numbers are still worth printing
        return "unknown ({})".format(exc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3, help="calls per timed repetition")
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch

    from dask_geomodeling_b200 import _native

    new = _native.lib()
    base = ctypes.CDLL(os.path.abspath(args.baseline_lib))
    for name in ("gm_temporal_aggregate", "gm_temporal_cumulative"):
        getattr(base, name).restype = getattr(new, name).restype
        getattr(base, name).argtypes = getattr(new, name).argtypes
    stream = torch.cuda.Stream()  # a stream of its own: a null handle would leave each library on its own stream

    def device(t):
        return _native.DeviceArray(tuple(t.shape), str(t.dtype).replace("torch.", ""), ptr=t.data_ptr(), owner=t)

    def stack(shape, dtype, nodata, seed):
        gen = torch.Generator(device="cuda").manual_seed(seed)
        out = torch.empty(shape, dtype=dtype, device="cuda")
        for a in range(shape[0]):
            if dtype.is_floating_point:
                out[a].uniform_(0, 100, generator=gen)
            else:
                out[a].copy_(torch.randint(0, 1000, shape[1:], device="cuda", generator=gen, dtype=dtype))
            out[a][torch.rand(shape[1:], device="cuda", generator=gen) < 0.03] = nodata
        return out

    def case(src, nodata, out_dtype, stat, cumulative=False, calls=None):
        calls = calls or args.calls
        T = src.shape[0]
        offsets = np.array([0, T], np.int32)
        frames = np.arange(T, dtype=np.int32)
        holder, nd_ptr = _native.scalar_ptr(nodata, np.dtype(str(src.dtype).replace("torch.", "")))
        dst_shape = (T if cumulative else 1,) + tuple(src.shape[1:])
        dsts = {k: torch.empty(dst_shape, dtype=out_dtype, device="cuda") for k in ("base", "new")}
        gm_src = _native.as_gm_array(device(src))
        gm_dst = {k: _native.as_gm_array(device(v)) for k, v in dsts.items()}

        def call(which):
            lib = base if which == "base" else new
            if cumulative:
                rc = lib.gm_temporal_cumulative(ctypes.byref(gm_src), ctypes.byref(gm_dst[which]), nd_ptr, 1,
                                                STATS[stat], offsets.ctypes.data, frames.ctypes.data,
                                                frames.ctypes.data, 1, ctypes.c_void_p(stream.cuda_stream))
            else:
                rc = lib.gm_temporal_aggregate(ctypes.byref(gm_src), ctypes.byref(gm_dst[which]), nd_ptr, 1,
                                               STATS[stat], 0.0, offsets.ctypes.data, frames.ctypes.data, 1,
                                               ctypes.c_void_p(stream.cuda_stream))
            assert rc == 0, "{} build failed on {}".format(which, stat)

        times = {"base": [], "new": []}
        for which in ("base", "new"):
            call(which)  # warm-up: module load, shared-memory opt-in
        stream.synchronize()
        for _ in range(args.reps):
            for which in ("base", "new"):
                start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                start.record(stream)
                for _ in range(calls):
                    call(which)
                stop.record(stream)
                stop.synchronize()
                times[which].append(start.elapsed_time(stop) / calls)
        stream.synchronize()
        a, b = dsts["base"], dsts["new"]
        same = bool(torch.equal(a, b)) if not a.is_floating_point() else bool(
            ((a == b) | (torch.isnan(a) & torch.isnan(b))).all())
        del holder
        row = {"equal_outputs": same}
        for which, ts in times.items():
            med = float(np.median(ts))
            row[which] = {"ms_median": med, "ms_min": min(ts), "ms_max": max(ts),
                          "spread": (max(ts) - min(ts)) / med}
        row["new_over_base"] = row["new"]["ms_median"] / row["base"]["ms_median"]
        return row

    result = {"card (name, power limit)": card(), "reps": args.reps, "calls_per_rep": args.calls, "cases": {}}
    f32_max = float(np.finfo(np.float32).max)
    odd = stack((64, 8191, 8191), torch.float32, f32_max, 7)
    for stat in ("sum", "std"):
        result["cases"]["{}_64x8191^2_f4".format(stat)] = case(odd, f32_max, torch.float32, stat)
        print(json.dumps({stat: result["cases"]["{}_64x8191^2_f4".format(stat)]}), flush=True)
    result["cases"]["cumulative_sum_64x8191^2_f4"] = case(odd, f32_max, torch.float32, "sum", cumulative=True)
    print(json.dumps(result["cases"]["cumulative_sum_64x8191^2_f4"]), flush=True)
    del odd
    torch.cuda.empty_cache()
    i16 = stack((365, 8192, 8192), torch.int16, 32767, 8)
    result["cases"]["sum_365x8192^2_i2"] = case(i16, 32767, torch.int32, "sum")
    print(json.dumps(result["cases"]["sum_365x8192^2_i2"]), flush=True)
    del i16
    torch.cuda.empty_cache()
    i4 = stack((600, 2048, 2048), torch.int32, 2 ** 31 - 1, 9)
    result["cases"]["median_600x2048^2_i4_f8"] = case(i4, 2 ** 31 - 1, torch.float64, "median", calls=1)
    print(json.dumps(result["cases"]["median_600x2048^2_i4_f8"]), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
