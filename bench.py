"""Benchmark of the per-tile raster compute path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--legs chain,zonal,...]

Headline workload at every N: BASELINE.json configs[1] -- Reclassify + Clip + Step + IsData on a
16384 x 16384 int16 / float32 MemorySource pair -- one such raster pair per GPU (weak scaling, no
data-path collective: pixels are independent).  A step is one pass of the fused chain.

  value     Gpixel/s with the inputs resident in HBM (CUDA events around K launches)
  e2e       the same metric through ``view.get_data(**request)`` with host NumPy inputs: pinned
            H2D of both rasters and D2H of the result in every step
  roofline  algorithmic bytes (2 + 4 in, 1 out = 7 B/px) / measured kernel time against
            MEASURED_PEAKS.json hbm_gbs; ``traffic`` = DRAM bytes per launch from the ncu capture
            listed in profiles/r02_dram_traffic.json (null when there is none for this size)
  cpu_baseline  the reference's CPU path for the same chain on the box's host cores (the real
            reference ``process`` functions when the reference checkout exists, else the oracle
            port), whole 16384 x 16384 request in 2048 x 2048 tiles on a thread pool

The other configurations of BASELINE.json are ``striped`` legs of the same JSON line -- ONE
workload sharded in row stripes over the N ranks (strong scaling; at N = 1 the single-GPU path):

  stencils  configs[2]: Smooth(5) / MovingMax(11) / HillShade on ONE 32768 x 32768 DEM, halo
            exchange (ncclSend/Recv) + kernel per step
  zonal     configs[3]: AggregateRaster mean / max / p90 of ~100 k polygons over ONE
            40000 x 40000 raster: stripe partials + all-reduce, order statistics by stripe owners
  temporal  configs[4]: TemporalAggregate sum / max over ONE 365 x 8192 x 8192 stack sharded by
            rows (no collective); at N = 1 also Cumulative, std and median on the first 64 frames

Each striped entry carries its own ``roofline`` (algorithmic bytes / time against N x the measured
HBM peak) and, at N > 1, ``single_gpu_ms`` (the same operation on the whole workload, measured on
rank 0 in the same run) and the speed-up over it.

``--impl reference`` times the CPU arm alone and prints the same JSON line with
``"impl": "reference"``.

``--dump-outputs DIR`` writes, on rank 0, what each timed GPU call returned in its last step as
``DIR/<leg>_<op>.npy`` (float32, float64 where float32 would not hold the values), so that two
builds can be compared output for output on the same seeded inputs: the whole array up to
DUMP_CELLS cells, else DUMP_CELLS cells at fixed, seeded positions of the flattened array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fused raster chain throughput (Reclassify+Clip+Step+IsData)"
UNIT = "Gpixel/s"
BYTES_PER_PIXEL = 7  # int16 + float32 in, bool out
ALL_LEGS = "chain,stencils,zonal,temporal"
DUMP_CELLS = 1 << 19        # per output: 2 MB as float32; the 17 outputs of all legs stay under DUMP_BYTES
DUMP_BYTES = 64 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=16384, help="raster edge of the chain (cfg2)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--legs", default=ALL_LEGS, help="comma list of chain,stencils,zonal,temporal")
    ap.add_argument("--dem-size", type=int, default=32768, help="raster edge of the stencil leg (cfg3)")
    ap.add_argument("--zonal-size", type=int, default=40000, help="raster edge of the zonal leg (cfg4)")
    ap.add_argument("--zonal-grid", type=int, default=316, help="polygons per side of the zonal leg")
    ap.add_argument("--temporal-frames", type=int, default=365)
    ap.add_argument("--temporal-size", type=int, default=8192)
    ap.add_argument("--leg-steps", type=int, default=10, help="timed calls per striped operation")
    ap.add_argument("--no-zonal", action="store_true", help="(kept for old command lines) skip the zonal leg")
    ap.add_argument("--no-single", action="store_true", help="skip the single-GPU reference runs at N > 1")
    ap.add_argument("--profile", action="store_true",
                    help="kernel-resident chain loop only (for ncu): no e2e, no CPU baseline, no other legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last step's output of every timed GPU call as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.leg_steps < 1 or args.e2e_steps < 1:
        ap.error("--steps, --leg-steps and --e2e-steps must be at least 1")
    args.legs = [x for x in args.legs.split(",") if x]
    if args.no_zonal and "zonal" in args.legs:
        args.legs.remove("zonal")
    if args.profile:
        args.legs = ["chain"]
    return args


# ----------------------------------------------------------------------------
# CPU arm (reference process functions or their oracle port, threaded over tiles)
# ----------------------------------------------------------------------------


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from dask_geomodeling_b200 import workloads
    from oracle import reference_chain

    size = args.size
    ints, floats = workloads.cfg2_arrays(size, seed=43)
    times, kind, threads, checksum = reference_chain.time_chain(
        ints, floats, workloads.CFG2_PAIRS, steps=args.steps, warmup=args.warmup)
    ms = 1e3 * sum(times) / len(times)
    value = size * size / (ms / 1e3) / 1e9
    sample = "whole {0}x{0} request per step, {1} tiles of 2048 x 2048 on {2} threads".format(
        size, len(reference_chain.tiles(size, size)), threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int16/float32->bool", "data": "synthetic",
        "config": {"workload": "cfg2 Reclassify+Clip+Step+IsData {0}x{0} int16/float32".format(size),
                   "same_config": True, "checksum_true_pixels": checksum},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if "zonal" in args.legs:
        gpx, seconds, zthreads, zkind = reference_chain.time_zonal()
        line["zonal"] = {"mean": {"value": gpx, "unit": UNIT}, "cores": zthreads, "kind": zkind,
                         "sample": "mean of 1024 polygons over 4096 x 4096 float32 (cfg4 scaled), "
                                   "{:.1f} s".format(seconds)}
    print(json.dumps(line))


# ----------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------


class NvmlSampler(object):
    """SM clock and throttle reasons sampled through NVML while the timed region runs."""

    def __init__(self, index, period=0.0005):
        import pynvml

        self.nvml = pynvml
        pynvml.nvmlInit()
        self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        self.period = period
        # the first queries of a process take tens to hundreds of milliseconds on a fresh box
        # (a 1000-step run once ended with ONE sample): pay that here, before the thread starts
        for _ in range(2):
            pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            try:
                pynvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        self.sm, self.reasons = [], set()
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        n = self.nvml
        flags = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "sw_power_cap": 0x4}
        while self.running:
            try:
                self.sm.append(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for name, bit in flags.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def mark(self):
        """The timed region starts here (samples before it were taken under the warm-up load)."""
        self.marked = len(self.sm)

    def stop(self):
        self.running = False
        self.thread.join(timeout=2)
        try:
            sm_max = self.nvml.nvmlDeviceGetMaxClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)
        except Exception:
            sm_max = None
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "samples_in_timed_region": len(self.sm) - getattr(self, "marked", 0), "source": "nvml"}


class SmiSampler(object):
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.samples = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def mark(self):
        self.marked = len(self.samples)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, sm_max, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.samples:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                sm_max = float(parts[1])
            except ValueError:
                continue
            for name, flag in zip(names, parts[2:6]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": sm_max,
                "reasons": sorted(reasons), "samples": len(sm),
                "samples_in_timed_region": len(self.samples) - getattr(self, "marked", 0), "source": "nvidia-smi"}


def make_sampler(index):
    try:
        return NvmlSampler(index)
    except Exception:
        return SmiSampler(index)


# ----------------------------------------------------------------------------
# helpers of the GPU arm
# ----------------------------------------------------------------------------


def bind_to_gpu_numa_node(local_rank, ranks_on_box):
    """Pin this rank to the host cores of its GPU's NUMA node (and thereby, by first touch, its
    host rasters and pinned staging to that node's memory): with every rank on node 0 the
    end-to-end leg at 8 GPUs was bound by one socket's memory and PCIe root (VERDICT r1).  The
    node's cores are divided among the ranks that share it.  Best effort: returns what was done."""
    info = {"numa_node": None, "cpus": None}
    try:
        import pynvml

        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(handle).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/{}/numa_node".format(bus)).read())
        allowed = sorted(os.sched_getaffinity(0))
        info["allowed_cpus"] = len(allowed)
        if node < 0:
            return info
        cpus = []
        for part in open("/sys/devices/system/node/node{}/cpulist".format(node)).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        cpus = [c for c in cpus if c in set(allowed)]
        info["numa_node"] = node
        if not cpus:
            return info
        # ranks on the same node (GPU order = rank order on one box) share its cores evenly
        same = [r for r in range(ranks_on_box) if _gpu_node(pynvml, r) == node]
        if local_rank in same and len(cpus) >= len(same):
            k = same.index(local_rank)
            per = len(cpus) // len(same)
            cpus = cpus[k * per:(k + 1) * per]
        os.sched_setaffinity(0, cpus)
        info["cpus"] = "{}-{} ({})".format(cpus[0], cpus[-1], len(cpus))
    except Exception as e:  # no NVML / sysfs: leave the affinity alone
        info["error"] = str(e)[:80]
    return info


def _gpu_node(pynvml, index):
    try:
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        return int(open("/sys/bus/pci/devices/{}/numa_node".format(bus)).read())
    except Exception:
        return -1


class Context(object):
    """What every leg needs: torch, the process group, the stream all kernels, collectives and
    CUDA events share, the roofline denominators."""

    def __init__(self, args, torch, dist, rank, local_rank, world):
        self.args, self.torch, self.dist = args, torch, dist
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            self.peak, self.peak_kind = json.load(open(peaks_path))["hbm_gbs"], "measured"
        else:
            self.peak, self.peak_kind = 6650.0, "fallback"
        self.traffic = {}
        path = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
        if os.path.exists(path):
            self.traffic = json.load(open(path))
        # a group of rank 0 alone: the single-GPU reference runs of the striped legs
        self.solo = dist.new_group([0]) if world > 1 else None
        self.outputs = {} if args.dump_outputs and rank == 0 else None

    def keep(self, name, result):
        """--dump-outputs: a sample of the arrays a timed call returned (see DUMP_CELLS)."""
        if self.outputs is None:
            return
        if isinstance(result, tuple):       # zonal_striped: (per-polygon values, polygons without cells)
            result = result[0]
        if isinstance(result, dict):        # a block's payload
            result = result["values"]
        self.outputs[name] = output_sample(self.torch, result, zlib.crc32(name.encode()))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def time_calls(self, fn, iters, warm=3, everyone=True):
        """ms per call of fn(): CUDA events on the launching stream, max over ranks."""
        from dask_geomodeling_b200 import _native

        torch = self.torch
        with _native.use_stream(self.stream.cuda_stream):
            for _ in range(warm):
                out = fn()
            if everyone:
                self.barrier()
            else:
                torch.cuda.synchronize()
            before = _native.launch_count()
            start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record(self.stream)
            for _ in range(iters):
                out = fn()
            stop.record(self.stream)
            torch.cuda.synchronize()
            launches = (_native.launch_count() - before) / float(iters)
        t = torch.tensor([start.elapsed_time(stop) / iters], dtype=torch.float64, device="cuda")
        if everyone and self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]), launches, out

    def roofline(self, nbytes, ms, kernel, n_gpus=None, traffic_key=None):
        n_gpus = n_gpus or self.world
        achieved = nbytes / ms / 1e6
        entry = self.traffic.get(traffic_key or kernel, {})
        return {"bound": "hbm", "achieved": achieved, "peak": self.peak * n_gpus, "unit": "GB/s",
                "frac": achieved / (self.peak * n_gpus), "traffic": entry.get("dram_bytes_per_launch"),
                "traffic_source": entry.get("source"), "peak_kind": self.peak_kind, "kernel": kernel,
                "algorithmic_bytes": nbytes}


def wrap(t):
    """torch CUDA tensor -> DeviceArray sharing its memory."""
    from dask_geomodeling_b200 import _native

    return _native.DeviceArray(tuple(t.shape), str(t.dtype).replace("torch.", ""), ptr=t.data_ptr(), owner=t)


class _CudaArrayView(object):
    """A DeviceArray as a torch CUDA tensor sharing its memory (``torch.as_tensor``)."""

    def __init__(self, array):
        self.__cuda_array_interface__ = {"shape": array.shape, "typestr": array.dtype.str,
                                         "data": (array.ptr, False), "version": 2}
        self.array = array


def output_sample(torch, values, seed):
    """Host copy of one output (DeviceArray, torch tensor or NumPy array): the whole array up to
    DUMP_CELLS cells, else DUMP_CELLS cells at `seed`-determined flat positions, gathered on the
    device; float32, or float64 where float32 would not hold every value."""
    from dask_geomodeling_b200 import _native

    if isinstance(values, _native.DeviceArray):
        values = torch.as_tensor(_CudaArrayView(values), device="cuda")
    elif not torch.is_tensor(values):
        values = torch.from_numpy(np.ascontiguousarray(values))
    shape = tuple(values.shape)
    values = values.reshape(-1)
    if values.numel() > DUMP_CELLS:
        index = np.sort(np.random.default_rng(seed).integers(0, values.numel(), DUMP_CELLS))
        values = values[torch.from_numpy(index).to(values.device)]
        shape = (DUMP_CELLS,)
    host = values.cpu().numpy().reshape(shape)
    exact32 = host.dtype.itemsize <= 2 or host.dtype == np.float32
    return host.astype(np.float32 if exact32 else np.float64)


def write_outputs(directory, outputs):
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_BYTES:
        raise RuntimeError("{} bytes of outputs exceed the dump limit of {}".format(total, DUMP_BYTES))
    os.makedirs(directory, exist_ok=True)
    for name, array in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), array)


def striped_entry(ctx, name, fn_striped, fn_single, pixels, nbytes, kernel, iters, traffic_key=None):
    """Time one operation on the sharded workload (all ranks) and, at N > 1, on the whole
    workload on rank 0 alone; returns the JSON object of the entry.  `name` is <leg>_<op>."""
    ms, launches, out = ctx.time_calls(fn_striped, iters)
    ctx.keep(name, out)
    entry = {"ms": ms, "gpx_s": pixels / ms / 1e6, "gpu_launches_per_call": launches,
             "roofline": ctx.roofline(nbytes, ms, kernel, traffic_key=traffic_key)}
    if ctx.world > 1 and not ctx.args.no_single:      # (every rank takes this branch: broadcast below)
        single = ctx.torch.zeros(1, dtype=ctx.torch.float64, device="cuda")
        if ctx.rank == 0 and fn_single is not None:
            single[0], _, _ = ctx.time_calls(fn_single, max(3, iters // 2), everyone=False)
        ctx.dist.broadcast(single, 0)
        entry["single_gpu_ms"] = float(single[0])
        entry["speedup_vs_1gpu"] = float(single[0]) / ms
    return entry


# ----------------------------------------------------------------------------
# configs[2]: stencils on ONE DEM in row stripes
# ----------------------------------------------------------------------------


def make_dem(torch, r0, r1, n, seed, nodata):
    """Rows [r0, r1) of the synthetic DEM: smooth terrain + noise, 1 % no data."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty((1, r1 - r0, n), dtype=torch.float32, device="cuda")
    x = torch.arange(n, device="cuda", dtype=torch.float32)[None, :]
    rows = max(1, (1 << 26) // n)
    for a in range(r0, r1, rows):     # chunked: bounded temporaries next to a 4 GB raster
        b = min(a + rows, r1)
        y = torch.arange(a, b, device="cuda", dtype=torch.float32)[:, None]
        z = 50 * torch.sin(x / 17.0) + 30 * torch.cos(y / 11.0) + 0.05 * x + 100
        z += torch.randn(b - a, n, device="cuda", generator=gen)
        z[torch.rand(b - a, n, device="cuda", generator=gen) < 0.01] = nodata
        out[0, a - r0:b - r0] = z
    return out


def run_stencils(ctx):
    from dask_geomodeling_b200 import parallel, raster, workloads

    torch, args = ctx.torch, ctx.args
    n = args.dem_size
    nodata = workloads.F32_MAX
    lw = parallel.smooth_halo(5.0)
    ops = [
        ("smooth", "Smooth(size=5.0), exact mode", lw, 5, raster.Smooth.process,
         (dict(smooth_mode="exact", fill=0, size=[5.0, 5.0], margin=(lw, 5)),), 8, "smooth_fast_kernel"),
        ("movingmax", "MovingMax(size=11)", 5, 5, raster.MovingMax.process, (11,), 8, "moving_max_block_kernel"),
        ("hillshade", "HillShade(altitude=45, azimuth=315)", 1, 1, raster.HillShade.process,
         (dict(resolution=(1.0, 1.0), altitude=45.0, azimuth=315.0, fill=0),), 5, "hillshade_quad_kernel"),
    ]
    out = {"workload": "cfg3 ONE {0}x{0} float32 DEM in {1} row stripe(s), halo exchange + kernel per step".format(
        n, ctx.world), "unit": UNIT, "steps": args.leg_steps}
    r0, r1 = parallel.stripe_rows(n, ctx.world)[ctx.rank]
    dem = make_dem(torch, r0, r1, n, 100 + ctx.rank, nodata)
    whole = None
    if ctx.world > 1 and ctx.rank == 0 and not args.no_single:
        whole = make_dem(torch, 0, n, n, 99, nodata)
    px = n * n
    for name, label, halo_rows, halo_cols, process, extra, bpp, kernel in ops:
        pitch = 4 if name in ("movingmax", "hillshade") else 1     # 16-byte row pitch: TMA tiles / quad loads
        stored = parallel.pad_columns(parallel.exchange_halo(dem, halo_rows, nodata), halo_cols, nodata, pitch)
        if name == "movingmax":
            extra = extra + (stored.shape[2] - (n + 2 * halo_cols),)
        if name == "hillshade":
            extra = (dict(extra[0], pad=stored.shape[2] - (n + 2 * halo_cols)),)
        stored_whole = None
        if whole is not None:
            stored_whole = parallel.pad_columns(
                parallel.exchange_halo(whole, halo_rows, nodata, group=ctx.solo), halo_cols, nodata, pitch)
        entry = striped_entry(
            ctx, "stencils_" + name,
            lambda: parallel.stencil_haloed(process, stored, nodata, halo_rows, halo_cols, *extra),
            None if stored_whole is None else (lambda: parallel.stencil_haloed(
                process, stored_whole, nodata, halo_rows, halo_cols, *extra, group=ctx.solo)),
            px, px * bpp, kernel, args.leg_steps)
        entry["op"] = label
        entry["halo_rows"] = halo_rows
        entry["bytes_per_pixel"] = bpp
        out[name] = entry
        del stored, stored_whole
    del dem, whole
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------
# configs[3]: zonal statistics of ONE raster in row stripes
# ----------------------------------------------------------------------------


def make_uniform(torch, shape, seed, nodata, fraction):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty(shape, dtype=torch.float32, device="cuda")
    flat = out.view(-1, shape[-1])
    rows = max(1, (1 << 27) // shape[-1])
    for a in range(0, flat.shape[0], rows):
        block = flat[a:a + rows]
        block.uniform_(0, 100, generator=gen)
        block[torch.rand(block.shape, device="cuda", generator=gen) < fraction] = nodata
    return out


def run_zonal(ctx, host_raster):
    from dask_geomodeling_b200 import _native, parallel, utils, workloads
    from dask_geomodeling_b200.core import fusion

    torch, args = ctx.torch, ctx.args
    n, g = args.zonal_size, args.zonal_grid
    nodata = workloads.F32_MAX
    rings = workloads.cfg4_rings(n, g, seed=7)          # the same polygons on every rank
    areas = workloads.ring_areas(rings)
    soup = utils.PolygonSoup([utils.Polygon(r) for r in rings]).to_device()
    bbox = (0, 0, n, n)
    r0, r1 = parallel.stripe_rows(n, ctx.world)[ctx.rank]
    stripe = make_uniform(torch, (1, r1 - r0, n), 200 + ctx.rank, nodata, 0.02)
    whole = None
    if ctx.world > 1 and ctx.rank == 0 and not args.no_single:
        whole = make_uniform(torch, (1, n, n), 199, nodata, 0.02)
    out = {"workload": "cfg4 AggregateRaster over ONE {0}x{0} float32 raster in {1} row stripe(s), {2} polygons".format(
        n, ctx.world, soup.n_polygons), "unit": UNIT, "bytes_per_pixel": 4, "steps": args.leg_steps,
        "polygons": {"count": soup.n_polygons, "mean_area_px": float(areas.mean()),
                     "area_fraction_of_raster": float(areas.sum() / (float(n) * n)),
                     "vertices": "6-12 per polygon, jittered cell boundaries, 5 % overlapping their neighbours",
                     "definition": "SURVEY.md section 8(d); dask_geomodeling_b200/workloads.py cfg4_rings"},
        "timed": "zonal_striped call: stripe kernels + collectives + download of the per-polygon results"}
    px = n * n
    kernels = {"mean": "zonal_reduce_warp_kernel<float, SUM>", "max": "zonal_reduce_warp_kernel<float, MAX>",
               "p90": "zonal_select_bracket/main/final_kernel<float>"}
    checks = {}
    with fusion.device_resident():
        for label, stat, q in (("mean", "mean", None), ("max", "max", None), ("p90", "percentile", 90.0)):
            def striped(stat=stat, q=q):
                return parallel.zonal_striped(soup, stripe, nodata, bbox, n, (r0, r1), stat, q)

            single = None
            if whole is not None:
                def single(stat=stat, q=q):
                    return parallel.zonal_striped(soup, whole, nodata, bbox, n, (0, n), stat, q, group=ctx.solo)
            entry = striped_entry(ctx, "zonal_" + label, striped, single, px, px * 4, kernels[label], args.leg_steps,
                                  traffic_key="zonal_" + label)
            with _native.use_stream(ctx.stream.cuda_stream):
                res, no_cells = striped()
            entry["checksum"] = float(np.nansum(np.asarray(res, dtype=np.float64)))
            entry["polygons_without_cells"] = len(no_cells)
            out[label] = entry
            checks[label] = res
    # size-independent property on the full result: min <= p90 <= max is implied by mean <= max etc.
    ok = np.asarray(checks["mean"]) <= np.asarray(checks["max"])
    out["property_mean_le_max"] = bool(np.all(ok | np.isnan(checks["mean"])))
    del stripe, whole
    torch.cuda.empty_cache()

    if ctx.world == 1 and host_raster is not None:
        out["e2e"] = zonal_e2e(ctx, host_raster)
        from oracle import reference_chain

        gpx, seconds, threads, kind = reference_chain.time_zonal()
        out["cpu_baseline"] = {"value": gpx, "unit": UNIT, "cores": threads, "kind": kind,
                               "sample": "mean of 1024 polygons over 4096 x 4096 float32 (cfg4 scaled): "
                                         "bucketize + GDAL-rule labels + scipy labelled mean, {:.1f} s".format(seconds)}
    return out


def zonal_e2e(ctx, host_raster):
    """AggregateRaster.get_data on a host MemorySource (the cfg2 float32 raster) and a
    MemoryGeometrySource: raster upload over PCIe, zonal kernels and the result frame inside the
    timed region."""
    from dask_geomodeling_b200 import _native, geometry, raster as raster_blocks, utils, workloads
    from dask_geomodeling_b200._compat import config as gm_config

    size = host_raster.shape[-1]
    grid = max(1, size // 128)
    src = raster_blocks.MemorySource(host_raster, workloads.F32_MAX, workloads.PROJECTION, pixel_size=1.0,
                                     pixel_origin=(0, size))
    source = geometry.MemoryGeometrySource(workloads.cfg4_polygons(size, grid, seed=7), None, workloads.PROJECTION)
    request = dict(mode="intersects", projection=workloads.PROJECTION, geometry=utils.box(0, 0, size, size))
    e2e = {"workload": "AggregateRaster.get_data, host raster {0}x{0} float32 + {1} polygons".format(size, grid * grid),
           "unit": UNIT, "h2d_bytes_per_step": int(host_raster.nbytes), "steps": 3}
    with gm_config.set({"geomodeling.raster-limit": 4 * size * size}):
        for label in ("mean", "p90"):
            view = geometry.AggregateRaster(source=source, raster=src, statistic=label)
            for _ in range(2):
                frame = view.get_data(**request)["features"]
            _native.synchronize()
            t0 = time.perf_counter()
            for _ in range(3):
                frame = view.get_data(**request)["features"]
            _native.synchronize()
            seconds = (time.perf_counter() - t0) / 3
            ctx.keep("zonal_e2e_" + label, frame["agg"].values)
            e2e[label] = {"value": size * size / seconds / 1e9, "ms_per_request": seconds * 1e3,
                          "d2h_bytes_per_step": 4 * len(frame),
                          "checksum": float(np.nansum(frame["agg"].values.astype(np.float64)))}
    return e2e


# ----------------------------------------------------------------------------
# configs[4]: temporal aggregation of ONE stack sharded by rows
# ----------------------------------------------------------------------------


def run_temporal(ctx):
    from datetime import datetime, timedelta

    from dask_geomodeling_b200 import parallel, raster, workloads
    from dask_geomodeling_b200.core import fusion

    torch, args = ctx.torch, ctx.args
    T, m = args.temporal_frames, args.temporal_size
    nodata = workloads.F32_MAX
    r0, r1 = parallel.stripe_rows(m, ctx.world)[ctx.rank]
    times = [datetime(2000, 1, 1) + timedelta(days=i) for i in range(T)]

    def kwargs_for(stat, dtype="f4"):
        return dict(mode="vals", start=times[-1], stop=None, frequency=None, timezone=None, closed=None,
                    label=None, dtype=dtype, statistic=stat)

    out = {"workload": "cfg5 TemporalAggregate over ONE {0} x {1} x {1} float32 stack, rows sharded over {2} rank(s), "
                       "no collective".format(T, m, ctx.world), "unit": "Gpixel-frames/s", "steps": max(3, args.leg_steps // 2)}
    stack = make_uniform(torch, (T, r1 - r0, m), 300 + ctx.rank, nodata, 0.03)
    sd = wrap(stack)
    whole = None
    if ctx.world > 1 and ctx.rank == 0 and not args.no_single:
        whole = wrap(make_uniform(torch, (T, m, m), 299, nodata, 0.03))
    px = T * m * m
    nbytes = T * m * m * 4 + m * m * 4
    iters = max(3, args.leg_steps // 2)
    resident = fusion.device_resident()
    resident.__enter__()           # results stay in HBM, as between the blocks of a view
    for stat in ("sum", "max"):
        kw = kwargs_for(stat)
        entry = striped_entry(
            ctx, "temporal_" + stat,
            lambda kw=kw: raster.TemporalAggregate.process(kw, {"time": times}, {"values": sd, "no_data_value": nodata}),
            None if whole is None else (lambda kw=kw: raster.TemporalAggregate.process(
                kw, {"time": times}, {"values": whole, "no_data_value": nodata})),
            px, nbytes, "temporal_stream_kernel<float, {}>".format(stat), iters, traffic_key="temporal_" + stat)
        entry["bytes"] = "T * itemsize in + itemsize out per pixel"
        out[stat] = entry
    if ctx.world == 1:
        # the rest of the temporal rows on the first 64 frames (outputs of Cumulative are T frames)
        t64 = min(64, T)
        sub = wrap(stack[:t64])
        sub_times = times[:t64]
        px64 = t64 * (r1 - r0) * m
        for stat, kernel in (("mean", "temporal_stream_kernel<float, mean>"), ("std", "temporal_moments_stream_kernel"),
                             ("median", "temporal_sort_reg_kernel")):
            kw = dict(kwargs_for(stat), start=sub_times[-1])
            ms, launches, res = ctx.time_calls(lambda kw=kw: raster.TemporalAggregate.process(
                kw, {"time": sub_times}, {"values": sub, "no_data_value": nodata}), iters)
            ctx.keep("temporal_{}_{}frames".format(stat, t64), res)
            nb = (2 if stat == "std" else 1) * px64 * 4 + (r1 - r0) * m * 4     # std reads the frames twice
            out["{}_{}frames".format(stat, t64)] = {
                "ms": ms, "gpx_s": px64 / ms / 1e6, "gpu_launches_per_call": launches,
                "roofline": ctx.roofline(nb, ms, kernel, traffic_key="temporal_" + stat)}
        kw = dict(mode="vals", start=sub_times[0], stop=sub_times[-1], frequency=None, timezone=None,
                  closed="right", label="right", dtype="<f4", statistic="sum")
        ms, launches, res = ctx.time_calls(lambda: raster.Cumulative.process(
            kw, {"time": sub_times}, {"values": sub, "no_data_value": nodata}), iters)
        ctx.keep("temporal_cumulative_sum_{}frames".format(t64), res)
        out["cumulative_sum_{}frames".format(t64)] = {
            "ms": ms, "gpx_s": px64 / ms / 1e6, "gpu_launches_per_call": launches,
            "roofline": ctx.roofline(2 * px64 * 4, ms, "temporal_cumulative_stream_kernel", traffic_key="cumulative_sum"),
            "bytes": "2 * T * itemsize per pixel (every frame read once, every running sum written once)"}
        del sub
    del stack, sd, whole
    torch.cuda.empty_cache()
    if ctx.world == 1:
        # the int16 variant of cfg5 (SURVEY 8d): the same stack shape, 2-byte cells, no data = 32767
        i16 = torch.empty((T, m, m), dtype=torch.int16, device="cuda")
        gen = torch.Generator(device="cuda").manual_seed(301)
        for a in range(0, T, 8):
            block = i16[a:a + 8]
            block.copy_(torch.randint(0, 1000, block.shape, device="cuda", generator=gen, dtype=torch.int16))
            block[torch.rand(block.shape, device="cuda", generator=gen) < 0.03] = 32767
            del block
        si = wrap(i16)
        for stat, out_bytes in (("sum", 4), ("max", 2)):
            kw = kwargs_for(stat, dtype="i4" if stat == "sum" else "i2")
            ms, launches, res = ctx.time_calls(lambda kw=kw: raster.TemporalAggregate.process(
                kw, {"time": times}, {"values": si, "no_data_value": 32767}), iters)
            ctx.keep("temporal_{}_int16".format(stat), res)
            nb = T * m * m * 2 + m * m * out_bytes
            out["{}_int16".format(stat)] = {
                "ms": ms, "gpx_s": px / ms / 1e6, "gpu_launches_per_call": launches,
                "roofline": ctx.roofline(nb, ms, "temporal_stream_kernel<short, {}>".format(stat),
                                         traffic_key="temporal_{}_int16".format(stat)),
                "bytes": "T * 2 in + out itemsize per pixel"}
        del i16, si
        torch.cuda.empty_cache()
    resident.__exit__(None, None, None)
    return out


# ----------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------


def host_link_ceiling(torch, dist, world, h2d, d2h, steps):
    """Seconds for `steps` rounds of bare page-locked copies of the end-to-end leg's bytes (h2d up,
    d2h down, on two streams so that they overlap as in the chunk pipeline), every rank at once."""
    up_host = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    down_host = torch.empty(d2h, dtype=torch.uint8).pin_memory()
    up_dev = torch.empty(h2d, dtype=torch.uint8, device="cuda")
    down_dev = torch.empty(d2h, dtype=torch.uint8, device="cuda")
    a, b = torch.cuda.Stream(), torch.cuda.Stream()

    def round_trip():
        with torch.cuda.stream(a):
            up_dev.copy_(up_host, non_blocking=True)
        with torch.cuda.stream(b):
            down_host.copy_(down_dev, non_blocking=True)

    round_trip()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        round_trip()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries the ONE JSON line and nothing else: whatever libraries print on file
    # descriptor 1 while the job runs (NCCL announces its version there) goes to stderr
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    os.environ.setdefault("GM_DEVICE", str(local_rank))
    binding = bind_to_gpu_numa_node(local_rank, world) if world > 1 else None
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from dask_geomodeling_b200 import _native, workloads
    from dask_geomodeling_b200._compat import config as gm_config
    from dask_geomodeling_b200.core import fusion
    from dask_geomodeling_b200.raster import _program

    ctx = Context(args, torch, dist, rank, local_rank, world)
    stream = ctx.stream
    size = args.size
    pixels = size * size
    ints, floats = workloads.cfg2_arrays(size, seed=43 + rank)
    view, _ = workloads.cfg2_views(ints, floats)
    request = workloads.request(size, size)

    # ---- end to end through the Block API: host arrays in, host array out ----------
    # exactly what a user of the reference does: view.get_data(**request) on NumPy
    # inputs; every step uploads both rasters (pinned H2D) and downloads the result
    h2d = ints.nbytes + floats.nbytes
    d2h = pixels  # one bool per pixel
    e2e_s = link_s = float("nan")
    e2e_checksum = None
    if not args.profile:
        result = view.get_data(**request)  # warm-up: tokens, page-locking, NVRTC, pools
        result = view.get_data(**request)
        _native.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            result = view.get_data(**request)
        _native.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_checksum = int(result["values"].sum())
        d2h = result["values"].nbytes
        del result
        link_s = host_link_ceiling(torch, dist, world, h2d, d2h, args.e2e_steps)

    # ---- kernel-resident measurement: compile once, launch K times -------------
    graph, name = view.get_compute_graph(**request)
    with gm_config.set({"geomodeling.stream": False}):  # resident launch, not the chunk pipeline
        fused = fusion.optimize(graph, name)
    task = fused[name]
    assert task[0] is fusion.fused_process, "the chain did not fuse into one task"
    plan, leaf_keys = task[1], task[2:]
    warmup = max(args.warmup, 3)
    with _native.use_stream(stream.cuda_stream), fusion.device_resident():
        leaf_payloads = [fused[k][0](*fused[k][1:]) for k in leaf_keys]  # H2D, once
        inputs = [p["values"] for p in leaf_payloads]
        leaf_types = [(p["values"].dtype, p["no_data_value"]) for p in leaf_payloads]
        compiled = _program.CompiledProgram([fusion.build_expression(plan)], leaf_types)
        out = _native.DeviceArray((1, size, size), compiled.results[0].dtype)
        # The clock sampler runs from the warm-up on: the warm-up is stretched to >= 60 ms of the
        # SAME launches (a 20-step timed region lasts 6.5 ms, one NVML query about a millisecond),
        # so that the median clock and the throttle reasons describe the load the timed region
        # runs under; `samples_in_timed_region` says how many fell inside it.
        sampler = make_sampler(local_rank) if rank == 0 else None
        t_load = time.perf_counter()
        done = 0
        while done < warmup or (time.perf_counter() - t_load < 0.06 and done < 4096):
            for _ in range(16):
                compiled.launch(inputs, [out])
            stream.synchronize()
            done += 16
        ctx.barrier()
        if sampler is not None:
            sampler.mark()
        launches_before = _native.launch_count()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for _ in range(args.steps):
            compiled.launch(inputs, [out])
        stop.record(stream)
        ctx.barrier()
        launches = _native.launch_count() - launches_before
        elapsed_ms = start.elapsed_time(stop)
        clocks = sampler.stop() if sampler else None
        checksum = int(np.asarray(out.to_host()).sum())
        ctx.keep("chain", out)
        del inputs, leaf_payloads, out
    assert e2e_checksum is None or e2e_checksum == checksum, "e2e result differs from the resident result"

    t = torch.tensor([elapsed_ms, e2e_s, link_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, e2e_s, link_s = float(t[0]), float(t[1]), float(t[2])

    striped = {}
    if "stencils" in args.legs:
        striped["stencils"] = run_stencils(ctx)
    if "zonal" in args.legs:
        striped["zonal"] = run_zonal(ctx, floats)
    if "temporal" in args.legs:
        striped["temporal"] = run_temporal(ctx)

    if rank == 0:
        ms_per_step = elapsed_ms / args.steps
        value = world * pixels / (ms_per_step / 1e3) / 1e9
        e2e_value = world * pixels * args.e2e_steps / e2e_s / 1e9
        roof = ctx.roofline(BYTES_PER_PIXEL * pixels, ms_per_step, "gm_fused (NVRTC-specialised evaluator, "
                            "V=4 px x U=4 groups per thread)", n_gpus=1, traffic_key="gm_fused_cfg2_{}".format(size))
        roof["bytes_per_pixel"] = BYTES_PER_PIXEL
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int16/float32->bool",
            "data": "synthetic",
            "config": {
                "workload": "cfg2 Reclassify+Clip+Step+IsData {0}x{0} int16/float32 per GPU".format(size),
                "l2": "inputs {:.2f} GiB per step >> 126 MB L2, no flush needed".format(h2d / 2 ** 30),
                "parallelism": "one raster pair per GPU, no collective (weak); the striped legs shard ONE workload (strong)",
                "checksum_true_pixels": checksum,
            },
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
                    "per_rank_link_gb_s": (h2d + d2h) * args.e2e_steps / e2e_s / 1e9,
                    # the same bytes per step as bare cudaMemcpyAsync calls (page-locked buffers, upload
                    # and download on two streams, all ranks at once): what the box's host side gives
                    # N ranks together, i.e. the ceiling of `value` above
                    "host_link_ceiling": {
                        "per_rank_gb_s": (h2d + d2h) * args.e2e_steps / link_s / 1e9,
                        "aggregate_gb_s": world * (h2d + d2h) * args.e2e_steps / link_s / 1e9,
                        "as_gpixel_s": world * pixels * args.e2e_steps / link_s / 1e9,
                        "e2e_fraction_of_ceiling": link_s / e2e_s},
                    "rank0_host_binding": binding},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if striped:
            line["striped"] = striped
        if world == 1 and not args.profile:
            from oracle import reference_chain

            times, kind, threads, cpu_checksum = reference_chain.time_chain(
                ints, floats, workloads.CFG2_PAIRS, steps=3, warmup=1)
            best = min(times)
            assert cpu_checksum == checksum, "CPU arm and GPU arm disagree on the result"
            line["cpu_baseline"] = {
                "value": pixels / best / 1e9, "unit": UNIT, "cores": threads, "kind": kind,
                "sample": "the whole {0}x{0} request, 2048 x 2048 tiles on a thread pool, best of 3 "
                          "({1:.2f} s); result equal to the GPU arm's".format(size, best),
            }
        if ctx.outputs is not None:
            write_outputs(args.dump_outputs, ctx.outputs)
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
