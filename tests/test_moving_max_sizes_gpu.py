"""MovingMax at sizes beyond the compile-time footprints (3...15 for uint8 / bool, int16, int32,
float32 and float64): the tiled kernel (radius <= 8; 8-byte cells below 7) and the chord kernel
(every other size, no cap), against the oracle's SciPy disc filter and, for sizes where that is too slow, a
chord-by-chord restatement of it."""
import os
import socket

import numpy as np
import pytest
from scipy import ndimage

from dask_geomodeling_b200 import raster, workloads
from oracle import raster as R

pytestmark = pytest.mark.gpu

ALL_DTYPES = ["u1", "i1", "u2", "i2", "u4", "i4", "i8", "f4", "f8"]
# dtypes without a compile-time footprint: sizes 3...15 run the tiled kernel (int64 at 15: the chord kernel)
NO_FIXED = ["i1", "u2", "u4", "i8"]


def random_values(shape, dtype, seed, nodata, nodata_fraction=0.3):
    """Values over the whole range of the dtype, 1 % of them the dtype minimum (a data value
    that equals what no data becomes inside the filter), `nodata_fraction` no data."""
    rng = np.random.default_rng(seed)
    d = np.dtype(dtype)
    if d.kind == "f":
        values = (rng.standard_normal(shape) * 1000).astype(d)
    else:
        # int64 within +-2**53: SciPy's maximum filter holds values in a double, so the oracle
        # rounds larger ones; the kernels return them exactly
        info = np.iinfo(d)
        lo, hi = max(info.min, -2 ** 53), min(info.max, 2 ** 53)
        values = rng.integers(lo, hi, shape, dtype=d, endpoint=False)
    values[rng.random(shape) < 0.01] = R.dtype_min(d)
    if nodata is not None:
        values[rng.random(shape) < nodata_fraction] = nodata
    return values


def chord_moving_max(values, nodata, size):
    """R.moving_max restated chord by chord: footprint row dy contributes a
    maximum_filter1d of width 2 hw[dy] + 1 over the rows the output needs."""
    r = size // 2
    lowest = R.dtype_min(values.dtype)
    missing = values == nodata if nodata is not None else np.zeros(values.shape, bool)
    work = np.where(missing, lowest, values).astype(values.dtype)
    t, sh, sw = work.shape
    h, w = sh - 2 * r, sw - 2 * r
    out = np.full((t, h, w), lowest, dtype=values.dtype)
    footprint = R.footprint(size)
    for dy in range(-r, r + 1):
        hw = (int(footprint[dy + r].sum()) - 1) // 2
        rows = work[:, r + dy:r + dy + h, :]
        out = np.maximum(out, ndimage.maximum_filter1d(rows, 2 * hw + 1, axis=2)[:, :, r:r + w])
    out[(out == lowest) & missing[:, r:r + h, r:r + w]] = nodata
    return out


def run(values, nodata, size):
    got = raster.MovingMax.process({"values": values, "no_data_value": nodata}, size)
    assert got["no_data_value"] == nodata
    return np.asarray(got["values"])


@pytest.mark.parametrize("dtype,size", [(d, s) for s in (17, 19, 33, 65, 67, 101) for d in ALL_DTYPES] +
                         [(d, s) for s in (3, 5, 11, 15) for d in NO_FIXED])
def test_parity_with_scipy(dtype, size):
    r = size // 2
    h, w = 37, 53          # odd, not multiples of the tile
    nodata = R.dtype_max(dtype)
    values = random_values((2, h + 2 * r, w + 2 * r), dtype, size, nodata)
    values[0, :size + 4, :size + 4] = nodata     # a hole larger than the footprint stays no data
    expected, _ = R.moving_max(values, nodata, size)
    assert (expected == nodata).any()
    got = run(values, nodata, size)
    assert got.dtype == expected.dtype and got.shape == (2, h, w)
    np.testing.assert_array_equal(got, expected)


@pytest.mark.parametrize("dtype", ["u1", "i8", "f4"])
@pytest.mark.parametrize("size", [17, 67])
def test_parity_without_nodata(dtype, size):
    r = size // 2
    values = random_values((2, 37 + 2 * r, 53 + 2 * r), dtype, 7, None)
    # R.moving_max's no-data step cannot store None in an integer array: without no data the
    # reference is the disc filter alone
    expected = ndimage.maximum_filter(values, footprint=R.footprint(size)[np.newaxis])[:, r:-r, r:-r]
    np.testing.assert_array_equal(run(values, None, size), expected)


@pytest.mark.parametrize("size", [33, 67, 101])
def test_chord_restatement_equals_the_oracle(size):
    r = size // 2
    for dtype in ("f4", "i2", "u1"):
        nodata = R.dtype_max(dtype)
        values = random_values((2, 19 + 2 * r, 23 + 2 * r), dtype, size, nodata)
        values[1, :size + 2, :size + 2] = nodata
        np.testing.assert_array_equal(chord_moving_max(values, nodata, size), R.moving_max(values, nodata, size)[0])


# ramp directions (a, b), value growing with a x + b y: the maximum over a disc lies on its rim
# where the rim's normal is (a, b); the steep ones reach the outermost footprint rows
RAMPS = [(1, 0), (0, -1), (1, 1), (-1, 2), (2, -1), (1, 4), (-1, 8)]


def rim_values(h, w, size, dtype, seed, nodata):
    """One band per ramp of RAMPS, shifted so that the maximum over the disc of the middle output
    is 100 + 10 * band and clipped to [0, 250], with 30 % no data."""
    r = size // 2
    dy, dx = np.nonzero(R.footprint(size))
    y = np.arange(h + 2 * r)[:, None] - (r + h // 2)
    x = np.arange(w + 2 * r)[None, :] - (r + w // 2)
    bands = []
    for k, (a, b) in enumerate(RAMPS):
        reach = int((a * (dx - r) + b * (dy - r)).max())
        bands.append(np.clip(a * x + b * y - reach + 100 + 10 * k, 0, 250))
    values = np.stack(bands).astype(dtype)
    values[np.random.default_rng(seed).random(values.shape) < 0.3] = nodata
    return values


@pytest.mark.parametrize("dtype", ["f4", "i2", "u1"])
@pytest.mark.parametrize("size", [257, 1025, 4097])
@pytest.mark.parametrize("out_shape", [(9, 13), (1, 1)])
def test_large_sizes(dtype, size, out_shape):
    h, w = out_shape
    nodata = R.dtype_max(dtype)
    values = rim_values(h, w, size, dtype, size + h, nodata)
    expected = chord_moving_max(values, nodata, size)
    # the outputs are set by the footprint's edge, not by one window-wide maximum
    assert np.unique(expected).size >= len(RAMPS)
    if h * w > 1:
        assert all(np.unique(band).size > 1 for band in expected)
    np.testing.assert_array_equal(run(values, nodata, size), expected)


@pytest.mark.parametrize("out_shape", [(5, 7), (1, 300), (300, 1), (1, 1)])
@pytest.mark.parametrize("dtype,size", [("f4", 67), ("i2", 67), ("f8", 17), ("u4", 9)])
def test_edge_shapes(out_shape, dtype, size):
    """Outputs narrower and shorter than the radius, three bands, a single row or column."""
    r = size // 2
    h, w = out_shape
    nodata = R.dtype_max(dtype)
    values = random_values((3, h + 2 * r, w + 2 * r), dtype, h * 1000 + w, nodata, nodata_fraction=0.6)
    expected = chord_moving_max(values, nodata, size)
    if size <= 67:
        np.testing.assert_array_equal(expected, R.moving_max(values, nodata, size)[0])
    np.testing.assert_array_equal(run(values, nodata, size), expected)


def test_wider_source_than_the_halo_is_refused_above_15():
    """Pitch padding is a form of the compile-time kernels only; the chord kernel refuses it."""
    from dask_geomodeling_b200._native import NativeLibraryError

    values = random_values((1, 20 + 16, 21 + 16 + 3), "f4", 1, R.dtype_max("f4"))
    with pytest.raises(NativeLibraryError, match="pitch padding"):
        raster.MovingMax.process({"values": values, "no_data_value": R.dtype_max("f4")}, 17, 3)


@pytest.mark.parametrize("size", [101, 201])
def test_view_through_get_data(size):
    r = size // 2
    n = 131 + 2 * r + 40
    a, _ = workloads.cfg1_arrays(n)
    src = workloads.source(a, workloads.F32_MAX)
    req = workloads.request(131, 131)
    x1, y1 = r + 10, r + 12
    req["bbox"] = (x1, y1, x1 + 131, y1 + 131)
    view = raster.MovingMax(src, size)
    (_, enlarged), _, (pad, _) = view.get_sources_and_requests(**req)
    assert pad == 0 and enlarged["width"] == 131 + 2 * r
    got = view.get_data(**req)
    window = a[:, n - (y1 + 131) - r:n - y1 + r, x1 - r:x1 + 131 + r]
    expected = R.moving_max(window, workloads.F32_MAX, size)[0] if size <= 101 else \
        chord_moving_max(window, workloads.F32_MAX, size)
    np.testing.assert_array_equal(got["values"], expected)


# ---- row stripes on two ranks (helpers as in tests/test_parallel_gpu.py) ----------------------

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(rank, world, port, n_gpus, fn):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    device = rank if n_gpus >= world else 0
    os.environ["GM_DEVICE"] = str(device)
    torch.cuda.set_device(device)
    if n_gpus >= world:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", device))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        fn(rank, world)
    finally:
        dist.destroy_process_group()


def spawn(fn, world=2):
    import torch
    import torch.multiprocessing as mp

    mp.spawn(_run, args=(world, _free_port(), torch.cuda.device_count(), fn), nprocs=world, join=True)


def _stripes_worker(rank, world):
    import torch

    from dask_geomodeling_b200 import parallel

    rng = np.random.default_rng(5)
    h, w, size = 97, 131, 67          # stripes of 49 and 48 rows, halo 33
    r = size // 2
    dem = (rng.standard_normal((2, h, w)) * 100).astype("f4")
    nodata = float(np.finfo("f4").max)
    dem[rng.random(dem.shape) < 0.3] = nodata
    r0, r1 = parallel.stripe_rows(h, world)[rank]
    assert r1 - r0 > r
    local = torch.from_numpy(dem[:, r0:r1].copy()).cuda()
    got = parallel.stencil_striped(raster.MovingMax.process, local, nodata, r, r, size)
    whole = np.pad(dem, ((0, 0), (r, r), (r, r)), constant_values=nodata)
    expected, _ = R.moving_max(whole, nodata, size)
    np.testing.assert_array_equal(np.asarray(got["values"]), expected[:, r0:r1])


def test_row_stripes_on_two_ranks():
    spawn(_stripes_worker)


def test_size_past_the_shared_memory_limit_names_the_limit():
    """float64 at 2147: the chord kernel's table needs more than the 227 KB a block may hold."""
    from dask_geomodeling_b200._native import NativeLibraryError

    values = np.zeros((1, 1 + 2146, 1 + 2146), dtype="f8")
    with pytest.raises(NativeLibraryError, match="the largest size for this dtype is 2145"):
        raster.MovingMax.process({"values": values, "no_data_value": None}, 2147)
