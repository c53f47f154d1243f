"""Stacks of any length: reduce_rasters past the evaluator's eight inputs (gm_reduce_stack), the
blocks built on it (Max, Group, Place "group" mode) and Place's warp mode at any number of
coordinates (gm_place); against the oracle, the evaluator and the former copy-and-reduce path."""
import ctypes

import numpy as np
import pytest

from dask_geomodeling_b200 import _native, _state, raster, workloads
from dask_geomodeling_b200.raster import _program
from dask_geomodeling_b200.raster.reduction import reduce_rasters
from oracle import raster as R

pytestmark = pytest.mark.gpu

DEVICE_STATS = ("last", "first", "count", "max", "min", "sum", "product")
FLOAT_ONLY = ("sum", "product")


@pytest.fixture(params=["interp", "auto"])
def eval_mode(request):
    lib = _native.lib()
    before = lib.gm_get_eval_mode()
    _native.check(lib.gm_set_eval_mode(1 if request.param == "interp" else 0))
    yield request.param
    _native.check(lib.gm_set_eval_mode(before))


def make_stack(n, dtypes, nodatas, shape, seed):
    rng = np.random.default_rng(seed)
    stack = []
    for k in range(n):
        dtype, nd = np.dtype(dtypes[k % len(dtypes)]), nodatas[k % len(nodatas)]
        if dtype.kind == "f":
            values = rng.uniform(-50, 50, shape).astype(dtype)
        else:
            info = np.iinfo(dtype)
            values = rng.integers(max(info.min, -100), min(info.max, 100), shape).astype(dtype)
        mask = rng.random(shape) < 0.3
        if nd is not None:
            if dtype.kind == "f" and not np.isnan(nd):
                near = rng.random(shape) < 0.05   # isclose hits and near-misses below the sentinel
                values[near] = (np.asarray(nd, dtype) * (1 - rng.choice([2e-6, 2e-5], near.sum()))).astype(dtype)
            values[mask] = nd
        stack.append((values, nd))
    return stack


def assert_reduced(got, expected, statistic, n):
    """Bit for bit, except float sums of more than 8 rasters: those are added in raster order (the
    evaluator's OVERLAY step), NumPy's nansum adds them pairwise -- the last bits may differ."""
    got = np.asarray(got)
    if statistic == "sum" and n > 8:
        assert got.dtype == expected.dtype
        np.testing.assert_allclose(got, expected, rtol=1e-5, atol=1e-3 * n)
    else:
        np.testing.assert_array_equal(got, expected)


def check_against_oracle(stack, statistic, on_device=False):
    payloads = [{"values": _native.DeviceArray.from_host(v) if on_device else v, "no_data_value": nd}
                for v, nd in stack]
    got = reduce_rasters(payloads, statistic)
    expected, nodata = R.reduce_rasters(stack, statistic)
    assert_reduced(got["values"], expected, statistic, len(stack))
    assert np.asarray(got["values"]).dtype == expected.dtype
    assert got["no_data_value"] is nodata or got["no_data_value"] == nodata or (
        np.isnan(got["no_data_value"]) and np.isnan(nodata))


CASES = [
    (("f4",), (np.float32(3.4028235e38),)),
    (("f8",), (-9999.0,)),
    (("f4",), (np.nan,)),
    (("f4",), (None,)),
    (("f4", "f8"), (1e-3, -9999.0)),
    (("i2",), (-32768,)),
    (("u1",), (255,)),
    (("i4", "i2", "u1"), (-1, 7, 0)),
]


@pytest.mark.parametrize("n", [9, 17, 64, 300])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_reduce_any_length_against_oracle(eval_mode, n, case):
    dtypes, nodatas = CASES[case]
    stack = make_stack(n, dtypes, nodatas, (2, 13, 21), seed=n + case)   # odd planes, two frames
    for statistic in DEVICE_STATS:
        if statistic in FLOAT_ONLY and np.dtype(dtypes[0]).kind != "f":
            with pytest.raises(NotImplementedError):
                reduce_rasters([{"values": v, "no_data_value": nd} for v, nd in stack], statistic)
            continue
        check_against_oracle(stack, statistic, on_device=(n == 17))


def test_misaligned_frame_views():
    """Group hands in (1, h, w) views at frame offsets: 47 x 53 float32 planes are not 16-byte
    aligned, and 12 of them exceed the evaluator's inputs."""
    stack = make_stack(4, ("f4",), (-1.0,), (3, 47, 53), seed=5)
    devs = [_native.DeviceArray.from_host(v) for v, _ in stack]
    payloads, frames = [], []
    for d, (v, nd) in zip(devs, stack):
        for f in range(3):
            view = _native.DeviceArray((1, 47, 53), d.dtype, owner=d, ptr=d.ptr + f * 47 * 53 * 4)
            payloads.append({"values": view, "no_data_value": nd})
            frames.append((v[f:f + 1], nd))
    for statistic in ("last", "max", "sum", "count"):
        got = reduce_rasters(payloads, statistic)
        expected, _ = R.reduce_rasters(frames, statistic)
        assert_reduced(got["values"], expected, statistic, len(frames))


def evaluator(stack, statistic, dtype, nodata):
    """The stack reduced by one evaluator program (gm_eval_program), as reduce_rasters lowers it."""
    node = _program.Node("reduce", [_program.Leaf(i) for i in range(len(stack))], statistic=statistic,
                         dtype=np.dtype(dtype).name, fillvalue=nodata)
    (values, _, _), = _program.evaluate([node], list(stack))
    return np.asarray(values)


@pytest.mark.parametrize("n", [1, 2, 5, 8])
def test_stack_kernel_matches_evaluator_bytes(eval_mode, n):
    stack = make_stack(n, ("f4", "i2", "f8"), (-9999.0, 3, np.nan), (1, 37, 41), seed=n)
    floats = make_stack(n, ("f4",), (-9999.0,), (1, 37, 41), seed=n)
    for statistic in DEVICE_STATS:
        rasters = floats if statistic in FLOAT_ONLY else stack
        dtype, nodata = rasters[0][0].dtype, rasters[0][1]
        evaluated = evaluator(rasters, statistic, dtype, nodata)
        direct = _program.run_stack(statistic, rasters, dtype, nodata, False)
        assert evaluated.tobytes() == np.asarray(direct).tobytes(), statistic


def test_sixty_four_rasters_cost_one_reduction_launch():
    stack = make_stack(64, ("f4",), (-1.0,), (1, 64, 64), seed=1)
    payloads = [{"values": _native.DeviceArray.from_host(v), "no_data_value": nd} for v, nd in stack]
    with _state.device_resident():
        before = _native.launch_count()
        reduce_rasters(payloads, "max")
        assert _native.launch_count() - before == 1


def test_unchanged_errors():
    stack = [{"values": v, "no_data_value": nd} for v, nd in make_stack(12, ("i2",), (0,), (1, 8, 8), 2)]
    with pytest.raises(NotImplementedError):
        reduce_rasters(stack, "median")
    with pytest.raises(NotImplementedError):
        reduce_rasters(stack, "sum")


def test_blocks_at_any_length():
    stack = make_stack(20, ("f4",), (np.float32(3.4028235e38),), (1, 48, 48), seed=8)
    nd = stack[0][1]
    sources = [workloads.source(v, nd) for v, _ in stack]
    request = workloads.request(48, 48)
    for n in (9, 20):
        got = raster.Max(*sources[:n]).get_data(**request)
        expected, _ = R.reduce_rasters(stack[:n], "max", nd, "float32")
        np.testing.assert_array_equal(got["values"], expected)
    got = raster.Multiply(raster.Max(*sources[:9]), 2.0).get_data(**request)
    best, _ = R.reduce_rasters(stack[:9], "max", nd, "float32")
    expected, _ = R.elementwise("multiply", "float32", nd, (best, nd), 2.0)
    np.testing.assert_array_equal(got["values"], expected)
    # Group of 12 overlapping non-temporal sources
    got = raster.Group(*sources[:12]).get_data(**request)
    expected, _ = R.reduce_rasters(stack[:12], "last", R.dtype_max("f4"), "float32")
    np.testing.assert_array_equal(got["values"], expected)


def test_group_of_many_aligned_temporal_sources():
    """Ten equidistant sources over the same three hours: ten contributions per output frame."""
    stack = make_stack(10, ("f4",), (np.float32(3.4028235e38),), (3, 24, 24), seed=12)
    nd = stack[0][1]
    hour = 3600 * 1000
    view = raster.Group(*[workloads.source(v, nd, time_first=0, time_delta=hour) for v, _ in stack])
    from datetime import datetime
    request = workloads.request(24, 24, start=datetime(1970, 1, 1), stop=datetime(1970, 1, 1, 2))
    got = view.get_data(**request)
    expected, fill = R.group_by_bands(stack, [(0, 3)] * 10, "f4", (3, 24, 24))
    np.testing.assert_array_equal(got["values"], expected)


# ---- Place --------------------------------------------------------------------------------------
def place_kwargs(coordinates, statistic, src_shape, dst_shape):
    _, sh, sw = src_shape
    dh, dw = dst_shape
    return {"mode": "warp", "anchor": (0.0, float(sh)), "coordinates": coordinates,
            "src_bbox": (0.0, 0.0, float(sw), float(sh)), "dst_bbox": (0.0, 0.0, float(dw), float(dh)),
            "cellsize": (1.0, 1.0), "statistic": statistic}


def old_place(values, nodata, kwargs):
    """The former warp mode: one request-sized copy per coordinate (gm_resample_nn), then
    reduce_rasters over the copies."""
    size_x, size_y = kwargs["cellsize"]
    anchor, src_bbox = kwargs["anchor"], kwargs["src_bbox"]
    anchor_px = ((anchor[0] - src_bbox[0]) / size_x, (anchor[1] - src_bbox[1]) / size_y)
    x1, y1, x2, y2 = kwargs["dst_bbox"]
    dst_h, dst_w = round((y2 - y1) / size_y), round((x2 - x1) / size_x)
    depth, src_h, src_w = values.shape
    shape = (depth, dst_h, dst_w)
    source = _native.DeviceArray.from_host(values)
    holder, nodata_ptr = _native.scalar_ptr(nodata, values.dtype)
    stack = []
    for cx, cy in kwargs["coordinates"]:
        di = round((cx - x1) / size_x - anchor_px[0])
        dj = dst_h - src_h - round((cy - y1) / size_y - anchor_px[1])
        if di <= -src_w or di >= dst_w or dj <= -src_h or dj >= dst_h:
            continue
        placed = _native.DeviceArray(shape, values.dtype)
        _native.check(_native.lib().gm_resample_nn(
            ctypes.byref(_native.as_gm_array(source)), ctypes.byref(_native.as_gm_array(placed)), nodata_ptr,
            float(-di), 1.0, float(-dj), 1.0, _native.current_stream()))
        stack.append({"values": placed, "no_data_value": nodata})
    if not stack:
        return np.full(shape, nodata, values.dtype)
    return np.asarray(reduce_rasters(stack, kwargs["statistic"])["values"])


def place_source(shape, dtype, nodata, seed):
    rng = np.random.default_rng(seed)
    values = rng.uniform(1, 100, shape).astype(dtype)
    values[rng.random(shape) < 0.3] = nodata
    return values


@pytest.mark.parametrize("n", [1, 3, 100, 5000])
def test_place_against_oracle(n):
    rng = np.random.default_rng(n)
    src_shape, dst_shape = (2, 9, 13), (70, 130)
    nodata = -9999.0
    values = place_source(src_shape, "f4", nodata, n)
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(-20, 150, n), rng.uniform(-20, 90, n))]
    for statistic in DEVICE_STATS:
        kwargs = place_kwargs(coordinates, statistic, src_shape, dst_shape)
        got = raster.Place.process(kwargs, {"values": values, "no_data_value": nodata})
        expected, _ = R.place_warp(values, nodata, kwargs)
        assert_reduced(got["values"], expected, statistic, n)


@pytest.mark.parametrize("nodata", [-9999.0, np.nan, None])
def test_place_non_finite_sources_against_old_path(nodata):
    rng = np.random.default_rng(7)
    src_shape, dst_shape = (1, 11, 7), (40, 50)
    values = place_source(src_shape, "f4", -9999.0 if nodata is None else nodata, 3)
    values[0, 2, :] = np.inf
    values[0, 5, 1:4] = np.nan
    values[0, 7, 2] = -np.inf
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(-5, 55, 40), rng.uniform(-5, 45, 40))]
    for statistic in DEVICE_STATS:
        kwargs = place_kwargs(coordinates, statistic, src_shape, dst_shape)
        got = raster.Place.process(kwargs, {"values": values, "no_data_value": nodata})
        expected = old_place(values, nodata, kwargs)
        assert np.asarray(got["values"]).tobytes() == expected.tobytes(), statistic


def test_place_integer_source_against_old_path():
    rng = np.random.default_rng(9)
    values = rng.integers(0, 50, (1, 6, 5)).astype("i2")
    values[values < 10] = -1
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(-3, 33, 30), rng.uniform(-3, 23, 30))]
    for statistic in ("last", "first", "count", "max", "min"):
        kwargs = place_kwargs(coordinates, statistic, values.shape, (20, 30))
        got = raster.Place.process(kwargs, {"values": values, "no_data_value": -1})
        assert np.asarray(got["values"]).tobytes() == old_place(values, -1, kwargs).tobytes(), statistic


def test_place_group_mode_with_many_coordinates():
    rng = np.random.default_rng(4)
    data = rng.uniform(1, 100, (1, 6, 8)).astype("f4")
    nodata = workloads.F32_MAX
    data[rng.random(data.shape) < 0.3] = nodata
    src = raster.MemorySource(data, nodata, workloads.PROJECTION, pixel_size=1.0, pixel_origin=(10, 26))
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(0, 12, 12), rng.uniform(0, 12, 12))]
    fine = dict(mode="vals", bbox=(4, 4, 8, 8), width=2, height=2, projection=workloads.PROJECTION)
    view = raster.Place(src, workloads.PROJECTION, (12.0, 22.0), coordinates, "max")
    plan = view.get_sources_and_requests(**fine)
    assert plan[0][0]["mode"] == "group" and len(plan) > 9
    stack = [(np.asarray(s.get_data(**r)["values"]), nodata) for s, r in plan[1:]]
    expected, _ = R.reduce_rasters(stack, "max")
    np.testing.assert_array_equal(view.get_data(**fine)["values"], expected)


def test_scale_sixteen_rasters_8192():
    rng = np.random.default_rng(0)
    stack = []
    for _ in range(16):
        v = rng.standard_normal((1, 8192, 8192), dtype=np.float32)
        v[v > 1.5] = -9999.0
        stack.append(v)
    got = np.asarray(reduce_rasters([{"values": v, "no_data_value": -9999.0} for v in stack], "max")["values"])
    masked = np.stack(stack)
    masked = np.where(masked == -9999.0, -np.inf, masked).max(axis=0)
    np.testing.assert_array_equal(got, np.where(np.isinf(masked), np.float32(-9999.0), masked))


def test_scale_place_2000_coordinates_16384():
    rng = np.random.default_rng(1)
    src = rng.uniform(1, 100, (1, 256, 256)).astype("f4")
    src[src < 20] = -9999.0
    n, size = 2000, 16384
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(-200, size + 200, n),
                                                         rng.uniform(-200, size + 200, n))]
    kwargs_max = place_kwargs(coordinates, "max", src.shape, (size, size))
    best = np.full((size, size), -np.inf, np.float32)
    count = np.zeros((size, size), np.float32)
    data = src[0] != -9999.0
    for cx, cy in coordinates:
        di = round(cx - 0.0)
        dj = size - 256 - round(cy - 256.0)
        j0, i0 = max(dj, 0), max(di, 0)
        j1, i1 = min(dj + 256, size), min(di + 256, size)
        if j0 >= j1 or i0 >= i1:
            continue
        part = src[0, j0 - dj:j1 - dj, i0 - di:i1 - di]
        ok = data[j0 - dj:j1 - dj, i0 - di:i1 - di]
        view = best[j0:j1, i0:i1]
        view[ok] = np.maximum(view[ok], part[ok])
        count[j0:j1, i0:i1] += ok
    got = np.asarray(raster.Place.process(kwargs_max, {"values": src, "no_data_value": -9999.0})["values"])[0]
    np.testing.assert_array_equal(got, np.where(np.isinf(best), np.float32(-9999.0), best))
    kwargs_count = place_kwargs(coordinates, "count", src.shape, (size, size))
    got = np.asarray(raster.Place.process(kwargs_count, {"values": src, "no_data_value": -9999.0})["values"])[0]
    np.testing.assert_array_equal(got, count)
