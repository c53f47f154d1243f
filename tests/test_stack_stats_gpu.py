"""mean, var, std, argmin and argmax of raster stacks on the device (gm_reduce_stack_stat) and in
Place's warp mode (gm_place_stat), against the oracle's reduce_rasters with NumPy's
nan-functions: out = nodata, out[some] = f(stacked[:, some], axis=0)."""
import numpy as np
import pytest

from dask_geomodeling_b200 import _native, _state, raster, workloads
from dask_geomodeling_b200.raster.reduction import reduce_rasters
from oracle import raster as R
from test_stack_reduce_gpu import CASES, make_stack, place_kwargs

pytestmark = pytest.mark.gpu

STATS = ("mean", "var", "std", "argmin", "argmax")
FLOAT_ONLY = ("mean", "var", "std")
NAN_FUNCTIONS = {"mean": np.nanmean, "var": np.nanvar, "std": np.nanstd, "argmin": np.nanargmin,
                 "argmax": np.nanargmax}


@pytest.fixture(autouse=True)
def oracle_statistics(monkeypatch):
    """The oracle's stacking rule (R.reduce_rasters, R.place_warp) with the five nan-functions."""
    for name, function in NAN_FUNCTIONS.items():
        monkeypatch.setitem(R._NAN_REDUCERS, name, function)


def payloads(stack, on_device=False):
    return [{"values": _native.DeviceArray.from_host(v) if on_device else v, "no_data_value": nd}
            for v, nd in stack]


def assert_stat(got, expected, statistic, n):
    """Bit for bit, except mean / var / std of 8 or more rasters: those add in raster order, while
    NumPy's reduction along the stack adds 8 or more values pairwise (eight partial sums, then a
    tree), so the last bits may differ."""
    got = np.asarray(got)
    assert got.dtype == expected.dtype
    if statistic in FLOAT_ONLY and n >= 8:
        np.testing.assert_allclose(got, expected, rtol=2e-4, atol={"var": 1.0}.get(statistic, 1e-2))
    else:
        np.testing.assert_array_equal(got, expected)


@pytest.mark.parametrize("n", [1, 2, 5, 8, 9, 17, 64, 300])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_reduce_against_oracle(n, case):
    dtypes, nodatas = CASES[case]
    stack = make_stack(n, dtypes, nodatas, (2, 13, 21), seed=1000 + n + case)
    for statistic in STATS:
        if statistic in FLOAT_ONLY and np.dtype(dtypes[0]).kind != "f":
            with pytest.raises(NotImplementedError):
                reduce_rasters(payloads(stack), statistic)
            continue
        got = reduce_rasters(payloads(stack, on_device=(n == 17)), statistic)
        expected, nodata = R.reduce_rasters(stack, statistic)
        assert_stat(got["values"], expected, statistic, n)
        assert got["no_data_value"] is nodata or got["no_data_value"] == nodata or (
            np.isnan(got["no_data_value"]) and np.isnan(nodata))


def test_edge_cells():
    """Per column: all no data, a single value, +inf, +inf and -inf, a tie, only -inf (raster 0
    without data), -inf and a value, a NaN value beside a value."""
    nd = np.float32(-9999.0)
    inf = np.inf
    columns = [
        [nd, nd, nd],
        [nd, 3.0, nd],
        [1.0, inf, 2.0],
        [inf, -inf, 1.0],
        [4.0, 7.0, 7.0],
        [nd, -inf, -inf],
        [-inf, 5.0, nd],
        [np.nan, 2.0, 6.0],
    ]
    values = np.array(columns, dtype=np.float32).T.reshape(3, 1, 1, len(columns))
    stack = [(values[k], nd) for k in range(3)]
    for statistic in STATS:
        got = reduce_rasters(payloads(stack), statistic)
        expected, _ = R.reduce_rasters(stack, statistic)
        np.testing.assert_array_equal(np.asarray(got["values"]), expected)
    got = np.asarray(reduce_rasters(payloads(stack), "argmax")["values"])[0, 0]
    assert got[0] == nd and got[4] == 1 and got[5] == 0
    got = np.asarray(reduce_rasters(payloads(stack), "var")["values"])[0, 0]
    assert got[1] == 0 and np.isnan(got[2]) and np.isnan(got[3])
    # the same in float64 and into an integer output for argmin / argmax
    stack64 = [(v.astype("f8"), -9999.0) for v, _ in stack]
    for statistic in STATS:
        expected, _ = R.reduce_rasters(stack64, statistic)
        np.testing.assert_array_equal(np.asarray(reduce_rasters(payloads(stack64), statistic)["values"]), expected)
    for statistic in ("argmin", "argmax"):
        got = reduce_rasters(payloads(stack), statistic, no_data_value=255, dtype="u1")
        expected, _ = R.reduce_rasters(stack, statistic, 255, "u1")
        np.testing.assert_array_equal(np.asarray(got["values"]), expected)


def test_uint8_output_rounds_wider_rasters_to_float16():
    """A uint8 first raster makes the working dtype float16: int16 values beyond +-2048 and int32
    values (beyond 65504: inf) round, which creates ties that decide argmin / argmax."""
    rng = np.random.default_rng(3)
    shape = (1, 40, 50)
    stack = [(rng.integers(0, 255, shape).astype("u1"), 255)]
    for k in range(12):
        if k % 2:
            v = rng.integers(-32768, 32767, shape).astype("i2")
            near = rng.random(shape) < 0.5
            v[near] = rng.choice([2049, 2050, 2051, 4097, 4099, -2049, -2051], near.sum())
            nd = -32768
        else:
            v = rng.choice([-100000, -65520, -65504, 65504, 65519, 65520, 70000, 3000, 3001, 3002], shape).astype("i4")
            nd = 3001
        stack.append((v, nd))
    for statistic in ("argmin", "argmax"):
        got = reduce_rasters(payloads(stack), statistic)
        expected, _ = R.reduce_rasters(stack, statistic)
        assert expected.dtype == np.uint8
        np.testing.assert_array_equal(np.asarray(got["values"]), expected)
    with pytest.raises(NotImplementedError):
        reduce_rasters(payloads(stack), "mean")


def test_device_resident_and_misaligned_frame_views():
    stack = make_stack(4, ("f4",), (-1.0,), (3, 47, 53), seed=5)
    devs = [_native.DeviceArray.from_host(v) for v, _ in stack]
    views, frames = [], []
    for d, (v, nd) in zip(devs, stack):
        for f in range(3):
            view = _native.DeviceArray((1, 47, 53), d.dtype, owner=d, ptr=d.ptr + f * 47 * 53 * 4)
            views.append({"values": view, "no_data_value": nd})
            frames.append((v[f:f + 1], nd))
    for statistic in STATS:
        with _state.device_resident():
            got = reduce_rasters(views, statistic)
        assert _native.is_device(got["values"])
        expected, _ = R.reduce_rasters(frames, statistic)
        assert_stat(got["values"].to_host(), expected, statistic, len(frames))


@pytest.mark.parametrize("statistic", ["mean", "var"])
def test_sixty_four_rasters_cost_one_launch(statistic):
    stack = make_stack(64, ("f4",), (-1.0,), (1, 64, 64), seed=1)
    devs = payloads(stack, on_device=True)
    with _state.device_resident():
        before = _native.launch_count()
        reduce_rasters(devs, statistic)
        assert _native.launch_count() - before == 1


def test_errors():
    ints = payloads(make_stack(3, ("i2",), (0,), (1, 8, 8), 2))
    floats = payloads(make_stack(3, ("f4",), (0.0,), (1, 8, 8), 2))
    for statistic in ("median", "p90"):
        with pytest.raises(NotImplementedError):
            reduce_rasters(floats, statistic)
    for statistic in FLOAT_ONLY:
        with pytest.raises(NotImplementedError):
            reduce_rasters(ints, statistic)
        with pytest.raises(NotImplementedError):
            reduce_rasters(floats, statistic, dtype="i4")
    with pytest.raises(KeyError):
        reduce_rasters(floats, "mode")


# ---- Place --------------------------------------------------------------------------------------
def place_source(shape, nodata, seed):
    rng = np.random.default_rng(seed)
    values = rng.uniform(1, 100, shape).astype("f4")
    values[rng.random(shape) < 0.3] = nodata
    values[..., 2, 3] = values[..., 1, 1]    # ties between copies
    return values


def check_place(values, nodata, coordinates, dst_shape):
    for statistic in STATS:
        kwargs = place_kwargs(coordinates, statistic, values.shape, dst_shape)
        got = raster.Place.process(kwargs, {"values": values, "no_data_value": nodata})
        expected, _ = R.place_warp(values, nodata, kwargs)
        assert_stat(got["values"], expected, statistic, len(coordinates))


@pytest.mark.parametrize("n", [1, 7, 1000])
@pytest.mark.parametrize("nodata", [-9999.0, np.nan])
def test_place_against_oracle(n, nodata):
    rng = np.random.default_rng(n)
    values = place_source((2, 9, 13), nodata, n)
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(-20, 150, n), rng.uniform(-20, 90, n))]
    check_place(values, nodata, coordinates, (70, 130))


def place_at(offsets, src_shape, dst_shape):
    """Coordinates that shift the source by (di, dj) (see place_kwargs)."""
    return [(float(di), float(dst_shape[0] - dj)) for di, dj in offsets]


def test_place_which_copies_are_stacked():
    """Band 0 holds data in the source's top-left corner only, band 1 none: a copy whose footprint
    meets the request with its data outside, a copy completely outside, copies with data inside."""
    nodata = -9999.0
    values = np.full((2, 6, 8), nodata, np.float32)
    values[0, :2, :2] = [[5.0, 1.0], [3.0, 5.0]]
    values[1, 4, 6] = 2.0    # data of band 1, right of the request for most copies
    dst = (12, 16)
    offsets = [(-3, 0), (30, 2), (2, 2), (-1, 5), (3, 3), (10, -1), (2, 2), (-6, -4), (12, 8)]
    check_place(values, nodata, place_at(offsets, values.shape, dst), dst)
    empty = np.full((2, 6, 8), nodata, np.float32)
    check_place(empty, nodata, place_at(offsets, values.shape, dst), dst)
    for statistic in STATS:
        kwargs = place_kwargs(place_at(offsets, values.shape, dst), statistic, values.shape, dst)
        got = raster.Place.process(kwargs, {"values": empty, "no_data_value": nodata})
        assert (np.asarray(got["values"]) == nodata).all()


def test_place_integer_source():
    rng = np.random.default_rng(9)
    values = rng.integers(0, 50, (1, 6, 5)).astype("i2")
    values[values < 10] = -1
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(-3, 33, 30), rng.uniform(-3, 23, 30))]
    for statistic in ("argmin", "argmax"):
        kwargs = place_kwargs(coordinates, statistic, values.shape, (20, 30))
        got = raster.Place.process(kwargs, {"values": values, "no_data_value": -1})
        expected, _ = R.place_warp(values, -1, kwargs)
        np.testing.assert_array_equal(np.asarray(got["values"]), expected)
    kwargs = place_kwargs(coordinates, "mean", values.shape, (20, 30))
    with pytest.raises(NotImplementedError):
        raster.Place.process(kwargs, {"values": values, "no_data_value": -1})


@pytest.mark.parametrize("statistic", ["mean", "argmax"])
def test_place_group_mode(statistic):
    rng = np.random.default_rng(4)
    data = rng.uniform(1, 100, (1, 6, 8)).astype("f4")
    nodata = workloads.F32_MAX
    data[rng.random(data.shape) < 0.3] = nodata
    src = raster.MemorySource(data, nodata, workloads.PROJECTION, pixel_size=1.0, pixel_origin=(10, 26))
    coordinates = [(float(x), float(y)) for x, y in zip(rng.uniform(0, 12, 12), rng.uniform(0, 12, 12))]
    fine = dict(mode="vals", bbox=(4, 4, 8, 8), width=2, height=2, projection=workloads.PROJECTION)
    view = raster.Place(src, workloads.PROJECTION, (12.0, 22.0), coordinates, statistic)
    plan = view.get_sources_and_requests(**fine)
    assert plan[0][0]["mode"] == "group" and len(plan) > 9
    stack = [(np.asarray(s.get_data(**r)["values"]), nodata) for s, r in plan[1:]]
    expected, _ = R.reduce_rasters(stack, statistic)
    assert_stat(view.get_data(**fine)["values"], expected, statistic, len(stack))

