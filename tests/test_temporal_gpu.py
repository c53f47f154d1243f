"""TemporalAggregate / Cumulative kernels against the oracle (NumPy nan-reductions
in the reference's working dtype)."""
from datetime import datetime, timedelta

import numpy as np
import pytest

from dask_geomodeling_b200 import _native, raster, workloads
from oracle import raster as R

pytestmark = pytest.mark.gpu


def stack(dtype, frames=11, seed=0, shape=(19, 45)):
    rng = np.random.default_rng(seed)
    nodata = R.dtype_max(dtype)
    if np.dtype(dtype).kind == "f":
        values = rng.uniform(0, 100, (frames,) + shape).astype(dtype)
    else:
        values = rng.integers(0, 100, (frames,) + shape).astype(dtype)
    values[rng.random(values.shape) < 0.3] = nodata
    values[:, 0, 0] = nodata  # a pixel without any data
    return values, nodata


def times(n):
    return [datetime(2000, 1, 1) + timedelta(hours=i) for i in range(n)]


# (19, 45): 855 cells, no whole 16-byte pixel groups -> one pixel per thread (VEC = 1);
# (16, 48): 768 cells -> 16-byte loads, several pixels per thread
SHAPES = [(19, 45), (16, 48)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype", ["f4", "u1", "i2", "i4", "f8"])
@pytest.mark.parametrize("statistic", ["sum", "count", "min", "max", "mean", "median", "std", "var", "p90", "p25"])
def test_aggregate_all_frames(dtype, statistic, shape):
    values, nodata = stack(dtype, shape=shape)
    name, q = (statistic, None) if not statistic.startswith("p") else ("percentile", float(statistic[1:]))
    expected, expected_nodata = R.temporal_aggregate(values, nodata, name, [range(len(values))], q)
    kwargs = dict(mode="vals", start=times(11)[-1], stop=None, frequency=None, timezone=None,
                  closed=None, label=None, dtype=expected.dtype.str, statistic=statistic)
    got = raster.TemporalAggregate.process(kwargs, {"time": times(11)},
                                           {"values": values, "no_data_value": nodata})
    out = got["values"]
    assert out.dtype == expected.dtype and out.shape == expected.shape
    assert got["no_data_value"] == expected_nodata
    # sequential-in-t accumulation, NumPy's nanvar two-pass form and nanpercentile's
    # linear interpolation in the working dtype: bit-exact for every statistic
    np.testing.assert_array_equal(out, expected)


@pytest.mark.parametrize("dtype", ["f4", "u1"])
@pytest.mark.parametrize("statistic", ["sum", "max", "mean"])
def test_aggregate_resampled(dtype, statistic):
    values, nodata = stack(dtype, frames=10)
    bins = [[0, 1, 2, 3], [4, 5, 6, 7], [8, 9]]
    expected, _ = R.temporal_aggregate(values, nodata, statistic, bins)
    kwargs = dict(mode="vals", start=datetime(2000, 1, 1), stop=datetime(2000, 1, 1, 8),
                  frequency="4h", timezone="UTC", closed="left", label="left",
                  dtype=expected.dtype.str, statistic=statistic)
    got = raster.TemporalAggregate.process(kwargs, {"time": times(10)},
                                           {"values": values, "no_data_value": nodata})
    np.testing.assert_array_equal(got["values"], expected)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype", ["f4", "u1", "i4", "f8"])
@pytest.mark.parametrize("statistic", ["sum", "count"])
@pytest.mark.parametrize("frequency", [None, "4h"])
def test_cumulative(dtype, statistic, frequency, shape):
    values, nodata = stack(dtype, frames=10, shape=shape)
    ts = times(10)
    if frequency is None:
        bins = [list(range(10))]
    else:  # closed right / label right: (.., 0h], (0h, 4h], (4h, 8h], (8h, 12h]
        bins = [[0], [1, 2, 3, 4], [5, 6, 7, 8], [9]]
    mask = np.array([2 <= i <= 8 for i in range(10)])
    expected, expected_nodata = R.cumulative(values, nodata, statistic, bins, mask)
    kwargs = dict(mode="vals", start=ts[2], stop=ts[8], frequency=frequency,
                  timezone=None if frequency is None else "UTC", closed="right", label="right",
                  dtype=expected.dtype.str, statistic=statistic)
    got = raster.Cumulative.process(kwargs, {"time": ts}, {"values": values, "no_data_value": nodata})
    assert got["values"].dtype == expected.dtype
    np.testing.assert_array_equal(got["values"], expected)
    assert got["no_data_value"] == expected_nodata


def test_temporal_aggregate_view():
    values, nodata = stack("f4", frames=12, shape=(32, 32))
    src = workloads.source(values, nodata, time_first=0, time_delta=3600 * 1000)
    for statistic in ("sum", "max"):
        view = raster.TemporalAggregate(src, None, statistic)
        got = view.get_data(**workloads.request(32, 32))
        expected, _ = R.temporal_aggregate(values, nodata, statistic, [range(12)])
        np.testing.assert_array_equal(got["values"], expected)
    view = raster.TemporalAggregate(src, "6h", "sum")
    got = view.get_data(**workloads.request(32, 32, start=datetime(1970, 1, 1), stop=datetime(1970, 1, 2)))
    expected, _ = R.temporal_aggregate(values, nodata, "sum", [range(0, 6), range(6, 12)])
    np.testing.assert_array_equal(got["values"], expected)


def offset_on_device(values):
    """``values`` on the device one element past a 16-byte aligned base: the plane is whole
    16-byte groups, the pointer is not."""
    flat = np.concatenate([np.zeros(1, values.dtype), values.ravel()])
    base = _native.DeviceArray.from_host(flat)
    view = _native.DeviceArray(values.shape, values.dtype, ptr=base.ptr + values.dtype.itemsize, owner=base)
    assert view.ptr % 16 != 0
    return view


@pytest.mark.parametrize("statistic", ["sum", "mean", "std"])
def test_aggregate_unaligned_source(statistic):
    values, nodata = stack("f4", shape=(16, 48))
    expected, _ = R.temporal_aggregate(values, nodata, statistic, [range(11)])
    kwargs = dict(mode="vals", start=times(11)[-1], stop=None, frequency=None, timezone=None,
                  closed=None, label=None, dtype=expected.dtype.str, statistic=statistic)
    got = raster.TemporalAggregate.process(kwargs, {"time": times(11)},
                                           {"values": offset_on_device(values), "no_data_value": nodata})
    np.testing.assert_array_equal(np.asarray(got["values"]), expected)


def test_cumulative_unaligned_source():
    values, nodata = stack("f4", frames=10, shape=(16, 48))
    ts = times(10)
    expected, _ = R.cumulative(values, nodata, "sum", [range(10)], np.ones(10, bool))
    kwargs = dict(mode="vals", start=ts[0], stop=ts[-1], frequency=None, timezone=None,
                  closed="right", label="right", dtype=expected.dtype.str, statistic="sum")
    got = raster.Cumulative.process(kwargs, {"time": ts},
                                    {"values": offset_on_device(values), "no_data_value": nodata})
    np.testing.assert_array_equal(np.asarray(got["values"]), expected)


@pytest.mark.parametrize("statistic", ["median", "p90"])
def test_aggregate_long_bin_float64(statistic):
    # 600 frames of an int32 source: float64 working dtype, 1024 sort slots per pixel
    values, nodata = stack("i4", frames=600)
    name, q = (statistic, None) if not statistic.startswith("p") else ("percentile", float(statistic[1:]))
    expected, _ = R.temporal_aggregate(values, nodata, name, [range(600)], q)
    kwargs = dict(mode="vals", start=times(600)[-1], stop=None, frequency=None, timezone=None,
                  closed=None, label=None, dtype=expected.dtype.str, statistic=statistic)
    got = raster.TemporalAggregate.process(kwargs, {"time": times(600)},
                                           {"values": values, "no_data_value": nodata})
    assert expected.dtype == np.float64
    np.testing.assert_array_equal(got["values"], expected)


def test_sum_int64_past_2_53():
    # int64 samples are added in float64, as NumPy adds them: 3 * (2**53 + 1) -> 3 * 2**53
    values = np.full((3, 16, 48), 2 ** 53 + 1, dtype=np.int64)
    nodata = R.dtype_max(np.int64)
    expected, _ = R.temporal_aggregate(values, nodata, "sum", [range(3)])
    assert expected[0, 0, 0] == 3 * 2 ** 53
    kwargs = dict(mode="vals", start=times(3)[-1], stop=None, frequency=None, timezone=None,
                  closed=None, label=None, dtype=expected.dtype.str, statistic="sum")
    got = raster.TemporalAggregate.process(kwargs, {"time": times(3)},
                                           {"values": values, "no_data_value": nodata})
    np.testing.assert_array_equal(got["values"], expected)
