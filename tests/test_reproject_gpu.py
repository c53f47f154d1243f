"""Requests in another CRS than their data (EPSG:4326, EPSG:3857, WGS 84 UTM zones): the device
warp (gm_warp_nn) against the NumPy restatement in oracle/warp.py, and the geometry paths that
transform vertices (AggregateRaster, MemoryGeometrySource)."""
import os
from datetime import datetime

import numpy as np
import pytest

from dask_geomodeling_b200 import _native, crs, geometry, geotiff, raster, utils
from dask_geomodeling_b200._compat import config
from dask_geomodeling_b200.raster import MemorySource, RasterFileSource, sources
from oracle import warp as oracle_warp

pytestmark = pytest.mark.gpu

CRSS = ["EPSG:4326", "EPSG:3857", "EPSG:32631", "EPSG:32733"]
PAIRS = [(s, d) for s in CRSS for d in CRSS if s != d]
DTYPES = ["u1", "i2", "i4", "f4", "f8"]
SOURCE_BOX = (6.5, -1.5, 11.5, 1.5)           # lon / lat; UTM 31N and 33S both cover it
REQUEST_BOX = (5.5, -2.5, 10.5, 1.0)          # partly outside the source
OUTSIDE_BOX = (20.0, 20.0, 21.0, 21.0)
TIMES = dict(start=datetime(1970, 1, 1), stop=datetime(1970, 1, 1, 0, 0, 10))


def box_in(projection, geo_box):
    return utils.Extent(geo_box, "EPSG:4326").transformed(projection).bbox


def make_source(projection, dtype, shape=(3, 160, 200), seed=0):
    n, h, w = shape
    x1, y1, x2, y2 = box_in(projection, SOURCE_BOX)
    rng = np.random.default_rng(seed)
    data = rng.integers(0, 99, shape).astype(dtype)
    nodata = 99
    data[rng.random(shape) < 0.05] = nodata
    if np.dtype(dtype).kind == "f":
        data[rng.random(shape) < 0.05] = np.nan
    source = MemorySource(data, nodata, projection, pixel_size=((x2 - x1) / w, (y2 - y1) / h),
                          pixel_origin=(x1, y2), time_first=0, time_delta=1000 if n > 1 else None)
    return source, data


def check(source, data, projection, bbox, width, height, max_edge=None):
    misses = _native.STATS.get("warp_window_misses", 0)
    got = source.get_data(mode="vals", projection=projection, bbox=bbox, width=width, height=height,
                          **TIMES)
    assert _native.STATS.get("warp_window_misses", 0) == misses
    values = np.asarray(got["values"])
    expected, near = oracle_warp.warp_nn(data, tuple(source.geo_transform), source.projection,
                                         source.no_data_value, bbox, height, width, projection)
    assert values.shape == expected.shape and values.dtype == expected.dtype
    differ = (values != expected).any(axis=0)
    assert not (differ & ~near).any(), "{} cells differ away from cell edges".format((differ & ~near).sum())
    assert differ.sum() <= (max_edge if max_edge is not None else max(2, values[0].size // 10000))
    return values


@pytest.mark.parametrize("size", [(300, 210), (90, 60)], ids=["finer", "coarser"])
@pytest.mark.parametrize("pair", PAIRS, ids=["{}->{}".format(s[5:], d[5:]) for s, d in PAIRS])
def test_warp_equals_oracle(pair, size):
    src_proj, dst_proj = pair
    dtype = DTYPES[PAIRS.index(pair) % len(DTYPES)]
    source, data = make_source(src_proj, dtype)
    width, height = size
    values = check(source, data, dst_proj, box_in(dst_proj, REQUEST_BOX), width, height)
    nodata = source.no_data_value
    assert (values == nodata).any() and (values != nodata).any()
    outside = check(source, data, dst_proj, box_in(dst_proj, OUTSIDE_BOX), 20, 20)
    assert (outside == nodata).all()


@pytest.mark.parametrize("dtype", DTYPES)
def test_warp_dtypes_utm_zone_to_zone(dtype):
    source, data = make_source("EPSG:32733", dtype, seed=3)
    check(source, data, "EPSG:32631", box_in("EPSG:32631", REQUEST_BOX), 170, 130)


@pytest.mark.parametrize("pair", [("EPSG:4326", "EPSG:3857"), ("EPSG:32631", "EPSG:4326")])
def test_resident_and_upload_agree(pair):
    source, data = make_source(pair[0], "f4")
    request = dict(mode="vals", projection=pair[1], bbox=box_in(pair[1], REQUEST_BOX), width=250,
                   height=200, **TIMES)
    uploaded = np.asarray(source.get_data(**request)["values"])
    with config.set({"geomodeling.device-cache-bytes": 1 << 30}):
        resident = np.asarray(source.get_data(**request)["values"])
        again = np.asarray(source.get_data(**request)["values"])
    np.testing.assert_array_equal(uploaded, resident)
    np.testing.assert_array_equal(resident, again)


def test_poles_into_web_mercator_are_no_data():
    data = np.arange(180 * 360, dtype="f4").reshape(180, 360)
    source = MemorySource(data, -1.0, "EPSG:4326", pixel_size=1.0, pixel_origin=(-180.0, 90.0))
    # columns beyond +-pi R map beyond +-180 degrees (longitudes are not wrapped)
    values = check(source, data[np.newaxis], "EPSG:3857", (-2.5e7, -3e7, 2.5e7, 3e7), 100, 150)
    assert (values[0, :, 0] == -1).all() and (values[0, :, -1] == -1).all()
    assert (values[0, :, 50] != -1).all()
    # and a geographic request reaching over a pole into a Web Mercator source
    merc, merc_data = make_source("EPSG:3857", "f8")
    values = check(merc, merc_data, "EPSG:4326", (0.0, 80.0, 10.0, 100.0), 10, 20)
    assert (values[:, :10] == merc.no_data_value).all()


def test_geotiff_source_equals_memory_source(tmp_path):
    source, data = make_source("EPSG:4326", "i2", shape=(2, 160, 200))
    path = os.path.join(str(tmp_path), "geo.tif")
    geotiff.write_geotiff(path, data, tuple(source.geo_transform), "EPSG:4326", 99)
    with config.set({"geomodeling.root": str(tmp_path)}):
        file_source = RasterFileSource("geo.tif", time_first=0, time_delta=1000)
        for projection in ("EPSG:3857", "EPSG:32631"):
            request = dict(mode="vals", projection=projection, bbox=box_in(projection, REQUEST_BOX),
                           width=230, height=170, **TIMES)
            from_file = file_source.get_data(**request)
            from_memory = source.get_data(**request)
            np.testing.assert_array_equal(np.asarray(from_file["values"]), np.asarray(from_memory["values"]))
            assert from_file["no_data_value"] == from_memory["no_data_value"]


def test_fused_chain_on_a_warped_source():
    source, data = make_source("EPSG:32631", "f4", shape=(1, 160, 200))
    projection, width, height = "EPSG:3857", 240, 180
    bbox = box_in(projection, REQUEST_BOX)
    warped, near = oracle_warp.warp_nn(data, tuple(source.geo_transform), source.projection,
                                       source.no_data_value, bbox, height, width, projection)
    # the oracle's warped raster as a source aligned with the request: same chain, no warp
    x1, y1, x2, y2 = bbox
    aligned = MemorySource(warped, source.no_data_value, projection,
                           pixel_size=((x2 - x1) / width, (y2 - y1) / height), pixel_origin=(x1, y2))
    request = dict(mode="vals", projection=projection, bbox=bbox, width=width, height=height)
    got = raster.Clip(source * 2.0 + 1.0, source > 20.0).get_data(**request)
    expected = raster.Clip(aligned * 2.0 + 1.0, aligned > 20.0).get_data(**request)
    g, e = np.asarray(got["values"]), np.asarray(expected["values"])
    assert got["no_data_value"] == expected["no_data_value"]
    np.testing.assert_array_equal(g[:, ~near], e[:, ~near])


def _squares(centres, half):
    return [[(x - half, y - half), (x + half, y - half), (x + half, y + half), (x - half, y + half)]
            for x, y in centres]


def test_aggregate_raster_with_polygons_in_another_crs():
    utm = "EPSG:32631"
    values = np.random.default_rng(5).random((1, 200, 200)).astype("f4")
    x0, y0 = 500000.0, 200000.0
    src = MemorySource(values, -1.0, utm, pixel_size=100.0, pixel_origin=(x0, y0 + 20000.0))
    rng = np.random.default_rng(6)
    lonlat = np.stack([rng.uniform(3.02, 3.15, 40), rng.uniform(1.83, 1.97, 40)], 1)
    polygons = _squares(lonlat, 0.01)
    window = utils.box(2.9, 1.7, 3.3, 2.1)
    for statistic in ("sum", "mean", "max", "median"):
        view = geometry.AggregateRaster(
            geometry.MemoryGeometrySource(polygons, [{"id": i} for i in range(40)], projection="EPSG:4326"),
            raster=src, statistic=statistic)
        got = view.get_data(mode="intersects", projection="EPSG:4326", geometry=window)
        transformed = [utils.shapely_transform(utils.Polygon(p), "EPSG:4326", utm) for p in polygons]
        direct = geometry.AggregateRaster(
            geometry.MemoryGeometrySource(transformed, [{"id": i} for i in range(40)], projection=utm),
            raster=src, statistic=statistic)
        expected = direct.get_data(mode="intersects", projection=utm,
                                   geometry=utils.Extent(window.bounds, "EPSG:4326").transformed(utm).as_geometry())
        assert len(got["features"]) == 40
        np.testing.assert_array_equal(got["features"]["agg"].values, expected["features"]["agg"].values)


def test_rasterize_memory_geometry_in_another_crs():
    rng = np.random.default_rng(7)
    lonlat = np.stack([rng.uniform(4.0, 6.0, 30), rng.uniform(50.0, 52.0, 30)], 1)
    polygons = _squares(lonlat, 0.1)
    props = [{"id": i, "value": float(i)} for i in range(30)]
    bbox = box_in("EPSG:3857", (3.8, 49.8, 6.2, 52.2))
    request = dict(mode="vals", projection="EPSG:3857", bbox=bbox, width=300, height=400)
    got = raster.Rasterize(geometry.MemoryGeometrySource(polygons, props, projection="EPSG:4326"),
                           "value").get_data(**request)
    transformed = [utils.shapely_transform(utils.Polygon(p), "EPSG:4326", "EPSG:3857") for p in polygons]
    expected = raster.Rasterize(geometry.MemoryGeometrySource(transformed, props, projection="EPSG:3857"),
                                "value").get_data(**request)
    np.testing.assert_array_equal(np.asarray(got["values"]), np.asarray(expected["values"]))
    assert (np.asarray(got["values"]) != got["no_data_value"]).any()


def test_extent_and_point_requests():
    merc, merc_data = make_source("EPSG:3857", "f4", shape=(1, 160, 200))
    utm, utm_data = make_source("EPSG:32733", "i4", shape=(1, 160, 200))
    for source in (merc, utm):
        native = utils.Extent(source.geo_transform.get_bbox((0, 0), source.data.shape[1:]), source.projection)
        np.testing.assert_allclose(source.extent, native.transformed("EPSG:4326").bbox)
        x1, y1, x2, y2 = source.extent
        assert x1 < 7.0 and x2 > 11.0 and y1 < -1.0 and y2 > 1.0
    rng = np.random.default_rng(8)
    for source, data in ((merc, merc_data), (utm, utm_data)):
        for lon, lat in zip(rng.uniform(6.0, 12.0, 20), rng.uniform(-2.0, 2.0, 20)):
            got = source.get_data(mode="vals", projection="EPSG:4326", bbox=(lon, lat, lon, lat), width=1, height=1)
            x, y = crs.transform([[lon, lat]], "EPSG:4326", source.projection)[0]
            rows, cols = source.geo_transform.get_indices([[x, y]])
            i, j = int(rows[0]), int(cols[0])
            inside = 0 <= i < data.shape[1] and 0 <= j < data.shape[2]
            expected = data[0, i, j] if inside else source.no_data_value
            if not np.isfinite(expected):
                expected = source.no_data_value
            assert got["values"][0, 0, 0] == expected


def test_window_miss_repeats_with_the_whole_source(monkeypatch):
    # a 600 km UTM request bows over the corners' latitudes by several source rows
    data = np.random.default_rng(9).random((2, 400, 500)).astype("f4")
    source = MemorySource(data, -1.0, "EPSG:4326", pixel_size=0.02, pixel_origin=(-2.0, 46.0),
                          time_first=0, time_delta=1000)
    bbox, width, height = (200000.0, 4400000.0, 800000.0, 5000000.0), 300, 300
    outline = sources.request_outline
    monkeypatch.setattr(sources, "request_outline", lambda b, n=1: outline(b, 1))
    monkeypatch.setattr(sources, "WINDOW_MARGIN", 0)
    before = _native.STATS.get("warp_window_misses", 0)
    got = source.get_data(mode="vals", projection="EPSG:32631", bbox=bbox, width=width, height=height, **TIMES)
    assert _native.STATS.get("warp_window_misses", 0) == before + 1
    expected, near = oracle_warp.warp_nn(data, tuple(source.geo_transform), "EPSG:4326", -1.0, bbox,
                                         height, width, "EPSG:32631")
    differ = (np.asarray(got["values"]) != expected).any(axis=0)
    assert not (differ & ~near).any()


def test_full_size_request_on_sampled_windows():
    n = 16384
    data = np.random.default_rng(10).random((1, n, n), dtype=np.float32)
    x1, y1, x2, y2 = box_in("EPSG:32631", (1.0, 40.0, 5.0, 44.0))
    source = MemorySource(data, -1.0, "EPSG:32631", pixel_size=((x2 - x1) / n, (y2 - y1) / n),
                          pixel_origin=(x1, y2))
    bbox = box_in("EPSG:3857", (1.2, 40.2, 4.8, 43.8))
    got = np.asarray(source.get_data(mode="vals", projection="EPSG:3857", bbox=bbox, width=n, height=n)["values"])
    assert got.shape == (1, n, n)
    total_edge = 0
    for r0, c0 in ((0, 0), (n - 256, n - 256), (n // 2, n // 3), (n // 5, n - 300)):
        rows, cols = slice(r0, r0 + 256), slice(c0, c0 + 256)
        expected, near = oracle_warp.warp_nn(data, tuple(source.geo_transform), "EPSG:32631", -1.0, bbox,
                                             n, n, "EPSG:3857", rows=rows, cols=cols)
        differ = (got[:, rows, cols] != expected).any(axis=0)
        assert not (differ & ~near).any()
        total_edge += int(differ.sum())
    assert total_edge <= 10
