"""AggregateRaster: zonal statistics of a raster per geometry, on the GPU.

Drop-in for the reference's geometry/aggregate.py (:255-646).  The reference
rasterises the geometries bucket by bucket with GDAL and then runs
scipy.ndimage / measurements.percentile over the label raster
(:113-203).  Here each geometry is scan-converted on the GPU with GDAL's
pixel-centre rule and the statistic is taken directly under its spans
(csrc/gm_polygons.cu): no label raster, no buckets, and overlapping geometries
are naturally independent.  ``bucketize`` is kept because it is public API in
the reference (tests/test_aggregate_raster.py:646-656); the CUDA path does not
need it.
"""
import ctypes
from collections import defaultdict
from math import ceil, floor, log, sqrt

import numpy as np
import pandas as pd

from .. import _native, utils
from .._compat import config
from ..raster import RasterBlock
from .base import GeometryBlock

__all__ = ["AggregateRaster", "AggregateRasterAboveThreshold"]

_STAT_CODES = {"sum": 0, "count": 1, "min": 2, "max": 3, "mean": 4, "median": 5, "percentile": 8}


def calculate_level_and_cells(bbox):
    """(level, cells): the <= 4 cells of a sparse grid with cell size 0.5**level
    that the bbox touches; level is chosen so that the bbox fits in one cell size."""
    x1, y1, x2, y2 = bbox
    level = -ceil(log(max(x2 - x1, y2 - y1), 2))
    size = 0.5 ** level
    j1, j2 = floor(x1 / size), floor(x2 / size)
    i1, i2 = floor(y1 / size), floor(y2 / size)
    return level, {(i1, j1), (i1, j2), (i2, j1), (i2, j2)}


def bucketize(bboxes):
    """Partition bbox indices into lists of mutually disjoint boxes (greedy, per
    size level) -- reference geometry/aggregate.py:75-110."""
    per_level = defaultdict(list)  # level -> [(occupied cells, indices)]
    for index, bbox in enumerate(bboxes):
        level, cells = calculate_level_and_cells(bbox)
        for occupied, indices in per_level[level]:
            if not (occupied & cells):
                occupied.update(cells)
                indices.append(index)
                break
        else:
            per_level[level].append((set(cells), [index]))
    return [indices for buckets in per_level.values() for _, indices in buckets]


def _frame_descriptor(values, frame):
    """GmArray of frame ``frame`` of a (t, h, w) host or device array."""
    t, h, w = values.shape
    desc = _native.GmArray()
    offset = frame * h * w * values.dtype.itemsize
    if _native.is_device(values):
        desc.data, desc.space = values.ptr + offset, _native.GM_DEVICE
    else:
        desc.data, desc.space = values.ctypes.data + offset, _native.GM_HOST
    desc.dtype = _native.dtype_code(values.dtype)
    desc.shape[0], desc.shape[1], desc.shape[2] = 1, h, w
    return desc


def _read_cells(values, rows, cols):
    """values[:, rows, cols] as a host array, for host or device rasters."""
    if not _native.is_device(values):
        return values[:, rows, cols]
    t, h, w = values.shape
    out = np.empty((t, len(rows)), dtype=values.dtype)
    item = values.dtype.itemsize
    lib = _native.lib()
    for k, (i, j) in enumerate(zip(rows, cols)):
        for frame in range(t):
            cell = np.empty(1, dtype=values.dtype)
            _native.check(lib.gm_memcpy_d2h(cell.ctypes.data, values.ptr + ((frame * h + int(i)) * w + int(j)) * item,
                                            item, _native.current_stream()))
            out[frame, k] = cell[0]
    return out


class _LazyTransformed(object):
    """``geometries[i]`` transformed from ``src`` to ``dst`` on access."""

    def __init__(self, geometries, src, dst):
        self.geometries, self.src, self.dst = geometries, src, dst

    def __getitem__(self, i):
        return utils.shapely_transform(self.geometries[i], self.src, self.dst)


def aggregate_polygons(geometries, values, no_data_value, agg_bbox, agg_srs, threshold_values,
                       statistic, percentile):
    """Statistic of ``values`` (t, h, w) under every geometry.

    Returns (float32 array (t, n), indices of geometries covering no cell centre)
    like the reference (geometry/aggregate.py:113-203)."""
    from ..raster._program import sentinel

    depth, height, width = values.shape
    # a ready-made PolygonSoup is accepted so that callers can reuse it between requests
    soup = geometries if isinstance(geometries, utils.PolygonSoup) else utils.PolygonSoup(list(geometries))
    if depth > 1:
        soup.to_device()  # several frames: upload the polygons once
    polys = soup.as_struct()
    geo = (ctypes.c_double * 6)(*utils.GeoTransform.from_bbox(agg_bbox, height, width))
    n = soup.n_polygons
    # page-locked result buffers: the library's device-to-host copies are then plain DMA
    # (one row per frame; the library writes every entry of `out` and `covered`)
    agg = _native.pinned_empty((depth, n), np.float32)
    covered = _native.pinned_empty((n,), np.int64)
    if n == 0 or depth == 0:
        covered[:] = 0
    s = sentinel(values.dtype, no_data_value)
    holder, nodata_ptr = _native.scalar_ptr(0 if s is None else s, values.dtype)
    thresholds = None
    if threshold_values is not None:
        thresholds = np.ascontiguousarray(threshold_values, dtype=np.float32)
    if not _native.is_device(values):
        values = np.ascontiguousarray(values)
    lib = _native.lib()
    for frame in range(depth):
        desc = _frame_descriptor(values, frame)
        out = agg[frame]
        _native.check(lib.gm_zonal_stats(
            ctypes.byref(desc), nodata_ptr, int(s is not None), ctypes.byref(polys), geo,
            _STAT_CODES[statistic], float(percentile or 0.0),
            None if thresholds is None else thresholds.ctypes.data, 0, height,
            out.ctypes.data, covered.ctypes.data, None, _native.current_stream()))
    return agg, np.nonzero(covered == 0)[0].tolist()


def aggregate_points(points, values, no_data_value, agg_bbox, threshold_values, statistic):
    """Value of the cell that contains each point (geometry/aggregate.py:206-252)."""
    _, height, width = values.shape
    gt = utils.GeoTransform.from_bbox(agg_bbox, height, width)
    xy = np.array([(p.x, p.y) for p in points], dtype=np.float64).reshape(-1, 2)
    rows, cols = gt.get_indices(xy)
    cells = _read_cells(values, np.clip(rows, 0, height - 1), np.clip(cols, 0, width - 1))
    active = cells != no_data_value
    if threshold_values is not None:
        thresholds = np.asarray(threshold_values)[np.newaxis, :]
        thresholds = np.broadcast_to(thresholds, cells.shape)
        valid = ~np.isnan(thresholds)
        active = active & valid
        active[valid] &= cells[valid] >= thresholds[valid]
    agg = cells.astype("f4")
    agg[~active] = np.nan
    if statistic == "count":
        agg[active] = 1.0
    return agg


class AggregateRaster(GeometryBlock):
    """Statistic of ``raster`` for every geometry of ``source``, added as column
    ``column_name``.

    Cells whose centre lies inside a polygon take part; geometries that cover no
    cell centre are sampled at their centroid.  statistic: sum, count, min, max,
    mean, median or p<percentile> (reference: geometry/aggregate.py:255-587).
    """

    STATISTICS = {
        "sum": {"extensive": True}, "count": {"extensive": True}, "min": {"extensive": False},
        "max": {"extensive": False}, "mean": {"extensive": False}, "median": {"extensive": False},
        "percentile": {"extensive": False},
    }

    def __init__(self, source, raster, statistic="sum", projection=None, pixel_size=None,
                 max_pixels=None, column_name="agg", auto_pixel_size=False, *args):
        if not isinstance(source, GeometryBlock):
            raise TypeError("'{}' object is not allowed".format(type(source)))
        if not isinstance(raster, RasterBlock):
            raise TypeError("'{}' object is not allowed".format(type(raster)))
        if not isinstance(statistic, str):
            raise TypeError("'{}' object is not allowed".format(type(statistic)))
        statistic, percentile = utils.parse_percentile_statistic(statistic.lower())
        if percentile:
            statistic = "p{0}".format(percentile)
        elif statistic not in self.STATISTICS or statistic == "percentile":
            raise ValueError("Unknown statistic '{}'".format(statistic))
        if projection is None:
            projection = raster.projection
        if not isinstance(projection, str):
            raise TypeError("'{}' object is not allowed".format(type(projection)))
        if pixel_size is None:
            geo_transform = raster.geo_transform
            if geo_transform is None:
                raise ValueError(
                    "Cannot get the pixel_size from the source raster. Please provide a pixel_size."
                )
            pixel_size = min(abs(float(geo_transform[1])), abs(float(geo_transform[5])))
        else:
            pixel_size = abs(float(pixel_size))
        if pixel_size == 0.0:
            raise ValueError("Pixel size cannot be 0")
        if max_pixels is not None:
            max_pixels = int(max_pixels)
        if not isinstance(auto_pixel_size, bool):
            raise TypeError("'{}' object is not allowed".format(type(auto_pixel_size)))
        super(AggregateRaster, self).__init__(
            source, raster, statistic, projection, pixel_size, max_pixels, column_name,
            auto_pixel_size, *args)

    source = property(lambda self: self.args[0])
    raster = property(lambda self: self.args[1])
    statistic = property(lambda self: self.args[2])
    projection = property(lambda self: self.args[3])
    pixel_size = property(lambda self: self.args[4])
    max_pixels = property(lambda self: self.args[5])
    column_name = property(lambda self: self.args[6])
    auto_pixel_size = property(lambda self: self.args[7])

    @property
    def columns(self):
        return self.source.columns | {self.column_name}

    def get_sources_and_requests(self, **request):
        if request.get("mode") == "extent":
            return [(self.source, request), (None, None), ({"mode": "extent"}, None)]
        req_srs, agg_srs = request["projection"], self.projection
        extent = self.source.get_data(**dict(request, mode="extent"))["extent"]
        if extent is None:
            return [(None, None), (None, None), ({"empty": True, "projection": req_srs}, None)]
        x1, y1, x2, y2 = utils.Extent(extent, req_srs).transformed(agg_srs).bbox

        pixel_size = self.pixel_size
        required = int(((x2 - x1) * (y2 - y1)) / (pixel_size ** 2))
        max_pixels = self.max_pixels
        if max_pixels is None:
            max_pixels = config.get("geomodeling.raster-limit")
        if required > max_pixels:
            if not self.auto_pixel_size:
                raise RuntimeError(
                    "The required raster size for the aggregation exceeded "
                    "the maximum ({} > {})".format(required, max_pixels))
            pixel_size *= ceil(sqrt(required / max_pixels))  # integer multiples only

        # snap outwards to multiples of the pixel size: no sub-pixel shifts
        x1, y1 = floor(x1 / pixel_size) * pixel_size, floor(y1 / pixel_size) * pixel_size
        x2, y2 = ceil(x2 / pixel_size) * pixel_size, ceil(y2 / pixel_size) * pixel_size
        width = max(int((x2 - x1) / pixel_size), 1)
        height = max(int((y2 - y1) / pixel_size), 1)
        if width == 1 and height == 1:
            bbox = ((x1 + x2) / 2, (y1 + y2) / 2) * 2   # a true point request
        else:
            bbox = (x1, y1, x2, y2)
        raster_request = {
            "mode": "vals", "projection": agg_srs, "start": request.get("start"),
            "stop": request.get("stop"), "aggregation": None, "bbox": bbox, "width": width,
            "height": height,
        }
        if "time_resolution" in request:
            raster_request["time_resolution"] = request["time_resolution"]
        process_kwargs = {
            "mode": request.get("mode", "intersects"), "pixel_size": self.pixel_size,
            "agg_srs": agg_srs, "req_srs": req_srs, "actual_pixel_size": pixel_size,
            "statistic": self.statistic, "result_column": self.column_name,
            "agg_bbox": (x1, y1, x2, y2),
        }
        return [(self.source, request), (self.raster, raster_request), (process_kwargs, None)]

    @staticmethod
    def process(geom_data, raster_data, process_kwargs):
        if process_kwargs.get("empty"):
            return {"features": pd.DataFrame([]), "projection": process_kwargs["projection"]}
        if process_kwargs["mode"] == "extent":
            return geom_data
        features = geom_data["features"]
        if len(features) == 0:
            return geom_data
        result = features.copy()
        req_srs, agg_srs = process_kwargs["req_srs"], process_kwargs["agg_srs"]
        column = features["geometry"]
        soup = None
        if hasattr(column, "to_crs"):
            agg_geometries = list(column.to_crs(agg_srs))
        elif utils.same_projection(req_srs, agg_srs):
            agg_geometries = column.values
            from .sources import prepared_soup_of

            prepared = prepared_soup_of(features)
            if prepared is not None:
                # the frame still holds the source's geometries: reuse their CSR form
                # (kept resident in HBM when it is the source's full set)
                full, positions, _ = prepared
                if len(positions) == full.n_polygons:
                    soup = full.to_device()
                else:
                    soup = full.subset(positions)
        else:
            # the vertices are transformed in one vectorised call on the CSR form; geometry
            # objects in the raster's CRS are built only for the centroid fallback below
            from .sources import prepared_soup_of

            prepared = prepared_soup_of(features)
            if prepared is not None:
                full, positions, _ = prepared
                soup = full if len(positions) == full.n_polygons else full.subset(positions)
            else:
                soup = utils.PolygonSoup(list(column.values))
            soup = soup.transformed(req_srs, agg_srs)
            agg_geometries = _LazyTransformed(column.values, req_srs, agg_srs)

        statistic, percentile = utils.parse_percentile_statistic(process_kwargs["statistic"])
        extensive = AggregateRaster.STATISTICS[statistic]["extensive"]
        result_column = process_kwargs["result_column"]
        threshold_name = process_kwargs.get("threshold_name")
        thresholds = features[threshold_name].values.astype("f4") if threshold_name else None

        values = no_data_value = None
        if raster_data is not None:
            values, no_data_value = raster_data["values"], raster_data["no_data_value"]
        if values is None:
            result[result_column] = 0 if extensive else np.nan
            return {"features": result, "projection": req_srs}

        agg, no_cells = aggregate_polygons(
            soup if soup is not None else agg_geometries, values, no_data_value,
            process_kwargs["agg_bbox"], agg_srs, thresholds, statistic, percentile)
        if no_cells:
            # geometries that touch no cell centre are sampled at their centroid
            agg[:, no_cells] = aggregate_points(
                [agg_geometries[i].centroid for i in no_cells], values, no_data_value,
                process_kwargs["agg_bbox"], None if thresholds is None else thresholds[no_cells],
                statistic)
        pixel_size, actual = process_kwargs["pixel_size"], process_kwargs["actual_pixel_size"]
        if extensive:
            agg[~np.isfinite(agg)] = 0
            if actual != pixel_size:
                agg *= (actual / pixel_size) ** 2
        else:
            agg[~np.isfinite(agg)] = np.nan
        if values.shape[0] == 1:
            result[result_column] = agg[0]
        else:
            result[result_column] = [[x] for x in agg.T]
        return {"features": result, "projection": req_srs}


class AggregateRasterAboveThreshold(AggregateRaster):
    """AggregateRaster restricted, per feature, to cells >= the value in column
    ``threshold_name`` (reference: geometry/aggregate.py:590-646)."""

    def __init__(self, source, raster, statistic="sum", projection=None, pixel_size=None,
                 max_pixels=None, column_name="agg", auto_pixel_size=False, threshold_name=None):
        if not isinstance(threshold_name, str):
            raise TypeError("'{}' object is not allowed".format(type(threshold_name)))
        if threshold_name not in source.columns:
            raise KeyError("Column '{}' is not available".format(threshold_name))
        super().__init__(source, raster, statistic, projection, pixel_size, max_pixels, column_name,
                         auto_pixel_size, threshold_name)

    threshold_name = property(lambda self: self.args[8])

    def get_sources_and_requests(self, **request):
        sources = super().get_sources_and_requests(**request)
        sources[2][0]["threshold_name"] = self.threshold_name
        return sources
