"""Helpers of the raster compute path.

Mirrors the names the reference blocks import from ``dask_geomodeling.utils``
(utils.py; line numbers cited per function).  CRS handling is limited to what
works without GDAL/pyproj: projections are compared by their normalised
string, coordinates are transformed between EPSG:4326, EPSG:3857 and the WGS 84
UTM zones (``crs.py``), and every other transformation raises.
"""
import math
import os
import re
import warnings
from datetime import timedelta

import numpy as np

# ---------------------------------------------------------------------------
# dtype helpers (utils.py:61-108, :813-845)
# ---------------------------------------------------------------------------


def get_index(values, no_data_value):
    """Boolean index of the cells that hold data: ``np.isclose`` decides for
    floating point rasters, exact equality otherwise (utils.py:61-64)."""
    if values.dtype.kind == "f":
        return ~np.isclose(values, no_data_value)
    return ~np.equal(values, no_data_value)


def get_dtype_max(dtype):
    d = np.dtype(dtype)
    return np.finfo(d).max.item() if d.kind == "f" else np.iinfo(d).max


def get_dtype_min(dtype):
    d = np.dtype(dtype)
    return np.finfo(d).min.item() if d.kind == "f" else np.iinfo(d).min


def get_int_dtype(n):
    """Smallest signed dtype holding ``n`` plus a spare no data value."""
    for code in ("i1", "i2", "i4", "i8"):
        info = np.iinfo(code)
        if info.min <= n and n - 1 <= info.max:
            return np.dtype(code)
    raise ValueError("Value does not fit in int dtype ({})".format(n))


def get_uint_dtype(n):
    """Smallest unsigned dtype holding ``n`` plus a spare no data value."""
    if n < 0:
        raise ValueError("Value does not fit in uint dtype ({})".format(n))
    for code in ("u1", "u2", "u4", "u8"):
        if n - 1 <= np.iinfo(code).max:
            return np.dtype(code)
    raise ValueError("Value does not fit in uint dtype ({})".format(n))


_PERCENTILE = re.compile(r"^p([\d.]+)$")


def parse_percentile_statistic(statistic):
    """'p<float>' -> ('percentile', float); anything else -> (statistic, None)."""
    found = _PERCENTILE.findall(statistic)
    if not found:
        return statistic, None
    q = float(found[0])
    if not 0 <= q <= 100:
        raise ValueError("Percentiles must be in the range [0, 100]")
    return "percentile", q


def _at_least_32bit(dtype):
    dtype = np.dtype(dtype)
    if dtype == bool or np.issubdtype(dtype, np.integer):
        return np.result_type(dtype, np.int32)
    if np.issubdtype(dtype, np.floating):
        return np.result_type(dtype, np.float32)
    return dtype


def dtype_for_statistic(dtype, statistic):
    """Result dtype of a temporal statistic (utils.py:826-845)."""
    if statistic in ("min", "max"):
        return dtype
    if statistic == "sum":
        return _at_least_32bit(dtype)
    if statistic == "count":
        return np.int32
    return np.result_type(np.float32, dtype)


def get_footprint(size):
    """Boolean disc of (odd) diameter ``size``: x^2 + y^2 < (size/2)^2
    (utils.py:536-547)."""
    s = size // 2 * 2 + 1
    half = (s - 1) // 2
    y, x = np.ogrid[-half : half + 1, -half : half + 1]
    return (x * x + y * y) < (s / 2) ** 2


# ---------------------------------------------------------------------------
# projections (string level only)
# ---------------------------------------------------------------------------


def get_epsg_or_wkt(text):
    """Normalise 'epsg:28992' -> 'EPSG:28992'; other strings are kept as is
    (the reference resolves WKT through GDAL, utils.py:514-533)."""
    text = str(text).strip()
    m = re.match(r"^(epsg):(\d+)$", text, flags=re.IGNORECASE)
    return "EPSG:{}".format(m.group(2)) if m else text


def same_projection(a, b):
    return get_epsg_or_wkt(a) == get_epsg_or_wkt(b)


def is_geographic(projection):
    return get_epsg_or_wkt(projection) in ("EPSG:4326", "EPSG:4258", "EPSG:4269")


class Extent(object):
    """Bounding box tagged with its projection (subset of utils.py:128-205)."""

    def __init__(self, bbox, projection):
        self.bbox = tuple(bbox)
        self.projection = get_epsg_or_wkt(projection)

    def transformed(self, projection):
        """The bounds of the box's corners transformed into ``projection``.  Only the four
        corners are transformed; whether the reference densifies the box edges first is not
        pinned (it transforms the box polygon through GDAL/OGR)."""
        if same_projection(self.projection, projection):
            return Extent(self.bbox, projection)
        from . import crs

        x1, y1, x2, y2 = self.bbox
        xy = crs.transform([(x2, y1), (x2, y2), (x1, y2), (x1, y1)], self.projection, projection)
        return Extent((xy[:, 0].min(), xy[:, 1].min(), xy[:, 0].max(), xy[:, 1].max()), projection)

    @classmethod
    def from_geometry(cls, geometry, projection=None):
        return cls(geometry.bounds, projection or getattr(geometry, "projection", None))

    def as_geometry(self):
        geometry = box(*self.bbox)
        geometry.projection = self.projection
        return geometry

    def intersection(self, other):
        x1, y1 = max(self.bbox[0], other.bbox[0]), max(self.bbox[1], other.bbox[1])
        x2, y2 = min(self.bbox[2], other.bbox[2]), min(self.bbox[3], other.bbox[3])
        if x2 <= x1 or y2 <= y1:
            return None
        return Extent((x1, y1, x2, y2), self.projection)


# ---------------------------------------------------------------------------
# GeoTransform (utils.py:208-393)
# ---------------------------------------------------------------------------


class GeoTransform(tuple):
    """GDAL style 6-tuple (p, a, b, q, c, d): x = p + a*col, y = q + d*row."""

    @classmethod
    def from_bbox(cls, bbox, height, width):
        x1, y1, x2, y2 = bbox
        return cls((x1, (x2 - x1) / width, 0, y2, 0, (y1 - y2) / height))

    def __init__(self, tpl):
        if len(tpl) != 6:
            raise ValueError("GeoTransform expected an iterable of length 6")
        if any(not math.isclose(tpl[i], 0.0, abs_tol=1e-7) for i in (2, 4)):
            raise ValueError("Tilted geo_transforms are not supported")
        if any(math.isclose(tpl[i], 0.0, abs_tol=1e-7) for i in (1, 5)):
            raise ValueError("Pixel size should not be zero")

    @property
    def origin(self):
        return self[0], self[3]

    @property
    def origin_normalized(self):
        return self[0] % self[1], self[3] % self[5]

    @property
    def cell_area(self):
        return abs(self[1] * self[5] - self[2] * self[4])

    def get_inverse(self):
        _, a, b, _, c, d = self
        det = 1 / (a * d - b * c)
        return d * det, -b * det, -c * det, a * det

    def shift(self, origin):
        p, a, b, q, c, d = self
        i, j = origin
        return type(self)([p + a * j + b * i, a, b, q + c * j + d * i, c, d])

    def scale(self, x, y):
        p, a, b, q, c, d = self
        return type(self)([p, a * x, b * x, q, c * y, d * y])

    def get_indices(self, points):
        """(rows, cols) int64 arrays of the cells containing ``points`` (N x 2)."""
        p, _, _, q, _, _ = self
        e, f, g, h = self.get_inverse()
        x, y = np.asarray(points).transpose()
        rows = np.floor(g * (x - p) + h * (y - q)).astype(np.int64)
        cols = np.floor(e * (x - p) + f * (y - q)).astype(np.int64)
        return rows, cols

    def get_bbox(self, offset, shape):
        p, a, b, q, c, d = self
        i, j = offset
        m, n = shape
        west, north = p + a * j + b * i, q + c * j + d * i
        return west, north + c * n + d * m, west + a * n + b * m, north

    def aligns_with(self, other):
        if not isinstance(other, GeoTransform):
            other = GeoTransform(other)
        if abs(self[1]) != abs(other[1]) or abs(self[5]) != abs(other[5]):
            return False
        return self.origin_normalized == other.origin_normalized


# ---------------------------------------------------------------------------
# time axis (utils.py:848-915)
# ---------------------------------------------------------------------------


def snap_start_stop(start, stop, time_first, time_delta, length):
    """Resolve request start/stop against an equidistant time axis.

    Returns ``(start, stop, first_index, last_index)``: both None -> last
    frame; stop None -> frame nearest to start; else the closed interval.
    """
    if length == 0:
        return None, None, None, None
    if length > 1 and time_delta is None:
        raise ValueError("Length > 1 requires a timedelta")
    last = time_first if length == 1 else time_first + (length - 1) * time_delta

    def frame(i):
        return time_first if i == 0 else time_first + time_delta * i

    if start is None:
        i = j = length - 1
    elif stop is None:
        if start <= time_first:
            i = j = 0
        elif start >= last:
            i = j = length - 1
        else:
            i = j = int(round((start - time_first) / time_delta))
    else:
        if start > last or stop < time_first:
            return None, None, None, None
        if length == 1:
            i = j = 0
        else:
            i = max(int(np.ceil((start - time_first) / time_delta)), 0)
            j = min(int(np.floor((stop - time_first) / time_delta)), length - 1)
    return frame(i), frame(j), i, j


def dt_to_ms(dt):
    from datetime import timezone

    if dt.tzinfo is None:
        dt = dt.replace(tzinfo=timezone.utc)
    return int(dt.timestamp() * 1000)


# ---------------------------------------------------------------------------
# light-weight geometries (stand-ins for shapely objects; duck-typed so that
# real shapely Polygons / MultiPolygons / Points are accepted as well)
# ---------------------------------------------------------------------------


def _ring(coords):
    ring = np.asarray(coords, dtype=np.float64).reshape(-1, 2)
    if len(ring) and not np.array_equal(ring[0], ring[-1]):
        ring = np.vstack([ring, ring[:1]])
    return ring


class _Ring(object):
    def __init__(self, coords):
        self.coords = _ring(coords)


class Polygon(object):
    """Simple polygon: exterior ring and optional holes."""

    geom_type = "Polygon"

    def __init__(self, shell, holes=None):
        self.exterior = _Ring(shell)
        self.interiors = [_Ring(h) for h in (holes or [])]

    @property
    def is_empty(self):
        return len(self.exterior.coords) == 0

    @property
    def bounds(self):
        c = self.exterior.coords
        return (c[:, 0].min(), c[:, 1].min(), c[:, 0].max(), c[:, 1].max())

    @property
    def centroid(self):
        area, cx, cy = 0.0, 0.0, 0.0
        for sign, ring in [(1, self.exterior)] + [(-1, r) for r in self.interiors]:
            a, x, y = _ring_moments(ring.coords)
            area += sign * abs(a)
            cx += sign * x * np.sign(a)
            cy += sign * y * np.sign(a)
        if area == 0:
            c = self.exterior.coords
            return Point(c[:, 0].mean(), c[:, 1].mean())
        return Point(cx / area, cy / area)


class MultiPolygon(object):
    geom_type = "MultiPolygon"

    def __init__(self, polygons):
        self.geoms = [p if isinstance(p, Polygon) else Polygon(*p) for p in polygons]

    @property
    def is_empty(self):
        return all(p.is_empty for p in self.geoms)

    @property
    def bounds(self):
        b = np.array([p.bounds for p in self.geoms])
        return (b[:, 0].min(), b[:, 1].min(), b[:, 2].max(), b[:, 3].max())

    @property
    def centroid(self):
        tot, cx, cy = 0.0, 0.0, 0.0
        for p in self.geoms:
            a = abs(_ring_moments(p.exterior.coords)[0]) - sum(
                abs(_ring_moments(r.coords)[0]) for r in p.interiors
            )
            c = p.centroid
            tot, cx, cy = tot + a, cx + a * c.x, cy + a * c.y
        return Point(cx / tot, cy / tot) if tot else self.geoms[0].centroid


class Point(object):
    geom_type = "Point"

    def __init__(self, x, y):
        self.x, self.y = float(x), float(y)

    is_empty = False

    @property
    def bounds(self):
        return (self.x, self.y, self.x, self.y)

    @property
    def centroid(self):
        return self


def box(x1, y1, x2, y2):
    """Rectangular polygon (counterpart of shapely.geometry.box)."""
    return Polygon([(x2, y1), (x2, y2), (x1, y2), (x1, y1), (x2, y1)])


class WKTReadingError(ValueError):
    pass


_WKT_NUMBER = r"[-+]?(?:\d+\.?\d*|\.\d+)(?:[eE][-+]?\d+)?"


def _wkt_rings(text):
    rings = []
    for body in re.findall(r"\(([^()]+)\)", text):
        pts = []
        for pair in body.split(","):
            nums = re.findall(_WKT_NUMBER, pair)
            if len(nums) < 2:
                raise WKTReadingError("malformed coordinate '{}'".format(pair))
            pts.append((float(nums[0]), float(nums[1])))
        rings.append(pts)
    return rings


def shapely_from_wkt(wkt):
    """Parse POINT / POLYGON / MULTIPOLYGON WKT into the light-weight geometry
    classes (shapely is used instead when it is installed)."""
    try:
        from shapely import from_wkt  # pragma: no cover

        try:
            return from_wkt(wkt)
        except Exception as e:  # pragma: no cover
            raise WKTReadingError(str(e))
    except ImportError:
        pass
    text = wkt.strip()
    m = re.match(r"^(?:SRID=\d+;)?\s*([A-Za-z]+)\s*(Z|M|ZM)?\s*(EMPTY|\(.*\))$", text, flags=re.S)
    if not m:
        raise WKTReadingError("cannot parse WKT '{}'".format(wkt[:40]))
    kind, body = m.group(1).upper(), m.group(3)
    if body.count("(") != body.count(")"):
        raise WKTReadingError("unbalanced parentheses")
    if kind == "POINT":
        nums = re.findall(_WKT_NUMBER, body)
        if len(nums) < 2:
            raise WKTReadingError("malformed point")
        return Point(float(nums[0]), float(nums[1]))
    if kind == "POLYGON":
        if body == "EMPTY":
            return Polygon([])
        rings = _wkt_rings(body)
        if not rings:
            raise WKTReadingError("polygon without rings")
        return Polygon(rings[0], rings[1:])
    if kind == "MULTIPOLYGON":
        if body == "EMPTY":
            return MultiPolygon([])
        parts = re.findall(r"\(\s*(\((?:[^()]+)\)(?:\s*,\s*\((?:[^()]+)\))*)\s*\)", body)
        polygons = []
        for part in parts:
            rings = _wkt_rings(part)
            polygons.append(Polygon(rings[0], rings[1:]))
        if not polygons:
            raise WKTReadingError("multipolygon without parts")
        return MultiPolygon(polygons)
    raise WKTReadingError("unsupported geometry type '{}'".format(kind))


def _map_coords(geometry, fn):
    """``geometry`` with every vertex array passed through ``fn`` (N x 2 -> N x 2); the classes
    above and shapely-like objects (rebuilt as the classes above)."""
    if geometry is None or getattr(geometry, "is_empty", False):
        return geometry
    if hasattr(geometry, "geoms"):
        return MultiPolygon([_map_coords(part, fn) for part in geometry.geoms])
    if hasattr(geometry, "exterior"):
        shell = fn(np.asarray(geometry.exterior.coords, dtype=np.float64)[:, :2])
        return Polygon(shell, [fn(np.asarray(r.coords, dtype=np.float64)[:, :2]) for r in geometry.interiors])
    kind = getattr(geometry, "geom_type", type(geometry).__name__)
    if kind == "Point":
        x, y = fn(np.array([[float(geometry.x), float(geometry.y)]]))[0]
        return Point(x, y)
    raise NotImplementedError("cannot transform geometries of type '{}'".format(kind))


def shapely_transform(geometry, src_srs, dst_srs):
    """``geometry`` with every vertex transformed from ``src_srs`` to ``dst_srs``, as
    shapely.ops.transform with a pyproj transformer does.  Unsupported CRS pairs raise
    NotImplementedError (see crs.py)."""
    if same_projection(src_srs, dst_srs):
        return geometry
    from . import crs

    crs.crs_pair(src_srs, dst_srs)
    return _map_coords(geometry, lambda xy: crs.transform(xy, src_srs, dst_srs))


def _ring_moments(c):
    """Signed area and area-weighted first moments of a closed ring."""
    x0, y0, x1, y1 = c[:-1, 0], c[:-1, 1], c[1:, 0], c[1:, 1]
    cross = x0 * y1 - x1 * y0
    area = cross.sum() / 2.0
    return area, ((x0 + x1) * cross).sum() / 6.0, ((y0 + y1) * cross).sum() / 6.0


def geometry_rings(geometry, points=False):
    """All rings (N x 2 float64 arrays, closed) of a (multi)polygon; works for
    the classes above and for shapely geometries.  ``points=True`` turns a Point into a
    one-vertex ring, which the rasteriser burns into the cell that contains it (GDAL's
    GDALdllImagePoint)."""
    if geometry is None or getattr(geometry, "is_empty", False):
        return []
    if hasattr(geometry, "geoms"):
        rings = []
        for part in geometry.geoms:
            rings.extend(geometry_rings(part))
        return rings
    if hasattr(geometry, "exterior"):
        rings = [_ring(np.asarray(geometry.exterior.coords)[:, :2])]
        rings.extend(_ring(np.asarray(r.coords)[:, :2]) for r in geometry.interiors)
        return rings
    kind = getattr(geometry, "geom_type", type(geometry).__name__)
    if kind == "Point" and points:
        return [np.array([[float(geometry.x), float(geometry.y)]], dtype=np.float64)]
    if kind in ("Point", "MultiPoint"):
        # no area: nothing to scan-convert.  AggregateRaster samples such features at the cell
        # that contains them (the cell GDAL's point burn would label); rasterize_geoseries
        # refuses them (see there)
        return []
    # GDAL burns lines with its own Bresenham variant (GDALdllImageLine); that rule is not
    # part of this build, and dropping the feature silently would be wrong
    raise NotImplementedError(
        "geometries of type '{}' are not supported by the CUDA rasteriser "
        "(polygons and multipolygons only)".format(kind))


def point_in_rings(rings, x, y):
    """Even-odd test of one point against a ring set (used for point requests)."""
    inside = False
    for ring in rings:
        x0, y0, x1, y1 = ring[:-1, 0], ring[:-1, 1], ring[1:, 0], ring[1:, 1]
        crosses = (y0 > y) != (y1 > y)
        with np.errstate(divide="ignore", invalid="ignore"):
            xi = x0 + (y - y0) * (x1 - x0) / (y1 - y0)
        inside ^= bool(np.count_nonzero(crosses & (x < xi)) & 1)
    return inside


def _expand_ranges(starts, counts):
    """Concatenation of arange(starts[i], starts[i] + counts[i]) without a Python loop."""
    starts, counts = np.asarray(starts, dtype=np.int64), np.asarray(counts, dtype=np.int64)
    total = int(counts.sum())
    if total == 0:
        return np.zeros(0, dtype=np.int64)
    keep = counts > 0
    starts, counts = starts[keep], counts[keep]
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    steps = np.ones(total, dtype=np.int64)
    steps[first] = starts - np.concatenate([[0], starts[:-1] + counts[:-1] - 1])
    return np.cumsum(steps)


class PolygonSoup(object):
    """CSR layout the CUDA rasteriser consumes: interleaved xy, ring offsets,
    polygon -> ring offsets (GmPolygons in include/geokernels.h)."""

    def __init__(self, geometries, points=False):
        xy, ring_offsets, poly_offsets = [], [0], [0]
        n_vertices = 0
        # features without area (points) hold no rings; consumers that cannot sample them
        # (rasterize_geoseries) check this flag instead of dropping them silently
        self.has_points = False
        for geometry in geometries:
            kind = getattr(geometry, "geom_type", None)
            if kind == "MultiPoint" or (kind == "Point" and not points):
                self.has_points = True
            for ring in geometry_rings(geometry, points):
                xy.append(ring)
                n_vertices += len(ring)
                ring_offsets.append(n_vertices)
            poly_offsets.append(len(ring_offsets) - 1)
        self.xy = np.ascontiguousarray(np.concatenate(xy) if xy else np.zeros((0, 2)), dtype=np.float64)
        self.ring_offsets = np.asarray(ring_offsets, dtype=np.int64)
        self.poly_offsets = np.asarray(poly_offsets, dtype=np.int64)

    @property
    def n_polygons(self):
        return len(self.poly_offsets) - 1

    def subset(self, ids):
        """The soup of the polygons `ids` (in that order); index arithmetic only."""
        ids = np.asarray(ids, dtype=np.int64)
        sub = PolygonSoup([])
        sub.has_points = self.has_points
        if len(ids) == 0:
            return sub
        ring_a, ring_n = self.poly_offsets[ids], self.poly_offsets[ids + 1] - self.poly_offsets[ids]
        rings = _expand_ranges(ring_a, ring_n)
        v_a, v_n = self.ring_offsets[rings], self.ring_offsets[rings + 1] - self.ring_offsets[rings]
        sub.xy = np.ascontiguousarray(self.xy[_expand_ranges(v_a, v_n)], dtype=np.float64).reshape(-1, 2)
        sub.ring_offsets = np.concatenate([[0], np.cumsum(v_n)]).astype(np.int64)
        sub.poly_offsets = np.concatenate([[0], np.cumsum(ring_n)]).astype(np.int64)
        return sub

    def transformed(self, src_srs, dst_srs):
        """The soup with every vertex transformed from ``src_srs`` to ``dst_srs`` in one call."""
        if same_projection(src_srs, dst_srs):
            return self
        from . import crs

        out = PolygonSoup([])
        out.has_points = self.has_points
        out.xy = np.ascontiguousarray(crs.transform(self.xy, src_srs, dst_srs))
        out.ring_offsets, out.poly_offsets = self.ring_offsets, self.poly_offsets
        return out

    def bounds(self):
        """(n, 4) array of (xmin, ymin, xmax, ymax) per polygon (NaN for empty ones)."""
        n = self.n_polygons
        out = np.full((n, 4), np.nan)
        starts = self.ring_offsets[self.poly_offsets[:-1]]
        ends = self.ring_offsets[self.poly_offsets[1:]]
        filled = np.nonzero(ends > starts)[0]
        if len(filled):
            out[filled, :2] = np.minimum.reduceat(self.xy, starts[filled], axis=0)
            out[filled, 2:] = np.maximum.reduceat(self.xy, starts[filled], axis=0)
        return out

    def as_struct(self):
        from ._native import GmPolygons

        s = GmPolygons()
        s.xy = self.xy.ctypes.data
        s.ring_offsets = self.ring_offsets.ctypes.data
        s.poly_offsets = self.poly_offsets.ctypes.data
        s.n_polygons = self.n_polygons
        s.n_rings = len(self.ring_offsets) - 1
        s.n_vertices = len(self.xy)
        s.resident = getattr(self, "_resident", None)
        return s

    def to_device(self):
        """Keep the CSR arrays in HBM (gm_polygons_upload) for as long as this soup lives:
        later rasterise / zonal calls skip the per-call upload."""
        import ctypes
        import weakref

        from . import _native

        if getattr(self, "_resident", None) is None:
            handle = ctypes.c_void_p()
            polys = self.as_struct()
            _native.check(_native.lib().gm_polygons_upload(ctypes.byref(polys), ctypes.byref(handle)))
            self._resident = handle.value
            weakref.finalize(self, _native.free_polygons, handle.value)
        return self


# ---------------------------------------------------------------------------
# rasterize_geoseries (utils.py:638-756) on the GPU scanline rasteriser
# ---------------------------------------------------------------------------


def _finalize_rasterize_result(array, no_data_value):
    if array.dtype == bool:         # burned on the device straight into a boolean raster
        return {"values": array, "no_data_value": None}
    if array.dtype == np.uint8:
        return {"values": array.astype(bool), "no_data_value": None}
    return {"values": array, "no_data_value": no_data_value}


def rasterize_geoseries(geoseries, bbox, projection, height, width, values=None, soup=None):
    """Burn geometries into a ``(1, height, width)`` raster.

    Same contract as the reference (utils.py:638-756): no values / bool values
    -> boolean raster; integer values -> int32 with int32-max as no data; float
    values -> float64 with float64-max as no data (non-finite values dropped).
    A cell is burned when its centre lies inside the polygon; later geometries
    overwrite earlier ones.  A point bbox returns the value of the last
    geometry containing the point.  ``soup`` = the PolygonSoup of ``geoseries`` when the
    caller already has it (geometry/sources.py prepares it once per polygon list).
    """
    import pandas as pd
    from . import _native
    import ctypes

    if geoseries is not None and not isinstance(geoseries, pd.Series):
        geoseries = pd.Series(list(geoseries), dtype=object)
    if values is not None and not isinstance(values, pd.Series):
        values = pd.Series(np.asarray(values), index=None if geoseries is None else geoseries.index)

    positions = None if geoseries is None else np.arange(len(geoseries))
    if soup is not None and (geoseries is None or soup.n_polygons != len(geoseries)):
        soup = None
    if values is None or values.dtype == bool:
        dtype, no_data_value = np.uint8, 0
        if values is not None and geoseries is not None:
            geoseries, positions = geoseries[values.values], positions[values.values]
        values = None
    elif str(values.dtype) == "category":
        values = pd.Series(np.asarray(values), index=values.index)

    if values is not None:
        if np.issubdtype(values.dtype, np.floating):
            dtype = np.float64
            no_data_value = get_dtype_max(dtype)
            if geoseries is not None:
                finite = np.isfinite(values.values)
                geoseries, values, positions = geoseries[finite], values[finite], positions[finite]
        elif np.issubdtype(values.dtype, np.integer):
            dtype = np.int32
            no_data_value = get_dtype_max(dtype)
        else:
            raise TypeError("Unsupported values dtype to rasterize: '{}'".format(values.dtype))

    if geoseries is None or len(geoseries) == 0:
        return _finalize_rasterize_result(
            np.full((1, height, width), no_data_value, dtype=dtype), no_data_value
        )

    present = ~geoseries.isnull().values
    geoseries, positions = geoseries[present], positions[present]
    if values is not None:
        values = values[present]

    x1, y1, x2, y2 = bbox
    if not ((x2 == x1 and y2 == y1) or (x1 < x2 and y1 < y2)):
        raise ValueError("Invalid bbox ({})".format(bbox))

    if x2 == x1 and y2 == y1:
        array = np.full((1, height, width), no_data_value, dtype=dtype)
        hits = [point_in_rings(geometry_rings(g), x1, y1) for g in geoseries]
        if any(hits):
            array[:] = True if values is None else values.values[np.nonzero(hits)[0][-1]]
        return _finalize_rasterize_result(array, no_data_value)

    if soup is None or soup.has_points:
        # (points are burned into the cell that contains them: one-vertex rings)
        soup = PolygonSoup(geoseries.values, points=True)
    elif len(positions) != soup.n_polygons:
        soup = soup.subset(positions)
    if soup.has_points:
        raise NotImplementedError(
            "MultiPoint geometries cannot be burned by the CUDA rasteriser (polygons and points only)")
    burn = (
        np.ones(soup.n_polygons, dtype=dtype)
        if values is None
        else np.ascontiguousarray(values.values, dtype=dtype)
    )
    geo = (ctypes.c_double * 6)(*GeoTransform.from_bbox(bbox, height, width))
    from . import _state

    if _state.keep_on_device():
        # inside a view the burned raster stays in HBM (Rasterize -> Clip / Mask fuse on it)
        array = _native.DeviceArray((1, height, width), bool if dtype == np.uint8 else dtype)
    else:
        array = _native.pinned_empty((1, height, width), dtype)
    nodata_holder, nodata_ptr = _native.scalar_ptr(no_data_value, dtype)
    dst = _native.as_gm_array(array)
    polys = soup.as_struct()
    lib = _native.lib()
    _native.check(
        lib.gm_rasterize_polygons(
            ctypes.byref(polys), geo, burn.ctypes.data, nodata_ptr, ctypes.byref(dst),
            _native.current_stream(),
        )
    )
    return _finalize_rasterize_result(array, no_data_value)


def safe_file_url(url, start=None):
    """``file://`` URL with an absolute path: relative paths are taken from ``geomodeling.root``,
    other protocols raise NotImplementedError, and with ``geomodeling.strict-file-paths`` the path
    must lie inside the root (reference utils.py:767-807)."""
    from ._compat import config

    try:
        protocol, path = url.split("://")
    except ValueError:
        protocol, path = "file", url
    else:
        if protocol != "file":
            raise NotImplementedError('Unknown protocol: "{}"'.format(protocol))
    if start is not None:
        warnings.warn("Using the start argument in safe_file_url is deprecated. Use the "
                      "'geomodeling.root' in the dask config", DeprecationWarning)
    else:
        start = config.get("geomodeling.root")
    if not os.path.isabs(path):
        if start is None:
            raise IOError("Relative path '{}' provided but start was not given.".format(path))
        abspath = os.path.abspath(os.path.join(start, path))
    else:
        abspath = os.path.abspath(path)
    if config.get("geomodeling.strict-file-paths") and not abspath.startswith(start):
        raise IOError("'{}' is not contained in '{}'".format(path, start))
    return "://".join([protocol, abspath])


def safe_abspath(url, start=None):
    """The path of ``safe_file_url`` without the protocol (reference utils.py:759-764)."""
    return safe_file_url(url, start).split("://")[1]


def offset_to_timedelta(freq):
    import pandas as pd

    return pd.tseries.frequencies.to_offset(freq) and timedelta(
        seconds=pd.Timedelta(pd.tseries.frequencies.to_offset(freq)).total_seconds()
    )
