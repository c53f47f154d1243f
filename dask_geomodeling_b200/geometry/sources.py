"""In-memory geometry source.

The reference ships only file/WKT based geometry sources (geometry/sources.py,
out of scope: vector file I/O); its tests feed AggregateRaster/Rasterize from
``MockGeometry`` (tests/factories.py:193-282).  ``MemoryGeometrySource`` is that
idea as a supported block: polygons (lists of rings or shapely-like objects)
plus per-feature properties, answered in the request's projection (EPSG:4326, EPSG:3857 and
the WGS 84 UTM zones; see crs.py).
"""
import numpy as np
import pandas as pd

from .. import utils
from .base import GeometryBlock

__all__ = ["MemoryGeometrySource"]


def _as_geometry(item):
    if hasattr(item, "geom_type") or hasattr(item, "exterior") or hasattr(item, "geoms"):
        return item
    arr = np.asarray(item, dtype=object if isinstance(item, (list, tuple)) and item and
                     isinstance(item[0], (list, tuple)) and item[0] and
                     isinstance(item[0][0], (list, tuple, np.ndarray)) else np.float64)
    if arr.dtype != object and arr.ndim == 2:
        return utils.Polygon(arr)               # a single ring
    rings = [np.asarray(r, dtype=np.float64) for r in item]
    return utils.Polygon(rings[0], rings[1:])   # shell + holes


class Literal(object):
    """Wrapper that carries a large list through the compute graph as ONE literal: the graph
    runtime walks plain lists element by element (they may hold task keys) and hands
    ``process`` a copy, which costs a pass over 100 k geometries per request and loses the
    identity the cache below is keyed on.  Copies of frames that carry one (``DataFrame.attrs``
    is deep-copied by pandas) share it."""

    def __init__(self, value):
        self.value = value

    def __deepcopy__(self, memo):
        return self

    def __copy__(self):
        return self


def prepared_soup_of(features):
    """The CSR form a MemoryGeometrySource attached to ``features`` -- (full soup, positions of the
    frame's rows in it, the source's geometry objects) -- if the frame still holds exactly those
    geometries in that order, else None.  ``DataFrame.attrs`` travels through most pandas
    operations, so a block in between may have dropped, reordered or replaced rows: the length and
    the identity of up to 64 evenly spaced rows (first and last included) are checked."""
    prepared = features.attrs.get("polygon_soup") if "geometry" in features else None
    prepared = getattr(prepared, "value", None)
    n = len(features)
    if prepared is None or n == 0 or len(prepared[1]) != n:
        return None
    full, positions, geometries = prepared
    column = features["geometry"].values
    for k in np.unique(np.linspace(0, n - 1, min(n, 64)).astype(np.int64)):
        if column[k] is not geometries[positions[k]]:
            return None
    return prepared


def _unwrap(x):
    return x.value if isinstance(x, Literal) else x


_PREPARED = {}   # id(polygons) -> (polygons, geometries, soup, bounds); a few sources at most


def _bounds(soup, geometries):
    """Bounding boxes from the CSR arrays; geometries without rings (points) are asked."""
    bounds = soup.bounds()
    for i in np.nonzero(np.isnan(bounds[:, 0]))[0]:
        if hasattr(geometries[i], "bounds") and not getattr(geometries[i], "is_empty", False):
            bounds[i] = geometries[i].bounds
    return bounds


def _prepared(polygons, projection=None, target=None):
    """Geometry objects, CSR soup and bounding boxes of a polygon list in CRS ``target``, built
    once per list object and target (the list is an argument of the block, i.e. it lives as long
    as the view).  In another CRS than the list's ``projection`` the soup's vertices are
    transformed in one vectorised call and the geometry objects vertex by vertex."""
    # the list must not be edited in place afterwards; a sample of its elements' identities
    # (first, last, 30 in between) catches the edits that keep its length
    n = len(polygons)
    sample = tuple(id(polygons[i]) for i in sorted(set(np.linspace(0, n - 1, 32).astype(int).tolist()))) if n else ()
    same = target is None or utils.same_projection(projection, target)
    key = (id(polygons), None if same else (utils.get_epsg_or_wkt(projection), utils.get_epsg_or_wkt(target)))
    hit = _PREPARED.get(key)
    if hit is not None and hit[0] is polygons and len(hit[1]) == n and hit[4] == sample:
        return hit[1], hit[2], hit[3]
    geometries = [_as_geometry(p) for p in polygons]
    soup = utils.PolygonSoup(geometries)
    if not same:
        soup = soup.transformed(projection, target)
        geometries = [utils.shapely_transform(g, projection, target) for g in geometries]
    bounds = _bounds(soup, geometries)
    if len(_PREPARED) >= 8:
        _PREPARED.pop(next(iter(_PREPARED)))
    _PREPARED[key] = (polygons, geometries, soup, bounds, sample)
    return geometries, soup, bounds


class MemoryGeometrySource(GeometryBlock):
    """Features held in memory.

    Args:
      polygons: list of geometries; each a list of (x, y) tuples (one ring), a list
        of rings (shell followed by holes) or a geometry object
      properties: optional list of dicts (one per feature); key ``id`` becomes the index
      projection: projection of the coordinates
    """

    def __init__(self, polygons, properties=None, projection="EPSG:3857"):
        super().__init__(polygons, properties, projection)

    polygons = property(lambda self: self.args[0])
    properties = property(lambda self: self.args[1])
    projection = property(lambda self: self.args[2])

    @property
    def columns(self):
        result = {"geometry"}
        if self.properties:
            result |= set(self.properties[0].keys())
        result.discard("id")
        return result

    def get_sources_and_requests(self, **request):
        literals = getattr(self, "_literals", None)
        if literals is None:
            literals = self._literals = (Literal(self.polygons), Literal(self.properties))
        return [(literals[0], None), (literals[1], None), (self.projection, None), (request, None)]

    @staticmethod
    def process(polygons, properties, projection, request):
        polygons, properties = _unwrap(polygons), _unwrap(properties)
        limit = request.get("limit")
        if limit is not None:
            polygons = polygons[:limit]
            properties = properties[:limit] if properties is not None else None
        mode = request.get("mode", "intersects")
        geometries, soup, bounds = _prepared(polygons, projection, request["projection"])
        if mode == "extent":
            extent = None
            if len(geometries):
                extent = (bounds[:, 0].min(), bounds[:, 1].min(), bounds[:, 2].max(), bounds[:, 3].max())
            return {"extent": extent, "projection": request["projection"]}
        if len(geometries) == 0:
            return {"features": pd.DataFrame([]), "projection": request["projection"]}
        df = pd.DataFrame.from_records(properties) if properties is not None else pd.DataFrame(index=range(len(geometries)))
        df["geometry"] = pd.Series(geometries, index=df.index, dtype=object)
        if "id" in df.columns:
            df = df.set_index("id", drop=True)
        else:
            df.index.name = "id"
        window = request.get("geometry")
        positions = np.arange(len(geometries))
        if window is not None and mode in ("intersects", "centroid"):
            x1, y1, x2, y2 = window.bounds
            if mode == "intersects":  # bounding boxes decide (no GEOS here)
                keep = (bounds[:, 2] >= x1) & (bounds[:, 0] <= x2) & (bounds[:, 3] >= y1) & (bounds[:, 1] <= y2)
            else:
                c = np.array([(g.centroid.x, g.centroid.y) for g in geometries])
                keep = (c[:, 0] >= x1) & (c[:, 0] <= x2) & (c[:, 1] >= y1) & (c[:, 1] <= y2)
            df = df[keep]
            positions = positions[keep]
        # the CSR form of the geometries travels with the frame, so that consumers on the GPU
        # path (AggregateRaster, Rasterize) need not walk the geometry objects again
        df.attrs["polygon_soup"] = Literal((soup, positions, geometries))
        return {"features": df, "projection": request["projection"]}
