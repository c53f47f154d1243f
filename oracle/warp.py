"""NumPy restatement of the nearest-neighbour warp across projections (gdal.ReprojectImage with
GRA_NearestNeighbour in the reference's raster/sources.py:119-149, without GDAL's approximate
transformer): every target cell centre is transformed exactly in float64 with the host CRS
module, then the source cell is floor((x - p) / a + 1e-10), floor((y - q) / d + 1e-10)."""
import numpy as np

from dask_geomodeling_b200 import crs

EDGE_PX = 1e-6   # source coordinates this close to a cell edge may round either way (libm ulps)


def warp_nn(array, geo_transform, source_projection, no_data_value, bbox, height, width,
            projection, rows=None, cols=None):
    """(values, near_edge) for target rows ``rows`` x columns ``cols`` (slices of the request
    grid, default all).  ``near_edge`` marks cells whose source coordinate lies within EDGE_PX
    of a cell edge, where the device's libm may pick the neighbouring cell."""
    array = np.asarray(array)
    if array.ndim == 2:
        array = array[np.newaxis]
    n, src_h, src_w = array.shape
    x1, y1, x2, y2 = bbox
    a_d, d_d = (x2 - x1) / width, (y1 - y2) / height
    i = np.arange(height)[rows or slice(None)]
    j = np.arange(width)[cols or slice(None)]
    x = x1 + (j[np.newaxis, :] + 0.5) * a_d + 0 * i[:, np.newaxis]
    y = y2 + (i[:, np.newaxis] + 0.5) * d_d + 0 * j[np.newaxis, :]
    src, dst = crs.crs_pair(source_projection, projection)
    sx, sy = crs.transform_xy(x, y, dst, src)
    p, a, _, q, _, d = geo_transform
    with np.errstate(invalid="ignore"):
        fc = (sx - p) / a + 1e-10
        fr = (sy - q) / d + 1e-10
        near = (np.abs(fc - np.round(fc)) < EDGE_PX) | (np.abs(fr - np.round(fr)) < EDGE_PX)
        c, r = np.floor(fc), np.floor(fr)
        inside = (c >= 0) & (c < src_w) & (r >= 0) & (r < src_h)
    out = np.full((n,) + x.shape, no_data_value, dtype=array.dtype)
    ri, ci = r[inside].astype(np.int64), c[inside].astype(np.int64)
    out[:, inside] = array[:, ri, ci]
    if out.dtype.kind == "f":
        out[~np.isfinite(out)] = no_data_value
    return out, near & np.isfinite(fc) & np.isfinite(fr)
