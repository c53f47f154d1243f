"""Raster sources feeding the CUDA path: arrays in host memory and GeoTIFF / VRT files.

``MemorySource`` keeps the reference's constructor, attributes and request
handling (raster/sources.py:157-393).  Its ``process`` replaces the GDAL
nearest-neighbour warp (raster/sources.py:119-149) by: upload of only the
source window the request touches (pinned host memory -> HBM), followed by a
nearest-neighbour gather kernel that also pads with no data outside the
source.  For aligned requests this equals the crop/pad GDAL produces.
Requests in another projection than the source take the nearest-neighbour warp
(``warp_window``, gm_warp_nn) when both CRSs are EPSG:4326, EPSG:3857 or a WGS 84
UTM zone (``dask_geomodeling_b200/crs.py``); other pairs need GDAL/pyproj and raise.

``RasterFileSource`` (raster/sources.py:396-564) reads a GeoTIFF or VRT without GDAL
(``dask_geomodeling_b200/geotiff.py``): only the tiles under the requested window are inflated,
then the window takes the same upload + gather path.
"""
import ctypes
import os
from datetime import datetime, timedelta, timezone

import numpy as np

from .. import _native, _state, crs, geotiff, utils
from .._compat import config
from .base import RasterBlock

__all__ = ["MemorySource", "RasterFileSource"]


def utc_from_ms_timestamp(timestamp):
    """Naive UTC datetime from a POSIX timestamp in milliseconds."""
    return datetime.fromtimestamp(timestamp / 1000, tz=timezone.utc).replace(tzinfo=None)


def _window(n_target, first, step, n_source):
    """Source index range [lo, hi) touched by target indices 0..n_target-1 where
    target i reads source floor(first + i*step); clipped to the source."""
    a = int(np.floor(first))
    b = int(np.floor(first + (n_target - 1) * step))
    lo, hi = min(a, b), max(a, b) + 1
    return max(lo, 0), min(hi, n_source)


def window_geometry(geo_transform, bbox, height, width):
    """(col0, col_step, row0, row_step): target cell (i, j) reads source cell
    (floor(row0 + i*row_step), floor(col0 + j*col_step))."""
    p, a, _, q, _, d = geo_transform
    x1, y1, x2, y2 = bbox
    tdx, tdy = (x2 - x1) / width, (y2 - y1) / height
    # source pixel coordinates of the target pixel centres; the 1e-10 is GDAL's
    # nearest-neighbour fudge (gdalwarpkernel.cpp, GWKNearestThread)
    col0 = (x1 + 0.5 * tdx - p) / a + 1e-10
    col_step = tdx / a
    row0 = (y2 - 0.5 * tdy - q) / d + 1e-10
    row_step = -tdy / d
    return col0, col_step, row0, row_step


_RESIDENT = {}         # id(host array) -> DeviceArray of the whole array
_RESIDENT_BYTES = [0]


def _drop_resident(key, nbytes):
    if _RESIDENT.pop(key, None) is not None:
        _RESIDENT_BYTES[0] -= nbytes


def resident_copy(array):
    """The HBM copy of a MemorySource array when ``geomodeling.device-cache-bytes`` allows one
    (uploaded on first use, dropped when the host array is garbage collected); else None."""
    import weakref

    budget = int(config.get("geomodeling.device-cache-bytes", 0) or 0)
    if budget <= 0:
        return None
    key = id(array)
    hit = _RESIDENT.get(key)
    if hit is not None and hit.shape == array.shape and hit.dtype == array.dtype:
        _native.STATS["resident_hits"] = _native.STATS.get("resident_hits", 0) + 1
        return hit
    if not array.flags.c_contiguous or _RESIDENT_BYTES[0] + array.nbytes > budget:
        return None
    copy = _native.DeviceArray.from_host(array)
    _native.synchronize()
    _RESIDENT[key] = copy
    _RESIDENT_BYTES[0] += array.nbytes
    weakref.finalize(array, _drop_resident, key, array.nbytes)
    return copy


def source_window(geo_transform, bbox, height, width, src_h, src_w):
    """(r_lo, r_hi, c_lo, c_hi): the cells of a (src_h, src_w) source that a request reads."""
    col0, col_step, row0, row_step = window_geometry(geo_transform, bbox, height, width)
    c_lo, c_hi = _window(width, col0, col_step, src_w)
    r_lo, r_hi = _window(height, row0, row_step, src_h)
    r_lo, c_lo = min(r_lo, src_h), min(c_lo, src_w)      # a request beyond the source: empty window
    return r_lo, max(r_hi, r_lo), c_lo, max(c_hi, c_lo)


def upload_window(array, b0, window, target):
    """Copy cells ``window = (r_lo, r_hi, c_lo, c_hi)`` of bands b0.. of a host array into the
    DeviceArray ``target`` of shape (bands, r_hi - r_lo, c_hi - c_lo)."""
    lib = _native.lib()
    stream = _native.current_stream()
    r_lo, r_hi, c_lo, c_hi = window
    n_bands, win_h, win_w = target.shape
    src_h, src_w = array.shape[1:]
    item = array.dtype.itemsize
    if win_w == src_w and array.flags.c_contiguous:
        for band in range(n_bands):
            src_ptr = array.ctypes.data + ((b0 + band) * src_h + r_lo) * src_w * item
            _native.check(lib.gm_memcpy_h2d(
                target.ptr + band * win_h * win_w * item, src_ptr, win_h * win_w * item, stream))
    else:
        strides = array.strides
        if strides[2] != item:
            array = np.ascontiguousarray(array)
            strides = array.strides
        for band in range(n_bands):
            src_ptr = array.ctypes.data + (b0 + band) * strides[0] + r_lo * strides[1] + c_lo * item
            _native.check(lib.gm_memcpy2d_h2d(
                target.ptr + band * win_h * win_w * item, win_w * item, src_ptr, strides[1],
                win_w * item, win_h, stream))


def resample_window(array, bands, geo_transform, no_data_value, bbox, height, width, keep_on_device,
                    row_range=None, origin=(0, 0)):
    """Nearest-neighbour resample of ``array[bands[0]:bands[1]]`` into the request grid.

    ``row_range=(r0, r1)`` produces only rows [r0, r1) of the request (used by the chunk
    pipeline for pixel-aligned requests, where row_step == 1 keeps the arithmetic exact).
    ``origin=(row, col)``: ``array`` holds only the part of the source that starts at that cell
    (a window decoded from a file); ``geo_transform`` is still the whole source's."""
    lib = _native.lib()
    stream = _native.current_stream()
    b0, b1 = bands
    n_bands = b1 - b0
    _, src_h, src_w = array.shape
    col0, col_step, row0, row_step = window_geometry(geo_transform, bbox, height, width)
    row0, col0 = row0 - origin[0], col0 - origin[1]
    if row_range is not None:
        row0 = row0 + row_range[0] * row_step
        height = row_range[1] - row_range[0]
    c_lo, c_hi = _window(width, col0, col_step, src_w)
    r_lo, r_hi = _window(height, row0, row_step, src_h)

    dtype = array.dtype
    out = _native.DeviceArray((n_bands, height, width), dtype)
    nodata_holder, nodata_ptr = _native.scalar_ptr(no_data_value, dtype)
    win_h, win_w = max(r_hi - r_lo, 0), max(c_hi - c_lo, 0)
    resident = None
    if win_h > 0 and win_w > 0 and n_bands > 0:
        resident = resident_copy(array)
    if win_h == 0 or win_w == 0 or n_bands == 0:
        _native.check(lib.gm_fill(out.ptr, _native.dtype_code(dtype), nodata_ptr, out.size, stream))
    elif resident is not None:
        # the whole source is in HBM: one gather from it (no upload), same arithmetic
        view = _native.DeviceArray((n_bands, src_h, src_w), dtype,
                                   ptr=resident.ptr + b0 * src_h * src_w * dtype.itemsize, owner=resident)
        src_desc = _native.as_gm_array(view)
        dst_desc = _native.as_gm_array(out)
        _native.check(lib.gm_resample_nn(
            ctypes.byref(src_desc), ctypes.byref(dst_desc), nodata_ptr,
            col0, col_step, row0, row_step, stream))
    else:
        exact = (
            dtype.kind != "f" and col_step == 1.0 and row_step == 1.0
            and c_lo == int(np.floor(col0)) and r_lo == int(np.floor(row0))
            and win_h == height and win_w == width
        )
        target = out if exact else _native.DeviceArray((n_bands, win_h, win_w), dtype)
        upload_window(array, b0, (r_lo, r_hi, c_lo, c_hi), target)
        if not exact:
            src_desc = _native.as_gm_array(target)
            dst_desc = _native.as_gm_array(out)
            _native.check(lib.gm_resample_nn(
                ctypes.byref(src_desc), ctypes.byref(dst_desc), nodata_ptr,
                col0 - c_lo, col_step, row0 - r_lo, row_step, stream))
    return out if keep_on_device else out.to_host()


WINDOW_EDGE_POINTS = 64   # outline points per edge of a request mapped into the source CRS
WINDOW_MARGIN = 2         # cells added around the mapped outline


def request_outline(bbox, n=WINDOW_EDGE_POINTS):
    """Points along the outline of a request bbox, ``n`` intervals per edge."""
    x1, y1, x2, y2 = bbox
    t = np.linspace(0.0, 1.0, n + 1)
    xs, ys = x1 + t * (x2 - x1), y1 + t * (y2 - y1)
    return np.concatenate([
        np.stack([xs, np.full_like(t, y1)], 1), np.stack([xs, np.full_like(t, y2)], 1),
        np.stack([np.full_like(t, x1), ys], 1), np.stack([np.full_like(t, x2), ys], 1),
    ])


def warp_source_window(geo_transform, bbox, projection, source_projection, src_h, src_w):
    """(r_lo, r_hi, c_lo, c_hi): the source cells a request in another CRS reads, estimated from
    its outline mapped into the source CRS plus a margin.  Cells the estimate leaves out are
    counted by the warp kernel, and the caller then repeats the warp with the whole source."""
    p, a, _, q, _, d = geo_transform
    xy = crs.transform(request_outline(bbox), projection, source_projection)
    with np.errstate(invalid="ignore"):
        cols = np.floor((xy[:, 0] - p) / a + 1e-10)
        rows = np.floor((xy[:, 1] - q) / d + 1e-10)
    finite = np.isfinite(cols) & np.isfinite(rows)
    if not finite.any():
        return 0, 0, 0, 0
    cols, rows = cols[finite], rows[finite]
    r_lo = int(np.clip(rows.min() - WINDOW_MARGIN, 0, src_h))
    r_hi = int(np.clip(rows.max() + 1 + WINDOW_MARGIN, r_lo, src_h))
    c_lo = int(np.clip(cols.min() - WINDOW_MARGIN, 0, src_w))
    c_hi = int(np.clip(cols.max() + 1 + WINDOW_MARGIN, c_lo, src_w))
    return r_lo, r_hi, c_lo, c_hi


def _warp_call(src, origin, src_shape, geo_transform, source_projection, no_data_value, bbox,
               height, width, projection, count_misses):
    """One gm_warp_nn call from the DeviceArray ``src`` (source cells from ``origin`` = (row, col)
    on) into a new DeviceArray; returns it with the number of reads outside ``src`` (None when not
    counted, which saves the stream synchronisation)."""
    (src_kind, src_zone), (dst_kind, dst_zone) = crs.crs_pair(source_projection, projection)
    warp = _native.GmWarp()
    warp.dst_kind, warp.dst_zone, warp.src_kind, warp.src_zone = dst_kind, dst_zone, src_kind, src_zone
    warp.dst_geo[:] = utils.GeoTransform.from_bbox(bbox, height, width)
    warp.src_geo[:] = geo_transform
    warp.src_height, warp.src_width = src_shape
    warp.win_row0, warp.win_col0 = origin
    out = _native.DeviceArray((src.shape[0], height, width), src.dtype)
    nodata_holder, nodata_ptr = _native.scalar_ptr(no_data_value, src.dtype)
    src_desc, dst_desc = _native.as_gm_array(src), _native.as_gm_array(out)
    misses = ctypes.c_int64(0)
    _native.check(_native.lib().gm_warp_nn(
        ctypes.byref(src_desc), ctypes.byref(dst_desc), nodata_ptr, ctypes.byref(warp),
        ctypes.byref(misses) if count_misses else None, _native.current_stream()))
    return out, (misses.value if count_misses else None)


def _count_window_miss():
    _native.STATS["warp_window_misses"] = _native.STATS.get("warp_window_misses", 0) + 1


def warp_window(array, bands, geo_transform, no_data_value, bbox, height, width, projection,
                source_projection, keep_on_device):
    """Nearest-neighbour warp of ``array[bands[0]:bands[1]]`` (a source in ``source_projection``)
    into a request grid in ``projection`` (the reference's gdal.ReprojectImage,
    raster/sources.py:119-149).  Uploads only the window the request reads, or reads the
    resident copy (``geomodeling.device-cache-bytes``)."""
    b0, b1 = bands
    n_bands = b1 - b0
    _, src_h, src_w = array.shape
    crs.crs_pair(source_projection, projection)     # unsupported pairs raise before any upload
    args = (geo_transform, source_projection, no_data_value, bbox, height, width, projection)
    resident = resident_copy(array) if n_bands > 0 else None
    if resident is not None:
        item = array.dtype.itemsize
        view = _native.DeviceArray((n_bands, src_h, src_w), array.dtype,
                                   ptr=resident.ptr + b0 * src_h * src_w * item, owner=resident)
        out, _ = _warp_call(view, (0, 0), (src_h, src_w), *args, count_misses=False)
    else:
        window = warp_source_window(geo_transform, bbox, projection, source_projection, src_h, src_w)
        r_lo, r_hi, c_lo, c_hi = window
        src = _native.DeviceArray((n_bands, r_hi - r_lo, c_hi - c_lo), array.dtype)
        upload_window(array, b0, window, src)
        out, misses = _warp_call(src, (r_lo, c_lo), (src_h, src_w), *args, count_misses=True)
        if misses:
            _count_window_miss()
            src = _native.DeviceArray((n_bands, src_h, src_w), array.dtype)
            upload_window(array, b0, (0, src_h, 0, src_w), src)
            out, _ = _warp_call(src, (0, 0), (src_h, src_w), *args, count_misses=False)
    return out if keep_on_device else out.to_host()


def point_cell(geo_transform, src_shape, bbox, projection, source_projection):
    """Cell of a point request (raster/sources.py:95-117) as (row, col), or None outside the
    source; the point is first transformed into the source CRS."""
    point = np.array([[bbox[0], bbox[1]]], dtype=np.float64)
    if not utils.same_projection(projection, source_projection):
        point = crs.transform(point, projection, source_projection)
        if not np.isfinite(point).all():
            return None
    rows, cols = geo_transform.get_indices(point)
    i, j = int(rows[0]), int(cols[0])
    return (i, j) if 0 <= i < src_shape[0] and 0 <= j < src_shape[1] else None


class RasterSourceBase(RasterBlock):
    @staticmethod
    def process(process_kwargs):
        mode = process_kwargs["mode"]
        if mode == "empty_vals":
            return None
        if mode == "empty_time":
            return {"time": []}
        if mode == "empty_meta":
            return {"meta": []}

        b0, b1 = process_kwargs["bands"]
        if mode == "time":
            start, delta = process_kwargs["start"], process_kwargs["delta"]
            return {"time": [start + i * delta for i in range(b1 - b0)]}
        dataset = None
        if "url" in process_kwargs:      # coming from a RasterFileSource block
            dataset = open_dataset(utils.safe_abspath(process_kwargs["url"]))
        if mode == "meta":
            if dataset is not None:
                return {"meta": [dataset.metadata(i) for i in range(b0, b1)]}
            return {"meta": list(process_kwargs["metadata"][b0:b1])}

        array = process_kwargs.get("array")
        dtype = process_kwargs["dtype"]
        bbox = process_kwargs["bbox"]
        width, height = process_kwargs["width"], process_kwargs["height"]
        fillvalue = process_kwargs["fillvalue"]
        # (a file without a no data tag: the dtype's maximum marks the cells outside it)
        no_data_value = utils.get_dtype_max(dtype) if fillvalue is None else fillvalue.item()
        if width == 0 or height == 0:
            return np.empty((b1 - b0, height, width), dtype=dtype)
        if dataset is not None:
            process_kwargs = dict(process_kwargs, source_projection=dataset.projection,
                                  geo_transform=dataset.geo_transform)
        projection, source_projection = process_kwargs["projection"], process_kwargs["source_projection"]
        same = utils.same_projection(projection, source_projection)
        if not same:
            crs.crs_pair(source_projection, projection)    # NotImplementedError for other CRSs
        geo_transform = utils.GeoTransform(process_kwargs["geo_transform"])
        if dataset is not None:
            return _file_values(dataset, (b0, b1), geo_transform, dtype, no_data_value, bbox, height, width,
                                projection)

        if bbox[0] == bbox[2] or bbox[1] == bbox[3]:
            # point request: the cell that contains the point (raster/sources.py:95-117)
            cell = point_cell(geo_transform, array.shape[1:], bbox, projection, source_projection)
            result = np.full((array.shape[0], 1, 1), no_data_value, dtype=dtype)
            if cell is not None:
                result[:, 0, 0] = array[:, cell[0], cell[1]]
            result = result[b0:b1]
            if result.dtype.kind == "f":
                result[~np.isfinite(result)] = no_data_value
            return {"values": result, "no_data_value": no_data_value}

        if config.get("geomodeling.pin-sources", True):
            _native.pin(array)
        if not same:
            values = warp_window(array, (b0, b1), geo_transform, no_data_value, bbox, height, width,
                                 projection, source_projection, _state.keep_on_device())
            return {"values": values, "no_data_value": no_data_value}
        values = resample_window(
            array, (b0, b1), geo_transform, no_data_value, bbox, height, width,
            _state.keep_on_device(),
        )
        return {"values": values, "no_data_value": no_data_value}


_DATASETS = {}


def open_dataset(path):
    """Header of a GeoTIFF / VRT file, kept until the file changes on disk."""
    stat = os.stat(path)
    key = (stat.st_mtime_ns, stat.st_size)
    hit = _DATASETS.get(path)
    if hit is None or hit[0] != key:
        if len(_DATASETS) >= 64:
            _DATASETS.clear()
        hit = _DATASETS[path] = (key, geotiff.open_raster(path))
    return hit[1]


def _file_values(dataset, bands, geo_transform, dtype, no_data_value, bbox, height, width, projection):
    """'vals' response of a file source: point requests read one cell, other requests inflate the
    tiles under their window and resample (or, in another projection, warp) it on the device."""
    b0, b1 = bands
    n_all, src_h, src_w = dataset.shape
    if bbox[0] == bbox[2] or bbox[1] == bbox[3]:
        cell = point_cell(geo_transform, (src_h, src_w), bbox, projection, dataset.projection)
        result = np.full((b1 - b0, 1, 1), no_data_value, dtype=dtype)
        if cell is not None:
            i, j = cell
            result[:, 0, 0] = dataset.read_window(b0, b1, i, i + 1, j, j + 1)[:, 0, 0]
        if result.dtype.kind == "f":
            result[~np.isfinite(result)] = no_data_value
        return {"values": result, "no_data_value": no_data_value}
    if not utils.same_projection(projection, dataset.projection):
        return {"values": _file_warp(dataset, bands, geo_transform, dtype, no_data_value, bbox, height,
                                     width, projection),
                "no_data_value": no_data_value}
    r_lo, r_hi, c_lo, c_hi = source_window(geo_transform, bbox, height, width, src_h, src_w)
    window = dataset.read_window(b0, b1, r_lo, r_hi, c_lo, c_hi)
    if window.dtype != dtype:
        window = window.astype(dtype)
    if window.size == 0:     # nothing of the file under the request: all no data
        window = np.empty((b1 - b0, 0, 0), dtype=dtype)
    values = resample_window(window, (0, b1 - b0), geo_transform, no_data_value, bbox, height, width,
                             _state.keep_on_device(), origin=(r_lo, c_lo))
    return {"values": values, "no_data_value": no_data_value}


def _file_warp(dataset, bands, geo_transform, dtype, no_data_value, bbox, height, width, projection):
    """Warp of a file source into a request in another CRS: the tiles under the estimated window
    are decoded; when the warp reads outside it, the whole file is."""
    b0, b1 = bands
    _, src_h, src_w = dataset.shape
    args = (geo_transform, dataset.projection, no_data_value, bbox, height, width, projection)

    def decoded(window):
        r_lo, r_hi, c_lo, c_hi = window
        host = np.ascontiguousarray(dataset.read_window(b0, b1, r_lo, r_hi, c_lo, c_hi), dtype=dtype)
        src = _native.DeviceArray((b1 - b0, r_hi - r_lo, c_hi - c_lo), dtype)
        if src.size:
            upload_window(host.reshape(src.shape), 0, (0, r_hi - r_lo, 0, c_hi - c_lo), src)
            _native.synchronize()     # the decoded window is a temporary
        return src

    window = warp_source_window(geo_transform, bbox, projection, dataset.projection, src_h, src_w)
    out, misses = _warp_call(decoded(window), (window[0], window[2]), (src_h, src_w), *args,
                             count_misses=True)
    if misses:
        _count_window_miss()
        out, _ = _warp_call(decoded((0, src_h, 0, src_w)), (0, 0), (src_h, src_w), *args,
                            count_misses=False)
    return out if _state.keep_on_device() else out.to_host()


class MemorySource(RasterSourceBase):
    """Raster held in (host) memory.

    The cell whose top-left corner is (x, y) covers [x, x + dx) x (y - dy, y].

    Args:
      data: 2D or 3D (t, y, x) array of cell values
      no_data_value: the value that marks missing data
      projection: projection of the data (EPSG code or WKT)
      pixel_size: cell size, scalar or (x, y)
      pixel_origin: (x, y) of the top-left corner of cell (0, 0)
      time_first: timestamp of the first frame (ms since epoch, or naive UTC datetime)
      time_delta: time between frames (ms or timedelta); required when t > 1
      metadata: optional list with one entry per frame
    """

    def __init__(self, data, no_data_value, projection, pixel_size, pixel_origin,
                 time_first=0, time_delta=None, metadata=None):
        data = np.asarray(data)
        if data.dtype == "i8":
            data = data.astype("i4")  # as the reference (GDAL had no int64)
        if data.ndim == 2:
            data = data[np.newaxis]
        if data.ndim != 3:
            raise ValueError("data should be two- or three-dimensional.")
        no_data_value = data.dtype.type(no_data_value)
        projection = utils.get_epsg_or_wkt(projection)
        if hasattr(pixel_size, "__iter__"):
            pixel_size = [float(x) for x in pixel_size]
            if len(pixel_size) != 2:
                raise ValueError("pixel_size should have length 2")
        else:
            pixel_size = [float(pixel_size)] * 2
        pixel_origin = [float(x) for x in pixel_origin]
        if len(pixel_origin) != 2:
            raise ValueError("pixel_origin should have length 2")
        time_first = utils.dt_to_ms(time_first) if isinstance(time_first, datetime) else int(time_first)
        if isinstance(time_delta, timedelta):
            time_delta = int(time_delta.total_seconds() * 1000)
        elif time_delta is not None:
            time_delta = int(time_delta)
        elif data.shape[0] > 1:
            raise ValueError("time_delta is required for temporal data")
        if metadata is not None:
            metadata = list(metadata)
            if len(metadata) != data.shape[0]:
                raise ValueError("Metadata length should match data length")
        super().__init__(data, no_data_value, projection, pixel_size, pixel_origin,
                         time_first, time_delta, metadata)

    data = property(lambda self: self.args[0])
    no_data_value = property(lambda self: self.args[1])
    projection = property(lambda self: self.args[2])
    pixel_size = property(lambda self: self.args[3])
    pixel_origin = property(lambda self: self.args[4])
    time_first = property(lambda self: self.args[5])
    time_delta = property(lambda self: self.args[6])
    metadata = property(lambda self: self.args[7])

    @property
    def dtype(self):
        return self.data.dtype

    @property
    def fillvalue(self):
        return self.no_data_value

    @property
    def geo_transform(self):
        (p, q), (a, d) = self.pixel_origin, self.pixel_size
        return utils.GeoTransform((p, a, 0, q, 0, -d))

    def _native_extent(self):
        if not self.data.size:
            return None
        return utils.Extent(self.geo_transform.get_bbox((0, 0), self.data.shape[1:]), self.projection)

    @property
    def extent(self):
        native = self._native_extent()
        return None if native is None else native.transformed("EPSG:4326").bbox

    @property
    def geometry(self):
        native = self._native_extent()
        return None if native is None else native.as_geometry()

    def __len__(self):
        return self.data.shape[0]

    @property
    def timedelta(self):
        return None if self.time_delta is None else timedelta(milliseconds=self.time_delta)

    @property
    def temporal(self):
        return self.time_delta is not None

    @property
    def period(self):
        n = len(self)
        if n == 0:
            return None
        first = utc_from_ms_timestamp(self.time_first)
        return (first, first) if n == 1 else (first, first + (n - 1) * self.timedelta)

    def get_sources_and_requests(self, **request):
        mode = request["mode"]
        if mode == "meta" and self.metadata is None:
            return [({"mode": "empty_meta"}, None)]
        start, stop, first_i, last_i = utils.snap_start_stop(
            request.get("start"), request.get("stop"),
            utc_from_ms_timestamp(self.time_first), self.timedelta, len(self),
        )
        if start is None:
            return [({"mode": "empty_" + mode}, None)]
        bands = (first_i, last_i + 1)
        if mode == "vals":
            kwargs = {
                "mode": "vals",
                "array": self.data,
                "geo_transform": tuple(self.geo_transform),
                "source_projection": self.projection,
                "bbox": request["bbox"],
                "width": request["width"],
                "height": request["height"],
                "projection": request["projection"],
                "bands": bands,
                "dtype": self.dtype,
                "fillvalue": self.fillvalue,
            }
        elif mode == "meta":
            kwargs = {"mode": "meta", "metadata": self.metadata, "bands": bands}
        elif mode == "time":
            kwargs = {"mode": "time", "start": start, "delta": self.timedelta or timedelta(0),
                      "bands": bands}
        else:
            raise RuntimeError("Unknown mode '{}'".format(mode))
        return [(kwargs, None)]


class RasterFileSource(RasterSourceBase):
    """A raster source that interfaces data from a file path (GeoTIFF or VRT).

    The value at raster cell with its topleft corner at [x, y] is assumed to define a value for
    ranges [x, x + dx) and (y - dy, y].

    :param url: the path to the file, inside the ``geomodeling.root`` setting when relative
    :param time_first: the timestamp of the first frame (ms since 1-1-1970 or datetime)
    :param time_delta: the difference between two consecutive frames (ms or timedelta),
        defaults to 5 minutes

    The object keeps the parsed file header; ``close_dataset`` drops it.
    """

    def __init__(self, url, time_first=0, time_delta=300000):
        url = utils.safe_file_url(url)
        time_first = utils.dt_to_ms(time_first) if isinstance(time_first, datetime) else int(time_first)
        if isinstance(time_delta, timedelta):
            time_delta = int(time_delta.total_seconds() * 1000)
        else:
            time_delta = int(time_delta)
        super().__init__(url, time_first, time_delta)

    url = property(lambda self: self.args[0])
    time_first = property(lambda self: self.args[1])
    time_delta = property(lambda self: self.args[2])

    @property
    def dataset(self):
        try:
            return self._dataset
        except AttributeError:
            self._dataset = open_dataset(utils.safe_abspath(self.url))
            return self._dataset

    gdal_dataset = dataset     # the reference's name for the open file

    def close_dataset(self):
        if hasattr(self, "_dataset"):
            del self._dataset

    @property
    def projection(self):
        return self.dataset.projection

    @property
    def dtype(self):
        return self.dataset.dtype

    @property
    def fillvalue(self):
        value = self.dataset.no_data_value
        return None if value is None else self.dtype.type(value)

    @property
    def geo_transform(self):
        return utils.GeoTransform(self.dataset.geo_transform)

    def _get_extent(self):
        bbox = self.geo_transform.get_bbox((0, 0), (self.dataset.height, self.dataset.width))
        return utils.Extent(bbox, self.projection)

    @property
    def extent(self):
        return self._get_extent().transformed("EPSG:4326").bbox

    @property
    def geometry(self):
        return self._get_extent().as_geometry()

    def __len__(self):
        return self.dataset.bands

    @property
    def period(self):
        n = len(self)
        if n == 0:
            return None
        first = utc_from_ms_timestamp(self.time_first)
        return (first, first) if n == 1 else (first, first + (n - 1) * self.timedelta)

    @property
    def timedelta(self):
        return None if len(self) <= 1 else timedelta(milliseconds=self.time_delta)

    @property
    def temporal(self):
        return len(self) > 1

    def get_sources_and_requests(self, **request):
        mode = request["mode"]
        start, stop, first_i, last_i = utils.snap_start_stop(
            request.get("start"), request.get("stop"),
            utc_from_ms_timestamp(self.time_first), self.timedelta, len(self),
        )
        if start is None:
            return [({"mode": "empty_" + mode}, None)]
        bands = (first_i, last_i + 1)
        if mode == "vals":
            kwargs = {"mode": "vals", "url": self.url, "bbox": request["bbox"], "width": request["width"],
                      "height": request["height"], "projection": request["projection"], "bands": bands,
                      "dtype": self.dtype, "fillvalue": self.fillvalue}
        elif mode == "meta":
            kwargs = {"mode": "meta", "url": self.url, "bands": bands}
        elif mode == "time":
            kwargs = {"mode": "time", "start": start, "delta": self.timedelta or timedelta(0), "bands": bands}
        else:
            raise RuntimeError("Unknown mode '{}'".format(mode))
        return [(kwargs, None)]
