"""Spatial stencil blocks: Dilate, MovingMax, Smooth, HillShade.

Drop-in for the stencil part of the reference's raster/spatial.py (``Place`` is
outside the hot path).  Each block enlarges the request by its halo exactly as
the reference does -- the halo is obtained by asking the source for a larger
bbox, not by neighbour communication (raster/spatial.py:27-108) -- and the
stencil itself runs in CUDA (csrc/gm_stencil.cu).
"""
import ctypes

import numpy as np

from .. import _native, _state, utils
from . import _program
from .base import BaseSingle

__all__ = ["Dilate", "Smooth", "MovingMax", "HillShade", "Place"]


def expand_request_pixels(request, radius=1):
    """Request enlarged by ``radius`` pixels on every side; None for non-'vals'
    and point requests.

    The bbox mixes the x and y amounts exactly as the reference does
    (raster/spatial.py:44); identical for square pixels."""
    if request["mode"] != "vals":
        return None
    width, height = request["width"], request["height"]
    x1, y1, x2, y2 = request["bbox"]
    span_x, span_y = x2 - x1, y2 - y1
    if span_x == 0 or span_y == 0:
        return None
    amount_x = span_x / width * radius
    amount_y = span_y / height * radius
    enlarged = request.copy()
    enlarged["bbox"] = (x1 - amount_x, y1 - amount_x, x2 + amount_y, y2 + amount_y)
    enlarged["width"] = width + 2 * radius
    enlarged["height"] = height + 2 * radius
    return enlarged


def expand_request_meters(request, radius_m=1):
    """Request enlarged by ``radius_m`` metres rounded to whole pixels.

    Returns (new request, radius in pixels as (y, x) floats)
    (raster/spatial.py:50-108).  Geographic projections would need a detour via
    EPSG:3857, i.e. a coordinate transformation, and are not supported here."""
    if utils.is_geographic(request["projection"]):
        raise NotImplementedError("Smooth on a geographic projection needs pyproj/GDAL")
    x1, y1, x2, y2 = request["bbox"]
    span_y, span_x = y2 - y1, x2 - x1
    if span_y > 0 and span_x > 0:
        per_m = request["height"] / span_y, request["width"] / span_x
        radius_px = [radius_m * r for r in per_m]
        margins_px = [int(round(r)) for r in radius_px]
        margins_m = [m / r for m, r in zip(margins_px, per_m)]
    else:
        radius_px = margins_px = [Smooth.MARGIN_THRESHOLD] * 2
        margins_m = [radius_m] * 2
    enlarged = request.copy()
    enlarged["bbox"] = (x1 - margins_m[1], y1 - margins_m[0], x2 + margins_m[1], y2 + margins_m[0])
    enlarged["height"] = request["height"] + 2 * margins_px[0]
    enlarged["width"] = request["width"] + 2 * margins_px[1]
    return enlarged, radius_px


def _call_stencil(values, out_shape, out_dtype, launch):
    """Allocate the output next to the input (device stays device, host stays
    host unless a graph is being computed) and run ``launch(src, dst, stream)``."""
    lib = _native.lib()
    on_device = _native.is_device(values) or _state.keep_on_device()
    if on_device and not _native.is_device(values):
        values = _native.DeviceArray.from_host(values)
    if not on_device:
        values = np.ascontiguousarray(values)
    target = _state.row_window() if on_device and out_shape[0] == 1 else None
    if target is not None:
        # a row window of a larger output (parallel.stencil_haloed computes the interior of a
        # stripe while its halo rows travel): the full raster is allocated once, this call
        # writes rows [r0, r0 + rows)
        if target.out is None:
            target.out = _native.DeviceArray((1, target.full_rows, out_shape[2]), out_dtype)
        full = target.out
        if full.dtype != np.dtype(out_dtype) or full.shape[2] != out_shape[2] or \
                target.r0 < 0 or target.r0 + out_shape[1] > full.shape[1]:
            raise ValueError("stencil row window does not fit its output raster")
        out = _native.DeviceArray(out_shape, out_dtype, owner=full,
                                  ptr=full.ptr + target.r0 * out_shape[2] * np.dtype(out_dtype).itemsize)
        src, dst = _native.as_gm_array(values), _native.as_gm_array(out)
        _native.check(launch(lib, ctypes.byref(src), ctypes.byref(dst), _native.current_stream()))
        return out
    out = (_native.DeviceArray(out_shape, out_dtype) if on_device
           else _native.pinned_empty(out_shape, out_dtype))
    src, dst = _native.as_gm_array(values), _native.as_gm_array(out)
    _native.check(launch(lib, ctypes.byref(src), ctypes.byref(dst), _native.current_stream()))
    if on_device and not _state.keep_on_device():
        out = out.to_host()
    return out


def _nodata_arg(values, no_data_value):
    """(holder, pointer, has_nodata) for ``values == no_data_value`` in the array dtype."""
    from ._program import sentinel

    s = sentinel(values.dtype, no_data_value)
    holder, ptr = _native.scalar_ptr(0 if s is None else s, values.dtype)
    return holder, ptr, int(s is not None)


class Dilate(BaseSingle):
    """Grow cells holding one of ``values`` by one cell (6-connected in t, y, x),
    later values on top (reference: raster/spatial.py:111-155)."""

    def __init__(self, store, values):
        values = np.asarray(values, dtype=store.dtype)
        super().__init__(store, values.tolist())

    values = property(lambda self: self.args[1])

    def get_sources_and_requests(self, **request):
        enlarged = expand_request_pixels(request, radius=1)
        if enlarged is None:
            return [(self.store, request)]
        return [(self.store, enlarged), (self.values, None)]

    @staticmethod
    def process(data, values=None):
        if data is None or values is None or "values" not in data:
            return data
        source = data["values"]
        wanted = np.ascontiguousarray(np.asarray(values, dtype=source.dtype)).reshape(-1)
        t, h, w = source.shape
        out = _call_stencil(
            source, (t, h - 2, w - 2), source.dtype,
            lambda lib, src, dst, stream: lib.gm_dilate(src, dst, wanted.ctypes.data, len(wanted), stream),
        )
        return {"values": out, "no_data_value": data["no_data_value"]}


class MovingMax(BaseSingle):
    """Maximum over a disc of (odd) diameter ``size``
    (reference: raster/spatial.py:158-213)."""

    def __init__(self, store, size):
        size = int(2 * round((size - 1) / 2) + 1)  # nearest odd integer
        if size < 3:
            raise ValueError("The size should be odd and larger than 1")
        super(MovingMax, self).__init__(store, size)

    size = property(lambda self: self.args[1])

    def get_sources_and_requests(self, **request):
        radius = int(self.size // 2)
        enlarged = expand_request_pixels(request, radius=radius)
        if enlarged is None:
            return [(self.store, request)]
        # 4-byte rasters: ask for a few more columns on the right so that a row of the window is
        # a whole number of 16-byte groups -- the kernel then stages its tiles by TMA (a tensor
        # map needs a 16-byte row pitch); the extra columns are never part of a footprint
        pad = 0
        if np.dtype(self.dtype).itemsize == 4 and self.size <= 15:
            pad = (-enlarged["width"]) % 4
        if pad:
            x1, y1, x2, y2 = enlarged["bbox"]
            cell = (request["bbox"][2] - request["bbox"][0]) / request["width"]
            enlarged["bbox"] = (x1, y1, x2 + pad * cell, y2)
            enlarged["width"] += pad
        return [(self.store, enlarged), (self.size, None), (pad, None)]

    @staticmethod
    def process(data, size=None, pad=0):
        if data is None or size is None or "values" not in data:
            return data
        source = data["values"]
        radius = int(size // 2)
        t, h, w = source.shape
        holder, nodata_ptr, has_nodata = _nodata_arg(source, data["no_data_value"])
        out = _call_stencil(
            source, (t, h - 2 * radius, w - 2 * radius - int(pad)), source.dtype,
            lambda lib, src, dst, stream: lib.gm_moving_max(src, dst, nodata_ptr, has_nodata,
                                                            int(size), stream),
        )
        return {"values": out, "no_data_value": data["no_data_value"]}


def _gaussian_weights(sigma):
    """scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, radius) with
    radius = int(4 * sigma + 0.5); (weights, radius).  sigma <= 1e-15: axis skipped."""
    if sigma <= 1e-15:
        return np.ones(1, dtype=np.float64), 0
    radius = int(4.0 * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return np.ascontiguousarray(phi / phi.sum()), radius


class Smooth(BaseSingle):
    """Gaussian smoothing with sigma = size / 3 (in projection units)
    (reference: raster/spatial.py:216-307)."""

    MARGIN_THRESHOLD = 6

    def __init__(self, store, size, fill=0):
        for x in (size, fill):
            if not isinstance(x, (int, float)):
                raise TypeError("'{}' object is not allowed".format(type(x)))
        super(Smooth, self).__init__(store, size, fill)

    size = property(lambda self: self.args[1])
    fill = property(lambda self: self.args[2])

    def get_sources_and_requests(self, **request):
        if request["mode"] != "vals":
            return [(self.store, request)]
        enlarged, size_px = expand_request_meters(request, self.size)
        if any(s > self.MARGIN_THRESHOLD for s in size_px):
            # large kernels: smooth a coarser grid over the enlarged extent, zoom back
            mode = "zoom"
            zoom = [enlarged[k] / request[k] for k in ("height", "width")]
            size_px = [s / z for s, z in zip(size_px, zoom)]
            enlarged["height"], enlarged["width"] = request["height"], request["width"]
        else:
            mode = "exact"
        return [(self.store, enlarged), (dict(smooth_mode=mode, fill=self.fill, size=size_px), None)]

    @staticmethod
    def process(data, process_kwargs=None):
        if data is None or process_kwargs is None:
            return data
        mode = process_kwargs["smooth_mode"]
        size_px = process_kwargs["size"]
        fill = process_kwargs["fill"]
        source = data["values"]
        t, ny, nx = source.shape
        wy, ly = _gaussian_weights(size_px[0] / 3)
        wx, lx = _gaussian_weights(size_px[1] / 3)
        holder, nodata_ptr, has_nodata = _nodata_arg(source, data["no_data_value"])
        if mode == "exact":
            # "margin" (rows, cols) overrides the cropped halo: row stripes carry the full
            # filter radius from their neighbours (parallel.stencil_striped)
            my, mx = process_kwargs.get("margin") or [int(round(s)) for s in size_px]
            out_shape = (t, ny - 2 * my, nx - 2 * mx)
            zoom, zy, zx, oy, ox = 0, 1.0, 1.0, 0.0, 0.0
        else:
            my = mx = 0
            out_shape = (t, ny, nx)
            zoom, zy, zx = 1, 1 - 2 * size_px[0] / ny, 1 - 2 * size_px[1] / nx
            oy, ox = float(size_px[0]), float(size_px[1])
        out = _call_stencil(
            source, out_shape, source.dtype,
            lambda lib, src, dst, stream: lib.gm_smooth(
                src, dst, nodata_ptr, has_nodata, float(fill), wy.ctypes.data, ly, wx.ctypes.data, lx,
                my, mx, zoom, zy, zx, oy, ox, stream),
        )
        return {"values": out, "no_data_value": data["no_data_value"]}


class HillShade(BaseSingle):
    """Hillshade (Horn) of an elevation raster, uint8 output
    (reference: raster/spatial.py:310-438)."""

    def __init__(self, store, altitude=45, azimuth=315, fill=0):
        for x in (altitude, azimuth, fill):
            if not isinstance(x, (int, float)):
                raise TypeError("'{}' object is not allowed".format(type(x)))
        super(HillShade, self).__init__(store, float(altitude), float(azimuth), fill)

    altitude = property(lambda self: self.args[1])
    azimuth = property(lambda self: self.args[2])
    fill = property(lambda self: self.args[3])
    dtype = np.dtype("u1")
    fillvalue = 256  # on purpose not representable in uint8: the result has no 'no data'

    def get_sources_and_requests(self, **request):
        enlarged = expand_request_pixels(request, radius=1)
        if enlarged is None:
            return [(self.store, request)]
        x1, y1, x2, y2 = request["bbox"]
        resolution = ((x2 - x1) / request["width"], (y2 - y1) / request["height"])
        # 4-byte rasters: a few more columns on the right make a row of the window a whole number
        # of 16-byte groups -- a lane of the kernel then reads its four columns with one load
        pad = (-enlarged["width"]) % 4 if np.dtype(self.store.dtype).itemsize == 4 else 0
        if pad:
            ex1, ey1, ex2, ey2 = enlarged["bbox"]
            enlarged["bbox"] = (ex1, ey1, ex2 + pad * resolution[0], ey2)
            enlarged["width"] += pad
        kwargs = dict(resolution=resolution, altitude=self.altitude, azimuth=self.azimuth,
                      fill=self.fill, pad=pad)
        return [(self.store, enlarged), (kwargs, None)]

    @staticmethod
    def process(data, process_kwargs=None):
        if process_kwargs is None:
            return data
        source = data["values"]
        t, h, w = source.shape
        xres, yres = process_kwargs["resolution"]
        holder, nodata_ptr, has_nodata = _nodata_arg(source, data["no_data_value"])
        out = _call_stencil(
            source, (t, h - 2, w - 2 - int(process_kwargs.get("pad", 0))), np.uint8,
            lambda lib, src, dst, stream: lib.gm_hillshade(
                src, dst, nodata_ptr, has_nodata, float(process_kwargs["fill"]), float(xres),
                float(yres), float(process_kwargs["altitude"]), float(process_kwargs["azimuth"]),
                stream),
        )
        return {"values": out, "no_data_value": 256}


class Place(BaseSingle):
    """Place a raster at given coordinates: the cell of ``store`` under ``anchor`` lands on each
    of ``coordinates``; where copies overlap they are merged with ``statistic``
    (reference: raster/spatial.py:440-731).

    The reference scatters the store's data cells into a fresh array per coordinate (np.where
    indices, :679-719) and merges the stack with ``reduce_rasters``.  Here a copy is one
    integer-shift gather on the device (``gm_resample_nn`` with unit steps) and the merge is the
    reduction program of raster/reduction.py.  Anchor and coordinates must be given in the
    projection of the request (this build has no PROJ)."""

    def __init__(self, store, place_projection, anchor, coordinates, statistic="last"):
        from .base import RasterBlock
        from .reduction import check_statistic

        if not isinstance(store, RasterBlock):
            raise TypeError("'{}' object is not allowed".format(type(store)))
        if not isinstance(place_projection, str) or not place_projection.strip():
            raise ValueError("'{}' is not a valid projection string".format(place_projection))
        anchor = list(anchor)
        if len(anchor) != 2:
            raise ValueError("Expected 2 numbers in the 'anchor' parameter")
        for x in anchor:
            if not isinstance(x, (int, float)):
                raise TypeError("'{}' object is not allowed".format(type(x)))
        if coordinates is None or len(coordinates) == 0:
            coordinates = []
        else:
            coordinates = np.asarray(coordinates, dtype=float)
            if coordinates.ndim != 2 or coordinates.shape[1] != 2:
                raise ValueError("Expected a list of lists of 2 numbers in the 'coordinates' parameter")
            coordinates = coordinates.tolist()
        check_statistic(statistic)
        super().__init__(store, utils.get_epsg_or_wkt(place_projection), anchor, coordinates, statistic)

    place_projection = property(lambda self: self.args[1])
    anchor = property(lambda self: self.args[2])
    coordinates = property(lambda self: self.args[3])
    statistic = property(lambda self: self.args[4])

    @property
    def projection(self):
        store_projection = self.store.projection
        if store_projection is not None and utils.same_projection(self.place_projection, store_projection):
            return store_projection
        return None

    @property
    def geo_transform(self):
        return self.store.geo_transform if self.projection is not None else None

    @property
    def geometry(self):
        store_geometry = self.store.geometry
        if store_geometry is None or not self.coordinates:
            return None
        x1, y1, x2, y2 = utils.Extent.from_geometry(store_geometry).transformed(self.place_projection).bbox
        p, q = self.anchor
        xs, ys = zip(*self.coordinates)
        return utils.Extent((x1 + min(xs) - p, y1 + min(ys) - q, x2 + max(xs) - p, y2 + max(ys) - q),
                            self.place_projection).as_geometry()

    @property
    def extent(self):
        geometry = self.geometry
        if geometry is None:
            return None
        return utils.Extent.from_geometry(geometry, self.place_projection).transformed("EPSG:4326").bbox

    def get_sources_and_requests(self, **request):
        import math

        if request["mode"] != "vals":
            return ({"mode": request["mode"]}, None), (self.store, request)
        if not utils.same_projection(self.place_projection, request["projection"]):
            raise NotImplementedError(
                "Place: anchor / coordinates in {} cannot be transformed to {} (no PROJ in this build)".format(
                    self.place_projection, request["projection"]))
        anchor, coordinates = tuple(self.anchor), [tuple(c) for c in self.coordinates]
        source_geometry = self.store.geometry
        if source_geometry is None:
            return (({"mode": "null"}, None),)
        xmin, ymin, xmax, ymax = utils.Extent.from_geometry(source_geometry).transformed(request["projection"]).bbox
        x1, y1, x2, y2 = request["bbox"]
        size_x, size_y = (x2 - x1) / request["width"], (y2 - y1) / request["height"]
        if size_x > 0 and size_y > 0:
            # when the whole store is smaller than the request: fetch it once, shift it on the device
            full_height = math.ceil((ymax - ymin) / size_y)
            full_width = math.ceil((xmax - xmin) / size_x)
            if full_height * full_width <= request["width"] * request["height"]:
                whole = dict(request, width=full_width, height=full_height,
                             bbox=(xmin, ymin, xmin + full_width * size_x, ymin + full_height * size_y))
                kwargs = {"mode": "warp", "anchor": anchor, "coordinates": coordinates, "src_bbox": whole["bbox"],
                          "dst_bbox": request["bbox"], "cellsize": (size_x, size_y), "statistic": self.statistic}
                return [(kwargs, None), (self.store, whole)]
        # otherwise: one request per coordinate, shifted backwards by (coordinate - anchor)
        shifted = []
        for cx, cy in coordinates:
            bbox = [x1 + anchor[0] - cx, y1 + anchor[1] - cy, x2 + anchor[0] - cx, y2 + anchor[1] - cy]
            # cells span [xmin, xmax) x (ymin, ymax]: a box that only touches xmax / ymin holds no data
            if bbox[0] >= xmax or bbox[1] > ymax or bbox[2] < xmin or bbox[3] <= ymin:
                continue
            shifted.append((self.store, dict(request, bbox=bbox)))
        if not shifted:
            kwargs = {"mode": "empty", "dtype": self.dtype, "fillvalue": self.fillvalue,
                      "width": request["width"], "height": request["height"], "statistic": self.statistic}
            return [(kwargs, None), (self.store, dict(request, mode="time"))]
        return [({"mode": "group", "statistic": self.statistic}, None)] + shifted

    @staticmethod
    def process(process_kwargs, *multi):
        from .reduction import device_statistic, reduce_rasters

        mode = process_kwargs["mode"]
        if mode in ("meta", "time"):
            return multi[0]
        if mode == "null":
            return None
        if mode == "empty":
            data = multi[0]
            if data is None:
                return None
            shape = (len(data["time"]), process_kwargs["height"], process_kwargs["width"])
            fill, dtype = process_kwargs["fillvalue"], process_kwargs["dtype"]
            return {"values": np.full(shape, fill, dtype), "no_data_value": fill}
        if mode == "group":
            stack = [d for d in multi if d is not None]
            if not stack:
                return None
            return reduce_rasters(stack, process_kwargs["statistic"])
        # "warp": ONE source raster (cell size already that of the request), shifted per coordinate
        data = multi[0]
        if data is None:
            return None
        source, nodata = data["values"], data["no_data_value"]
        dtype = source.dtype
        size_x, size_y = process_kwargs["cellsize"]
        anchor, src_bbox = process_kwargs["anchor"], process_kwargs["src_bbox"]
        anchor_px = ((anchor[0] - src_bbox[0]) / size_x, (anchor[1] - src_bbox[1]) / size_y)
        x1, y1, x2, y2 = process_kwargs["dst_bbox"]
        dst_h, dst_w = round((y2 - y1) / size_y), round((x2 - x1) / size_x)
        depth, src_h, src_w = source.shape
        shape = (depth, dst_h, dst_w)
        offsets = []
        for cx, cy in process_kwargs["coordinates"]:
            di = round((cx - x1) / size_x - anchor_px[0])
            dj = round((cy - y1) / size_y - anchor_px[1])
            dj = dst_h - src_h - dj          # rows count from the northern edge
            if di <= -src_w or di >= dst_w or dj <= -src_h or dj >= dst_h:
                continue                      # shifted completely outside
            offsets.append((di, dj))
        if not offsets:
            return {"values": np.full(shape, nodata, dtype), "no_data_value": nodata}
        # out[:, j, i] = reduction over the copies of source[:, j - dj, i - di]; outside the source
        # and at non-finite source cells a copy holds 'nodata' (as gm_resample_nn fills it)
        statistic = device_statistic(process_kwargs["statistic"])
        if statistic == "first":
            offsets = offsets[::-1]
        if statistic in _program.STACK_STATS:
            # mean / var / std / argmin / argmax: a copy enters the stack when it puts a data cell
            # inside the request, so argmin / argmax count only those copies (gm_place_stat)
            place, args = _native.lib().gm_place_stat, _program.stack_stat_params(statistic, dtype, nodata)
        else:
            place, args = _native.lib().gm_place, _program.stack_params(statistic, dtype, nodata)
        if not _native.is_device(source):
            source = _native.DeviceArray.from_host(np.ascontiguousarray(source))
        holder, nodata_ptr = _native.scalar_ptr(nodata, dtype)
        test = _program.stack_input(source, nodata)
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        out = _native.DeviceArray(shape, dtype)
        _native.check(place(
            ctypes.byref(_native.as_gm_array(source)), ctypes.byref(_native.as_gm_array(out)), nodata_ptr,
            offsets.ctypes.data, len(offsets), ctypes.byref(test), *args, _native.current_stream()))
        return {"values": out if _state.keep_on_device() else out.to_host(), "no_data_value": nodata}
