"""ctypes binding of libgeokernels.so (the C ABI in include/geokernels.h).

There is deliberately no CPU fallback: importing this module is cheap, but the
first call into the library raises ``NativeLibraryError`` when the shared
object is missing or no sm_100 device is present.
"""
import ctypes
import os
import threading
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgeokernels.so")

GM_HOST, GM_DEVICE = 0, 1

# storage dtypes (GmDType)
_DTYPE_CODES = {
    "bool": 0, "uint8": 1, "int8": 2, "uint16": 3, "int16": 4,
    "uint32": 5, "int32": 6, "int64": 7, "float32": 8, "float64": 9,
}
_CODE_DTYPES = {v: np.dtype(k) for k, v in _DTYPE_CODES.items()}


class NativeLibraryError(RuntimeError):
    pass


def dtype_code(dtype):
    name = np.dtype(dtype).name
    try:
        return _DTYPE_CODES[name]
    except KeyError:
        raise TypeError("dtype '{}' is not supported by the CUDA raster path".format(name))


class GmArray(ctypes.Structure):
    _fields_ = [
        ("data", ctypes.c_void_p),
        ("dtype", ctypes.c_int32),
        ("space", ctypes.c_int32),
        ("shape", ctypes.c_int64 * 3),
    ]


class GmInstr(ctypes.Structure):
    _fields_ = [
        ("op", ctypes.c_uint8),
        ("cls", ctypes.c_uint8),
        ("cls_a", ctypes.c_uint8),
        ("cls_b", ctypes.c_uint8),
        ("cls_out", ctypes.c_uint8),
        ("src_kind", ctypes.c_uint8),
        ("src", ctypes.c_uint8),
        ("flags", ctypes.c_uint8),
        ("aux", ctypes.c_uint32),
        ("reserved", ctypes.c_uint32),
        ("k", ctypes.c_uint64 * 6),
    ]


class GmTable(ctypes.Structure):
    _fields_ = [
        ("keys", ctypes.c_void_p),
        ("vals", ctypes.c_void_p),
        ("hit", ctypes.c_void_p),
        ("base", ctypes.c_int64),
        ("n", ctypes.c_int32),
        ("kind", ctypes.c_int32),
    ]


GM_NREG, GM_MAX_INSTR, GM_MAX_INPUTS, GM_MAX_OUTPUTS, GM_MAX_TABLES = 4, 40, 8, 4, 2


class GmProgram(ctypes.Structure):
    _fields_ = [
        ("n_instr", ctypes.c_int32),
        ("n_inputs", ctypes.c_int32),
        ("n_outputs", ctypes.c_int32),
        ("word", ctypes.c_int32),
        ("n_tables", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("instr", GmInstr * GM_MAX_INSTR),
        ("tables", GmTable * GM_MAX_TABLES),
    ]


class GmPolygons(ctypes.Structure):
    _fields_ = [
        ("xy", ctypes.c_void_p),
        ("ring_offsets", ctypes.c_void_p),
        ("poly_offsets", ctypes.c_void_p),
        ("n_polygons", ctypes.c_int64),
        ("n_rings", ctypes.c_int64),
        ("n_vertices", ctypes.c_int64),
        ("resident", ctypes.c_void_p),
    ]


class GmZonalPartial(ctypes.Structure):
    _fields_ = [
        ("count", ctypes.c_int64),
        ("sum", ctypes.c_double),
        ("vmin", ctypes.c_double),
        ("vmax", ctypes.c_double),
    ]


class GmWarp(ctypes.Structure):
    _fields_ = [
        ("dst_kind", ctypes.c_int32),
        ("dst_zone", ctypes.c_int32),
        ("src_kind", ctypes.c_int32),
        ("src_zone", ctypes.c_int32),
        ("dst_geo", ctypes.c_double * 6),
        ("src_geo", ctypes.c_double * 6),
        ("src_height", ctypes.c_int64),
        ("src_width", ctypes.c_int64),
        ("win_row0", ctypes.c_int64),
        ("win_col0", ctypes.c_int64),
    ]


class GmStackInput(ctypes.Structure):
    _fields_ = [
        ("data", ctypes.c_void_p),
        ("dtype", ctypes.c_int32),
        ("cls", ctypes.c_uint8),
        ("flags", ctypes.c_uint8),
        ("reserved", ctypes.c_uint16),
        ("k2", ctypes.c_uint64),
        ("k4", ctypes.c_uint64),
    ]


# every symbol include/geokernels.h declares: name -> (restype, argtypes)
_vp, _i, _i64, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
_P = ctypes.POINTER
SYMBOLS = {
    "gm_abi_version": (_i, []),
    "gm_init": (_i, [_i]),
    "gm_shutdown": (_i, []),
    "gm_last_error": (ctypes.c_char_p, []),
    "gm_device_info": (_i, [_P(_i), _P(_i64), _P(_i), _P(_i)]),
    "gm_launch_count": (_i64, []),
    "gm_default_stream": (_vp, []),
    "gm_stream_sync": (_i, [_vp]),
    "gm_malloc": (_i, [_P(_vp), _i64, _vp]),
    "gm_free": (_i, [_vp, _vp]),
    "gm_host_alloc": (_i, [_P(_vp), _i64]),
    "gm_host_free": (_i, [_vp]),
    "gm_host_register": (_i, [_vp, _i64]),
    "gm_host_unregister": (_i, [_vp]),
    "gm_memcpy_h2d": (_i, [_vp, _vp, _i64, _vp]),
    "gm_memcpy_d2h": (_i, [_vp, _vp, _i64, _vp]),
    "gm_memcpy_d2d": (_i, [_vp, _vp, _i64, _vp]),
    "gm_memcpy_d2h_async": (_i, [_vp, _vp, _i64, _vp]),
    "gm_stream_create": (_i, [_P(_vp)]),
    "gm_stream_destroy": (_i, [_vp]),
    "gm_memcpy2d_h2d": (_i, [_vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "gm_fill": (_i, [_vp, ctypes.c_int32, _vp, _i64, _vp]),
    "gm_eval_program": (_i, [_P(GmProgram), _P(GmArray), _P(GmArray), _i64, _vp]),
    "gm_set_eval_mode": (_i, [_i]),
    "gm_get_eval_mode": (_i, []),
    "gm_jit_source": (_i, [_P(GmProgram), _P(ctypes.c_int32), _P(ctypes.c_int32), ctypes.c_char_p, _i64,
                           _P(_i64)]),
    "gm_jit_baked_source": (_i, [_P(GmProgram), _P(ctypes.c_int32), _P(ctypes.c_int32), ctypes.c_char_p, _i64,
                                 _P(_i64)]),
    "gm_jit_check": (_i, [_P(GmProgram), _P(ctypes.c_int32), _P(ctypes.c_int32), _P(_i64)]),
    "gm_jit_compile_count": (_i64, []),
    "gm_reduce_stack": (_i, [_P(GmStackInput), _i64, _i, _i, ctypes.c_uint64, ctypes.c_uint64, _P(GmArray), _vp]),
    "gm_place": (_i, [_P(GmArray), _P(GmArray), _vp, _vp, _i64, _P(GmStackInput), _i, _i, ctypes.c_uint64,
                      ctypes.c_uint64, _vp]),
    "gm_reduce_stack_stat": (_i, [_P(GmStackInput), _i64, _i, _i, ctypes.c_uint64, _P(GmArray), _vp]),
    "gm_place_stat": (_i, [_P(GmArray), _P(GmArray), _vp, _vp, _i64, _P(GmStackInput), _i, _i, ctypes.c_uint64,
                           _vp]),
    "gm_resample_nn": (_i, [_P(GmArray), _P(GmArray), _vp, _d, _d, _d, _d, _vp]),
    "gm_warp_nn": (_i, [_P(GmArray), _P(GmArray), _vp, _P(GmWarp), _P(_i64), _vp]),
    "gm_hillshade": (_i, [_P(GmArray), _P(GmArray), _vp, _i, _d, _d, _d, _d, _d, _vp]),
    "gm_moving_max": (_i, [_P(GmArray), _P(GmArray), _vp, _i, _i, _vp]),
    "gm_dilate": (_i, [_P(GmArray), _P(GmArray), _vp, _i, _vp]),
    "gm_set_smooth_mode": (_i, [_i]),
    "gm_get_smooth_mode": (_i, []),
    "gm_smooth": (_i, [_P(GmArray), _P(GmArray), _vp, _i, _d, _vp, _i, _vp, _i, _i, _i, _i,
                       _d, _d, _d, _d, _vp]),
    "gm_temporal_aggregate": (_i, [_P(GmArray), _P(GmArray), _vp, _i, _i, _d, _vp, _vp, _i, _vp]),
    "gm_temporal_cumulative": (_i, [_P(GmArray), _P(GmArray), _vp, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "gm_rasterize_polygons": (_i, [_P(GmPolygons), _P(_d), _vp, _vp, _P(GmArray), _vp]),
    "gm_zonal_stats": (_i, [_P(GmArray), _vp, _i, _P(GmPolygons), _P(_d), _i, _d, _vp,
                            _i64, _i64, _vp, _vp, _vp, _vp]),
    "gm_polygons_upload": (_i, [_P(GmPolygons), _P(_vp)]),
    "gm_polygons_free": (_i, [_vp]),
    "gm_zonal_values": (_i, [_P(GmArray), _vp, _i, _P(GmPolygons), _P(_d), _vp, _vp, _vp, _vp]),
    "gm_segment_order_stat": (_i, [_vp, ctypes.c_int32, _vp, _i64, _i, _d, _vp, _vp]),
    "gm_zonal_partials_device": (_i, [_P(GmArray), _vp, _i, _P(GmPolygons), _P(_d), _vp, _i64, _i64,
                                      _vp, _vp, _i, _vp]),
    "gm_zonal_finalize_device": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _P(GmPolygons), _vp]),
}

_lib = None
_lib_lock = threading.Lock()
_initialised = False


def load_library():
    """dlopen the library and declare prototypes (no CUDA call is made)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                "{} not found: build it with `python -m dask_geomodeling_b200.csrc.build` "
                "(there is no CPU fallback)".format(LIB_PATH)
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.gm_abi_version() != 1:
            raise NativeLibraryError("libgeokernels.so ABI version mismatch")
        _lib = lib
    return _lib


def lib():
    """The library with the device initialised; raises loudly when impossible."""
    global _initialised
    handle = load_library()
    if not _initialised:
        device = int(os.environ.get("GM_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        if handle.gm_init(device) != 0:
            raise NativeLibraryError(handle.gm_last_error().decode())
        _initialised = True
    return handle


def check(rc):
    if rc != 0:
        raise NativeLibraryError(_lib.gm_last_error().decode())


_stream = threading.local()


def current_stream():
    """cudaStream_t (int) used for calls from this thread; 0/None = library stream."""
    return getattr(_stream, "value", None)


class use_stream:
    """Context manager: enqueue this thread's kernels on a caller-owned stream
    (e.g. ``torch.cuda.current_stream().cuda_stream``)."""

    def __init__(self, stream):
        self.stream = stream

    def __enter__(self):
        self.previous = current_stream()
        _stream.value = self.stream
        return self

    def __exit__(self, *exc):
        _stream.value = self.previous
        return False


def synchronize():
    check(lib().gm_stream_sync(current_stream()))


def launch_count():
    return int(load_library().gm_launch_count())


def _free_device(ptr, stream):
    # stream-ordered free on the stream the block was allocated (and used) on
    if _lib is not None and ptr:
        _lib.gm_free(ptr, stream)


def _free_pinned(ptr):
    if _lib is not None and ptr:
        _lib.gm_host_free(ptr)


class DeviceArray:
    """A C-contiguous array resident in HBM (what flows between blocks while a
    graph is being computed).  ``np.asarray(x)`` / ``x.to_host()`` copy it back."""

    __array_priority__ = 100

    def __init__(self, shape, dtype, ptr=None, owner=None):
        self.shape = tuple(int(s) for s in shape)
        self.dtype = np.dtype(dtype)
        self.size = int(np.prod(self.shape, dtype=np.int64)) if self.shape else 1
        self.nbytes = self.size * self.dtype.itemsize
        self._owner = owner  # keeps foreign memory (e.g. a torch tensor) alive
        if ptr is None:
            p = ctypes.c_void_p()
            stream = current_stream()
            check(lib().gm_malloc(ctypes.byref(p), self.nbytes, stream))
            self.ptr = p.value
            self._finalizer = weakref.finalize(self, _free_device, self.ptr, stream)
        else:
            self.ptr = int(ptr)
            self._finalizer = None

    @property
    def ndim(self):
        return len(self.shape)

    @classmethod
    def from_host(cls, array):
        array = np.ascontiguousarray(array)
        out = cls(array.shape, array.dtype)
        check(lib().gm_memcpy_h2d(out.ptr, array.ctypes.data, array.nbytes, current_stream()))
        # pageable copies are staged synchronously by the driver; pinned ones are
        # asynchronous, so keep the source alive until the stream is drained
        out._owner = array
        return out

    def to_host(self):
        out = pinned_empty(self.shape, self.dtype)
        check(lib().gm_memcpy_d2h(out.ctypes.data, self.ptr, self.nbytes, current_stream()))
        return out

    def __array__(self, dtype=None, copy=None):
        host = self.to_host()
        return host if dtype is None else host.astype(dtype)

    def reshape(self, *shape):
        if len(shape) == 1 and isinstance(shape[0], (tuple, list)):
            shape = tuple(shape[0])
        view = DeviceArray(shape, self.dtype, ptr=self.ptr, owner=self)
        if view.size != self.size:
            raise ValueError("cannot reshape device array of size {} into {}".format(self.size, shape))
        return view

    def __repr__(self):
        return "DeviceArray(shape={}, dtype={})".format(self.shape, self.dtype)


STATS = {"pinned_allocations": 0}
_pinned_free = {}          # nbytes -> [ptr, ...] page-locked blocks ready for reuse
_pinned_cached_bytes = 0
PINNED_CACHE_LIMIT = int(os.environ.get("GM_PINNED_CACHE_BYTES", 8 << 30))


def _recycle_pinned(ptr, nbytes):
    """Finalizer of a pinned result array: keep the block for the next result of
    the same size (cudaHostAlloc costs ~0.1 s/GB), free it beyond the cache limit."""
    global _pinned_cached_bytes
    if _lib is None or not ptr:
        return
    with _lib_lock:
        if _pinned_cached_bytes + nbytes <= PINNED_CACHE_LIMIT:
            _pinned_free.setdefault(nbytes, []).append(ptr)
            _pinned_cached_bytes += nbytes
            return
    _lib.gm_host_free(ptr)


def pinned_empty(shape, dtype):
    """numpy array backed by page-locked host memory (recycled with the array)."""
    global _pinned_cached_bytes
    dtype = np.dtype(dtype)
    shape = tuple(int(s) for s in shape)
    nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
    if nbytes == 0:
        return np.empty(shape, dtype)
    ptr = None
    with _lib_lock:
        blocks = _pinned_free.get(nbytes)
        if blocks:
            ptr = blocks.pop()
            _pinned_cached_bytes -= nbytes
    if ptr is None:
        p = ctypes.c_void_p()
        check(lib().gm_host_alloc(ctypes.byref(p), nbytes))
        ptr = p.value
        STATS["pinned_allocations"] += 1
    buf = (ctypes.c_uint8 * nbytes).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    weakref.finalize(buf, _recycle_pinned, ptr, nbytes)
    return arr


_registered = {}


def pin(array):
    """Page-lock a user array in place (idempotent) so uploads run at full PCIe speed."""
    if not isinstance(array, np.ndarray) or array.nbytes == 0 or not array.flags.c_contiguous:
        return False
    key = (array.ctypes.data, array.nbytes)
    if key in _registered:
        return True
    if lib().gm_host_register(array.ctypes.data, array.nbytes) != 0:
        return False  # e.g. memory already pinned by its allocator
    ref = weakref.ref(array, lambda _r, k=key: _unpin(k))
    _registered[key] = ref
    return True


def _unpin(key):
    if _registered.pop(key, None) is not None and _lib is not None:
        _lib.gm_host_unregister(key[0])


def is_device(x):
    return isinstance(x, DeviceArray)


def as_gm_array(x, shape3=None):
    """GmArray descriptor for a numpy array (host) or DeviceArray (device)."""
    desc = GmArray()
    if isinstance(x, DeviceArray):
        desc.data = x.ptr
        desc.space = GM_DEVICE
    else:
        if not (isinstance(x, np.ndarray) and x.flags.c_contiguous):
            raise ValueError("expected a C-contiguous numpy array")
        desc.data = x.ctypes.data
        desc.space = GM_HOST
    desc.dtype = dtype_code(x.dtype)
    shape = tuple(shape3) if shape3 is not None else tuple(x.shape)
    if len(shape) != 3:
        shape = (1,) * (3 - len(shape)) + shape if len(shape) < 3 else (int(np.prod(shape[:-2])),) + shape[-2:]
    desc.shape[0], desc.shape[1], desc.shape[2] = shape
    return desc


def scalar_ptr(value, dtype):
    """Pointer to one element of `dtype` holding `value` (kept alive by the caller)."""
    holder = np.array([value], dtype=dtype)
    return holder, holder.ctypes.data


def zonal_values(raster_desc, nodata_ptr, has_nodata, polys, geo, thresholds, counts):
    """Active cell values under every polygon (gm_zonal_values): (counts, packed values)."""
    counts = np.ascontiguousarray(counts, dtype=np.int64)
    values = np.empty(int(counts.sum()), dtype=_CODE_DTYPES[raster_desc.dtype])
    check(lib().gm_zonal_values(
        ctypes.byref(raster_desc), nodata_ptr, has_nodata, ctypes.byref(polys), geo,
        None if thresholds is None else thresholds.ctypes.data, counts.ctypes.data,
        values.ctypes.data if values.size else None or np.empty(1, values.dtype).ctypes.data,
        current_stream()))
    return counts, values


_ORDER_STATS = {"median": 5, "percentile": 8}


def segment_order_statistic(values, offsets, statistic, percentile=None):
    """float32 median / percentile of every segment values[offsets[k]:offsets[k+1]]."""
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    out = np.empty(n, dtype=np.float32)
    if n == 0:
        return out
    values = np.ascontiguousarray(values)
    check(lib().gm_segment_order_stat(
        values.ctypes.data if values.size else None, dtype_code(values.dtype), offsets.ctypes.data, n,
        _ORDER_STATS[statistic], float(percentile or 0.0), out.ctypes.data, current_stream()))
    return out


SMOOTH_MODES = {"exact": 0, "fma": 1, "float32": 2}


class smooth_arithmetic:
    """Context manager: arithmetic of Smooth's tap sums ('exact' = SciPy bit for bit, 'fma' =
    float64 with fused multiply-add (default), 'float32' = float32 accumulation); see
    gm_set_smooth_mode in include/geokernels.h."""

    def __init__(self, mode):
        self.mode = SMOOTH_MODES[mode]

    def __enter__(self):
        self.previous = lib().gm_get_smooth_mode()
        check(lib().gm_set_smooth_mode(self.mode))
        return self

    def __exit__(self, *exc):
        lib().gm_set_smooth_mode(self.previous)
        return False


_pipeline_streams = []


def pipeline_streams(n=3):
    """`n` extra CUDA streams (created once) for chunk pipelines."""
    while len(_pipeline_streams) < n:
        p = ctypes.c_void_p()
        check(lib().gm_stream_create(ctypes.byref(p)))
        _pipeline_streams.append(p.value)
    return _pipeline_streams[:n]


def stream_sync(stream):
    check(lib().gm_stream_sync(stream))


def free_polygons(handle):
    if _lib is not None and handle:
        _lib.gm_polygons_free(handle)
