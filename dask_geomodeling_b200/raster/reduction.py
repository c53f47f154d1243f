"""Reductions over several aligned rasters, on the CUDA evaluator.

Drop-in for the reference's raster/reduction.py: ``reduce_rasters`` (:38-119) and the ``Max``
block (:215-231).  The reference stacks the rasters into an (n, t, y, x) float array with NaN for
'no data' and calls NumPy's nan-functions along the first axis; here the rasters are the inputs
of ONE evaluator program that keeps the running result of a pixel in a register (OVERLAY steps
with a reduction kind, include/gm_bytecode.h) -- one pass over the inputs, no stack.  Inside a
view the program is fused with the element-wise blocks around it (core/fusion.py).  Stacks the
evaluator cannot take (more than GM_MAX_INPUTS rasters) go to gm_reduce_stack, which runs the same
OVERLAY step over any number of rasters in one launch.

mean, var, std, argmin and argmax keep more than one value per pixel, which an OVERLAY step does
not: a stack of any length, also of one raster, goes to gm_reduce_stack_stat, one launch that
stacks the rasters in NumPy's working dtype (np.result_type(dtype, float16)) and reduces them as
np.nanmean / nanvar / nanstd / nanargmin / nanargmax do (var and std read the stack twice).

Statistics on the CUDA path: last, first, count, max, min, argmin, argmax (any dtype: exact in the
float dtype NumPy would use), sum, product, mean, var and std (float32 / float64 outputs:
sequential in the raster order, as NumPy's axis-0 reduction).  median and percentiles of a stack of
rasters raise NotImplementedError (TemporalAggregate offers them along the time axis).
"""
import numpy as np

from ..utils import Extent, parse_percentile_statistic
from .. import _native, _state
from . import _lowering, _program
from ._program import Node
from .base import RasterBlock
from .elemwise import BaseElementwise

__all__ = ["Max"]

STATISTICS = ("first", "last", "count", "sum", "mean", "min", "max", "argmin", "argmax", "std", "var",
              "median", "product")
ON_DEVICE = ("first", "last", "count", "sum", "min", "max", "product", "mean", "var", "std", "argmin",
             "argmax")


def check_statistic(statistic):
    if statistic not in STATISTICS:
        statistic, percentile = parse_percentile_statistic(statistic)
        if percentile is None:
            raise ValueError('Unknown statistic "{}"'.format(statistic))


def _lower_reduce(statistic):
    def lower(args):
        kwargs = args[0]
        children = [a for a in args[1:] if a is not None]
        return Node("reduce", children, statistic=statistic, dtype=kwargs["dtype"],
                    fillvalue=kwargs["fillvalue"])

    return lower


def statistic_name(statistic):
    """The name of ``statistic`` without a percentile ("p90" -> "percentile"); KeyError if unknown."""
    if statistic in STATISTICS:
        return statistic
    name, percentile = parse_percentile_statistic(statistic)
    if percentile is None:
        raise KeyError('Unknown statistic "{}"'.format(statistic))
    return name


def on_device(name):
    """``name`` (a statistic_name); NotImplementedError for a statistic the CUDA path lacks."""
    if name not in ON_DEVICE:
        raise NotImplementedError(
            "reduce_rasters: statistic '{}' is not part of the CUDA raster path "
            "(available: {})".format(name, ", ".join(ON_DEVICE)))
    return name


def device_statistic(statistic):
    """``statistic`` as the CUDA stack reductions name it; raises for those they do not offer."""
    return on_device(statistic_name(statistic))


def reduce_rasters(stack, statistic, no_data_value=None, dtype=None):
    """Apply ``statistic`` pixel by pixel to a list of raster payloads (dicts with "values" and
    "no_data_value"), skipping 'no data'.  Output dtype and no data value default to those of
    the first raster; sums and counts hold 0 where every input is 'no data'."""
    statistic = statistic_name(statistic)
    if len(stack) == 0:
        raise ValueError("Cannot reduce a zero-length stack")
    on_device(statistic)
    shape = tuple(stack[0]["values"].shape)
    if any(tuple(d["values"].shape) != shape for d in stack[1:]):
        raise ValueError("all rasters of the stack must have the same shape")
    if dtype is None:
        dtype = stack[0]["values"].dtype
    if no_data_value is None:
        no_data_value = stack[0]["no_data_value"]
    payloads = [(d["values"], d.get("no_data_value")) for d in stack]
    if statistic in _program.STACK_STATS:
        values = _program.run_stack_stat(statistic, payloads, np.dtype(dtype), no_data_value,
                                         _state.keep_on_device())
        return {"values": values, "no_data_value": no_data_value}
    kwargs = {"dtype": np.dtype(dtype).name, "fillvalue": no_data_value}
    if len(stack) <= _native.GM_MAX_INPUTS:
        try:
            result = _lowering.run_single(lambda ops: _lower_reduce(statistic)([kwargs] + ops), list(stack))
            result["no_data_value"] = no_data_value
            return result
        except _program.FusionLimit:
            pass    # the stack kernel below takes any length
    values = _program.run_stack(statistic, payloads, np.dtype(dtype), no_data_value, _state.keep_on_device())
    return {"values": values, "no_data_value": no_data_value}


def wrap_reduction_function(statistic):
    lower = _lower_reduce(statistic)

    def reduction_function(process_kwargs, *args):
        stack = []
        for arg in args:
            if arg is None:
                continue
            if "time" in arg or "meta" in arg:
                return arg      # time / meta requests are answered by the first source
            stack.append(arg)
        if not stack:
            return None
        return reduce_rasters(stack, statistic, process_kwargs["fillvalue"], process_kwargs["dtype"])

    reduction_function.__name__ = "reduce_{}_process".format(statistic)
    reduction_function._gm_lower = lower
    reduction_function._gm_skip_none = True
    return reduction_function


class BaseReduction(BaseElementwise):
    """Reduction of two or more rasters; stricter than BaseElementwise: without a common
    period there is no data (reference: raster/reduction.py:122-186)."""

    def __init__(self, *args):
        for arg in args:
            if not isinstance(arg, RasterBlock):
                raise TypeError("'{}' object is not allowed".format(type(arg)))
        super().__init__(*args)

    def get_sources_and_requests(self, **request):
        process_kwargs = {"dtype": self.dtype.name, "fillvalue": self.fillvalue}
        period = self.period
        if period is None:
            return [(process_kwargs, None)]
        # limit the request to the common period so that the sources answer aligned frames
        start, stop = request.get("start"), request.get("stop")
        if start is None:
            request["start"] = period[1]
        elif stop is None:
            request["start"] = min(max(start, period[0]), period[1])
        else:
            request["start"], request["stop"] = max(start, period[0]), min(stop, period[1])
        return [(process_kwargs, None)] + [(source, request) for source in self.args]

    @property
    def extent(self):
        extents = [e for e in (x.extent for x in self.args) if e is not None]
        if not extents:
            return None
        return (min(e[0] for e in extents), min(e[1] for e in extents),
                max(e[2] for e in extents), max(e[3] for e in extents))

    @property
    def geometry(self):
        geometries = [g for g in (x.geometry for x in self.args) if g is not None]
        if not geometries:
            return None
        boxes = [Extent.from_geometry(g).bbox for g in geometries]
        projection = getattr(geometries[0], "projection", None)
        union = (min(b[0] for b in boxes), min(b[1] for b in boxes),
                 max(b[2] for b in boxes), max(b[3] for b in boxes))
        return Extent(union, projection).as_geometry()


class Max(BaseReduction):
    """Maximum of two or more rasters, ignoring 'no data'
    (reference: raster/reduction.py:215-231)."""

    process = staticmethod(wrap_reduction_function("max"))

    @property
    def dtype(self):
        return np.result_type(*self.args)   # not widened to >= 32 bit, unlike the math blocks
