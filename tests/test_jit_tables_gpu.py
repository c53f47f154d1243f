"""Lookup-table placements and the IsData fold of the specialiser, bit for bit against the
interpreter and the oracle.  Small dense ND_ONLY Reclassify tables (n <= 64) become two 32-bit
literal words, larger ones stay in shared memory; an IsData / IsNoData right after a Step is folded
into it in baked kernels.  Every case runs the interpreter, the unbaked specialised kernel and the
baked one (the same constants twice on >= 2^22 pixels) on a raster whose pixel count is not a
multiple of the group width or of a chunk."""
import numpy as np
import pytest

from dask_geomodeling_b200 import _native
from dask_geomodeling_b200.raster import _program
from dask_geomodeling_b200.raster._program import Leaf, Node
from oracle import raster as R

pytestmark = pytest.mark.gpu

SHAPE = (1, 2049, 2053)          # 4 206 597 pixels: >= 2^22 (baked), odd
F32_MAX = float(np.finfo("f4").max)


def backends(monkeypatch, node, leaves):
    """The outputs of the interpreter, the unbaked and the baked specialised kernel."""
    lib = _native.lib()
    previous = lib.gm_get_eval_mode()
    got = []
    try:
        lib.gm_set_eval_mode(1)
        got.append(_program.evaluate([node], leaves)[0][0])
        lib.gm_set_eval_mode(2)
        monkeypatch.setenv("GM_JIT_NO_BAKE", "1")
        got.append(_program.evaluate([node], leaves)[0][0])
        monkeypatch.delenv("GM_JIT_NO_BAKE")
        _program.evaluate([node], leaves)
        got.append(_program.evaluate([node], leaves)[0][0])
    finally:
        lib.gm_set_eval_mode(previous)
    return [np.asarray(g) for g in got]


def check(monkeypatch, node, leaves, expected):
    for name, got in zip(("interpreter", "unbaked", "baked"), backends(monkeypatch, node, leaves)):
        assert got.dtype == expected.dtype, name
        np.testing.assert_array_equal(got, expected, err_msg=name)


def keys_raster(dtype, base, n, nodata, seed):
    """Keys of `dtype` around [base, base + n): inside, at base - 1 and base + n, far outside, and
    the no-data value."""
    rng = np.random.default_rng(seed)
    info = np.iinfo(dtype)
    near = rng.integers(base - 3, base + n + 3, SHAPE)
    far = rng.integers(info.min, int(info.max) + 1, SHAPE)
    values = np.where(rng.random(SHAPE) < 0.8, near, far)
    values = np.clip(values, info.min, info.max).astype(dtype)
    values[rng.random(SHAPE) < 0.05] = nodata
    return values


# (source dtype, base, n, no-data value): n around the 32 / 64 boundaries of the bit tables,
# base != 0, negative keys, the no-data key inside and outside the table range
TABLES = [
    ("int16", 0, 1, 32767),
    ("int16", 5, 31, 32767),
    ("int8", -20, 32, -128),
    ("uint8", 3, 33, 255),
    ("int32", -40, 63, 2147483647),
    ("int16", -70, 64, -40),        # no data inside the table range
    ("int32", 1000, 65, 2147483647),
    ("uint8", 0, 200, 255),
    ("int16", -100, 200, -30),      # larger table, no data inside it
]


@pytest.mark.parametrize("select", [True, False])
@pytest.mark.parametrize("dtype,base,n,nodata", TABLES)
@pytest.mark.parametrize("op", ["isdata", "isnodata"])
def test_dense_reclassify_tables(monkeypatch, dtype, base, n, nodata, select, op):
    rng = np.random.default_rng(n * 7 + base)
    # the first and the last key span the table; the keys between them leave gaps (found = 0)
    keys = [k for k in range(base, base + n) if k in (base, base + n - 1) or rng.random() < 0.6]
    # outside every source dtype: an unmapped key kept by select=False never equals it (the lowering
    # counts a kept key as data even when it equals the fill value, the oracle does not)
    fill = 1 << 40
    # some keys map onto the fill value (no data after Reclassify)
    pairs = [(k, fill if rng.random() < 0.2 else int(rng.integers(0, 5))) for k in keys]
    values = keys_raster(dtype, base, n, nodata, seed=n)
    node = Node(op, [Node("reclassify", [Leaf(0)], dtype="int64", fillvalue=fill, data=pairs, select=select)])
    mapped = R.reclassify(values, nodata, pairs, select, np.dtype("int64"), fill)
    expected = (R.is_data if op == "isdata" else R.is_nodata)(*mapped)[0]
    check(monkeypatch, node, [(values, nodata)], expected)


def floats(seed, specials):
    rng = np.random.default_rng(seed)
    values = rng.uniform(-10, 10, SHAPE).astype("f4")
    values[rng.random(SHAPE) < 0.1] = 0.5          # == location
    pick = rng.random(SHAPE)
    for i, v in enumerate(specials):
        values[(pick >= 0.02 * i) & (pick < 0.02 * (i + 1))] = v
    return values


SPECIALS = [F32_MAX, np.nan, np.inf, -np.inf]


@pytest.mark.parametrize("op", ["isdata", "isnodata"])
@pytest.mark.parametrize("left,at,right", [(0.0, 0.5, 1.0), (F32_MAX, 0.5, 1.0), (0.0, F32_MAX, F32_MAX),
                                           (np.nan, 2.0, np.inf)])
def test_is_data_over_step(monkeypatch, op, left, at, right):
    values = floats(1, SPECIALS)
    node = Node(op, [Node("step", [Leaf(0)], left=left, right=right, value=0.5, at=at)])
    stepped = R.step(values, F32_MAX, left, right, 0.5, at)
    expected = (R.is_data if op == "isdata" else R.is_nodata)(*stepped)[0]
    check(monkeypatch, node, [(values, F32_MAX)], expected)


def test_is_data_over_cfg2_shaped_chain(monkeypatch):
    """Reclassify (bit table) -> Clip -> Step -> IsData, the chain bench.py times."""
    ints = keys_raster("int16", 0, 49, 32767, seed=3)
    values = floats(4, SPECIALS)
    pairs = [(k, int(k % 3)) for k in range(0, 49, 2)]
    r = Node("reclassify", [Leaf(0)], dtype="int64", fillvalue=np.iinfo("i8").max, data=pairs, select=True)
    node = Node("isdata", [Node("step", [Node("clip", [Leaf(1), r])], left=0, right=1, value=0.5, at=F32_MAX)])
    mask = R.reclassify(ints, 32767, pairs, True, np.dtype("int64"), np.iinfo("i8").max)
    clipped = R.clip(values, F32_MAX, *mask)
    expected = R.is_data(*R.step(*clipped, 0, 1, 0.5, F32_MAX))[0]
    check(monkeypatch, node, [(ints, 32767), (values, F32_MAX)], expected)


@pytest.mark.parametrize("op", ["isdata", "isnodata"])
@pytest.mark.parametrize("producer", ["clip", "mask", "mask_fill", "maskbelow"])
def test_is_data_over_other_producers(monkeypatch, op, producer):
    values = floats(5, SPECIALS)
    other = floats(6, [F32_MAX])
    if producer == "clip":
        inner = Node("clip", [Leaf(0), Leaf(1)])
        produced = R.clip(values, F32_MAX, other, F32_MAX)
        leaves = [(values, F32_MAX), (other, F32_MAX)]
    elif producer in ("mask", "mask_fill"):
        value = 0 if producer == "mask_fill" else 3.0      # Mask(0) fills with 1: the value of data
        inner = Node("mask", [Leaf(0)], value=value)
        produced = R.mask(values, F32_MAX, value)
        leaves = [(values, F32_MAX)]
    else:
        inner = Node("maskbelow", [Leaf(0)], value=-1.0)
        produced = R.mask_below(values, F32_MAX, -1.0)
        leaves = [(values, F32_MAX)]
    expected = (R.is_data if op == "isdata" else R.is_nodata)(*produced)[0]
    check(monkeypatch, Node(op, [inner]), leaves, expected)
