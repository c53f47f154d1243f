"""Load placement and register footprint of the specialised kernel, without a GPU (SASS through
tools/jit_sass.py).  In the two-set hot loop of the cfg2 chain, baked and unbaked, the loads of chunk
c + 1 are issued before chunk c is evaluated, and nothing spills: a change of the generator, the
prelude or the compiler that lets ptxas sink those loads into the evaluation again (what the bench
chain lost time to) fails here.  Programs with more input per chunk keep the single-set loop and do
not spill either."""
import importlib.util
import os
import shutil

import numpy as np
import pytest

from dask_geomodeling_b200 import workloads
from dask_geomodeling_b200.raster._program import Leaf, Node

from test_jit_cpu import nvrtc_available

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def tools_available():
    return nvrtc_available() and bool(shutil.which("cuobjdump") or
                                      os.path.exists(os.path.join(CUDA, "bin", "cuobjdump")))


def jit_sass():
    spec = importlib.util.spec_from_file_location("jit_sass", os.path.join(ROOT, "tools", "jit_sass.py"))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


def cfg2():
    r = Node("reclassify", [Leaf(0)], dtype="int64", fillvalue=np.iinfo("i8").max,
             data=workloads.CFG2_PAIRS, select=True)
    st = Node("step", [Node("clip", [Leaf(1), r])], left=0, right=1, value=50.0, at=0.5)
    return Node("isdata", [st]), [(np.dtype("i2"), 32767), (np.dtype("f4"), workloads.F32_MAX)]


@pytest.mark.skipif(not tools_available(), reason="no NVRTC / cuobjdump in this environment")
@pytest.mark.parametrize("baked", [False, True], ids=["unbaked", "baked"])
def test_cfg2_loads_the_next_chunk_before_evaluating(baked):
    tool = jit_sass()
    sources = tool.generate(*cfg2())
    a = tool.analyse(sources[1] if baked else sources[0])
    assert a["spills"] == 0, a["log"]
    assert a["two_sets"] and len(a["halves"]) == 2
    for half in a["halves"]:
        # int16 + float32 at V = 4, U = 4: one 64-bit and one 128-bit load per group
        assert len(half["ldg"]) == 8, half
        assert max(half["ldg"]) < half["first_compare"], half


@pytest.mark.skipif(not tools_available(), reason="no NVRTC / cuobjdump in this environment")
@pytest.mark.parametrize("shape", ["cfg1", "add4_f4", "add8_f4"])
@pytest.mark.parametrize("baked", [False, True], ids=["unbaked", "baked"])
def test_wider_programs_keep_one_register_set_and_do_not_spill(shape, baked):
    tool = jit_sass()
    sources = tool.generate(*tool.shapes()[shape])
    a = tool.analyse(sources[1] if baked else sources[0])
    assert not a["two_sets"]
    assert a["spills"] == 0, a["log"]
