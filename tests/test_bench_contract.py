"""bench.py's reference arm runs on the CPU alone: its JSON line is checked here against the
contract (one line on stdout; metric / unit / config of the GPU arm; `impl`, `cpu_baseline`,
`e2e` with zero copy bytes), on a small raster so that the CPU suite stays short.  The GPU arm's
--steps and --dump-outputs are checked on small legs."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, RANK="0")
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "2048",
         "--steps", "2", "--warmup", "1", "--legs", "chain"],
        cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["higher_is_better"] is True
    assert line["unit"] == "Gpixel/s" and line["value"] > 0 and line["steps"] == 2 and line["warmup"] == 1
    assert line["ms_per_step"] > 0 and abs(line["value"] - 2048 * 2048 / line["ms_per_step"] / 1e6) < 1e-6 * line["value"] + 1e-9
    assert line["config"]["same_config"] is True and "cfg2" in line["config"]["workload"]
    base = line["cpu_baseline"]
    assert base["kind"] in ("stub harness", "port") and base["cores"] >= 1 and base["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["vs_baseline"] is None


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--size", "2048"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_dumps_the_outputs_of_its_timed_calls(tmp_path):
    """Every leg at a small size: --steps timed launches of the chain, one float32 / float64 file
    per timed call, and the chain's file equal to the oracle at the same sampled cells."""
    import torch

    import bench
    from dask_geomodeling_b200 import workloads
    from oracle import workloads as oracle_workloads

    size = 1024
    env = dict(os.environ, RANK="0", LOCAL_RANK="0", WORLD_SIZE="1")
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--size", str(size),
         "--e2e-steps", "1", "--leg-steps", "2", "--dem-size", "1024", "--zonal-size", "2048", "--zonal-grid", "16",
         "--temporal-frames", "70", "--temporal-size", "256", "--dump-outputs", str(tmp_path)],
        cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout)
    assert line["steps"] == 3 and line["gpu_launches"] == 3
    dumps = {name[:-4]: np.load(str(tmp_path / name)) for name in os.listdir(str(tmp_path))}
    assert set(dumps) == {
        "chain", "stencils_smooth", "stencils_movingmax", "stencils_hillshade", "zonal_mean", "zonal_max",
        "zonal_p90", "zonal_e2e_mean", "zonal_e2e_p90", "temporal_sum", "temporal_max", "temporal_mean_64frames",
        "temporal_std_64frames", "temporal_median_64frames", "temporal_cumulative_sum_64frames",
        "temporal_sum_int16", "temporal_max_int16"}
    assert all(a.dtype in (np.float32, np.float64) and a.size for a in dumps.values())
    assert sum(a.nbytes for a in dumps.values()) <= bench.DUMP_BYTES
    ints, floats = workloads.cfg2_arrays(size, seed=43)
    (isdata, _), _ = oracle_workloads.cfg2(ints, floats, workloads.CFG2_PAIRS)
    expected = bench.output_sample(torch, isdata, zlib.crc32(b"chain"))
    assert dumps["chain"].shape == (bench.DUMP_CELLS,) and np.array_equal(dumps["chain"], expected)
