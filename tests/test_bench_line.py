"""bench.py's host-side logic without a GPU (tests/bench_mock.py stands in for the device, the library and
torch.distributed): the JSON line carries the contract's keys and the per-job row accounting of both scaling modes."""
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def run(world, scaling, *bench_args):
    out = subprocess.run([sys.executable, os.path.join(HERE, "bench_mock.py"), str(world), scaling, *bench_args], capture_output=True,
                         text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


@pytest.mark.parametrize("world,scaling", [(1, "weak"), (2, "weak"), (2, "strong")])
def test_bench_line(world, scaling):
    d = run(world, scaling)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "gpu_launches", "clocks", "roofline", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == world and d["scaling"] == scaling and d["dtype"] == "f64"
    rows = 1_000_001
    job = rows * world if scaling == "weak" else rows
    assert d["config"]["total_rows"] == job
    assert abs(d["value"] - job * d["steps"] / (d["ms_per_step"] * d["steps"] / 1e3)) < 1e-3 * d["value"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"], k
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    if world > 1 and scaling == "weak":   # the e2e legs stream rows/N rows per rank: one table across the job
        assert e["rows_per_step"] <= rows + world * 200_000
    elif world == 1:
        assert e["rows_per_step"] == job
    else:   # (the stand-in all-reduce multiplies rank 0's count, whose shard may hold one batch more than the others)
        assert abs(e["rows_per_step"] - job) <= world * 200_000


@pytest.mark.parametrize("world", [1, 2])
def test_bench_dumps_the_last_timed_step(world, tmp_path):
    """--dump-outputs writes the final rows of Q1 (2 string keys, 8 aggregates) and of Q6 (1 aggregate) as float64 arrays;
    --steps is the number of timed steps."""
    import numpy as np
    d = run(world, "strong", "--steps", "7", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 7
    assert sorted(os.listdir(tmp_path)) == ["q1_keys.npy", "q1_values.npy", "q6_values.npy"]
    keys, values, q6 = (np.load(tmp_path / f) for f in ("q1_keys.npy", "q1_values.npy", "q6_values.npy"))
    assert keys.dtype == values.dtype == q6.dtype == np.float64
    assert keys.shape == (1, 2, 1) and (keys == ord("N")).all()
    assert values.shape == (1, 8) and (values == 1.0).all()
    assert q6.shape == (1, 1)
