"""bench.py's output contract on a GPU box: exactly ONE line on stdout, a JSON object with the keys the driver reads."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*flags):
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True, env=env,
                       timeout=600)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.split("\n") if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_one_json_line_with_the_contract_keys():
    # a reduced ensemble keeps the test short; the contract is the same as for the default run
    line = _run("--steps", "2", "--warmup", "3", "--members", "8192", "--no-cpu-baseline")
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 3
    assert line["dtype"] == "f64" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["gpu_launches"] > 0
    assert "workload" in line["config"] and "model" not in line["config"]
    e2e = line["e2e"]
    assert e2e["value"] > 0 and e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0
    assert e2e["value"] <= line["value"] * 1.02  # host buffers and copies inside the timed region: not faster than device-resident
    roof = line["roofline"]
    assert roof["bound"] == "fp64" and roof["unit"] == "TFLOP/s"
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-12 and 0.0 < roof["frac"] < 1.0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"])


def test_dump_outputs_repeat_across_runs_and_match_the_reference_arm(tmp_path):
    """--dump-outputs: float64 arrays of at most 64 MB in all; the seeded inputs make two runs with different step
    counts write identical outputs, and the members both arms computed are bit-identical to the reference arm's."""
    dirs = [tmp_path / n for n in ("a", "b", "ref")]
    line = _run("--steps", "1", "--warmup", "0", "--members", "4096", "--no-cpu-baseline", "--dump-outputs", str(dirs[0]))
    assert line["steps"] == 1
    _run("--steps", "3", "--warmup", "0", "--members", "4096", "--no-cpu-baseline", "--dump-outputs", str(dirs[1]))
    _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--members", "64", "--dump-outputs", str(dirs[2]))
    names = sorted(p.name for p in dirs[0].iterdir())
    assert names == sorted(p.name for p in dirs[2].iterdir())
    assert sum(p.stat().st_size for p in dirs[0].iterdir()) <= 64 << 20
    a, b, ref = ({p.stem: np.load(p) for p in d.iterdir()} for d in dirs)
    assert np.array_equal(a["members"], np.arange(4096)) and a["nu4_u"].shape == (4096, 50, 1)
    assert (a["nu4_status"] == 0).all()
    rows = ref["members"].astype(np.int64)
    assert len(rows) > 0
    for k in a:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k], equal_nan=True), k
        assert np.array_equal(a[k][rows], ref[k], equal_nan=True), k
