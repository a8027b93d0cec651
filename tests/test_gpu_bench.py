"""bench.py end to end on the device at smoke size: `--steps` sets the timed steps and `--dump-outputs` writes the result tables
of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("workload,tables,rows", [
    ("tiny", ["measures_of_counts", "measures_of_centralTendency", "measures_of_cardinality", "measures_of_dispersion",
              "measures_of_percentiles", "measures_of_shape"], 200_000),
    ("tiny_stream", ["drift_statistics", "source.measures_of_counts", "source.measures_of_shape", "target.measures_of_counts",
                     "target.measures_of_shape"], 300_000),
    ("c1", ["measures_of_centralTendency"], None)], ids=["tiny", "tiny_stream", "c1"])
def test_bench_steps_and_dumped_outputs(tmp_path, workload, tables, rows):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                        "--workload", workload, "--no-extras", "--dump-outputs", str(out)],
                       cwd=str(tmp_path), env=dict(os.environ, ANV_BENCH_CLOCK_PERIOD_MS="0"), capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1, r.stdout[-2000:]
    line = json.loads(lines[0])
    assert line["steps"] == 3 and line["ms_per_step"] > 0
    if workload == "tiny":
        assert len(line["config"]["wall_ms_each_step_rank0"]) == 3
    files = {p.name: np.load(p) for p in out.iterdir()}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in files.values()), \
        [n for n, a in files.items() if not np.isfinite(a).all()]
    assert sum(a.nbytes for a in files.values()) <= 64 << 20
    for t in tables:
        assert files[t + ".attribute.crc32.npy"].size > 0, t
    if rows is not None:
        counts = tables[0] if workload == "tiny" else "source.measures_of_counts"
        assert np.all(files[counts + ".fill_count.npy"] + files[counts + ".missing_count.npy"] == rows)
    else:
        assert files["measures_of_centralTendency.attribute.crc32.npy"].size == 17       # every column of the income dataset
