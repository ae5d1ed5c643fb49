"""bench.py --dump-outputs: the outputs of the last timed step of the headline leg (65,536 scenarios, so a sample of them),
float64 and under 64 MB, identical from run to run with the same arguments; --steps sets how many steps were timed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--gpus", "1", "--warmup", "5", "--quick", "--no-e2e", "--no-cpu-baseline"]
PER_SCENARIO = ("x", "xbar", "e", "status", "cost", "v", "iters", "xbar_traj", "tube")


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--steps", str(steps), "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    files = sorted(os.listdir(out_dir))
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in files) <= 64e6
    arrays = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}
    assert set(arrays) == set(PER_SCENARIO) | {"scenario", "stats"}
    assert all(a.dtype == np.float64 for a in arrays.values())
    return line, arrays


def test_dump_is_reproducible_and_follows_steps(cuda_lib, tmp_path):
    line, a = _bench(tmp_path / "a", 4)
    _, b = _bench(tmp_path / "b", 4)
    line5, c = _bench(tmp_path / "c", 5)
    assert line["steps"] == 4 and line5["steps"] == 5 and line["gpu_launches"] < line5["gpu_launches"]
    S = line["config"]["scenarios_total"]
    idx = a["scenario"]
    assert 0 < len(idx) < S and np.all(np.diff(idx) > 0) and idx[-1] < S          # a sample of the scenarios, sorted
    n = 5
    assert a["x"].shape == (n, len(idx)) and a["status"].shape == (1, len(idx)) and a["tube"].shape[1] == len(idx)
    assert np.all(a["status"] == 0)
    for k in PER_SCENARIO + ("scenario",):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    np.testing.assert_allclose(a["stats"], b["stats"], rtol=1e-10)            # atomic sums: equal up to summation order
    assert a["stats"][7] == S                                                 # one count per scenario of the step
    np.testing.assert_array_equal(c["scenario"], idx)
    assert not np.array_equal(a["x"], c["x"])                                 # one more step timed, a different state
