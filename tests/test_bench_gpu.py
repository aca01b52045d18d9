"""``bench.py --dump-outputs``: the last timed step's outputs as float32 .npy files, the same for the same
arguments, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENVS = 65536        # more than bench.DUMP_ROWS: the per-env arrays are a sample


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "2",
           "--envs-per-gpu", str(ENVS), "--quick", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["config"]["envs_per_gpu"] == ENVS
    return {f[:-len(".npy")]: np.load(out / f) for f in sorted(os.listdir(out))}


def test_bench_dump_outputs_are_reproducible(tmp_path):
    import bench
    a = _bench(tmp_path / "a", 3)
    b = _bench(tmp_path / "b", 3)
    rows = bench.DUMP_ROWS
    assert {"env_ids", "obs", "rew", "reset", "time_outs", "episode_terrain_levels"} <= set(a)
    assert a["obs"].shape == (rows, 259) and a["rew"].shape == (rows,)
    ids = a["env_ids"]
    assert ids.dtype == np.float64 and len(np.unique(ids)) == rows and 0 <= ids.min() and ids.max() < ENVS
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.isfinite(a["obs"]).all() and 0 < a["reset"].sum() < rows
    assert set(a) == set(b)
    for k, v in a.items():
        assert v.dtype in (np.float32, np.float64), k
        np.testing.assert_allclose(v, b[k], rtol=1e-6, atol=1e-7, err_msg=k)
