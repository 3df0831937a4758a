"""GPU: `bench.py --dump-outputs` writes what the last timed step computed.  The inputs are seeded and every step rebuilds
the grid from them, so two runs with a different number of timed steps must write the same arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--scale", "0.01",
                          "--no-e2e", "--no-cpu-baseline", "--no-full-path", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_are_the_timed_results_and_repeat(tmp_path):
    one, two = _bench(tmp_path / "one", 1), _bench(tmp_path / "two", 2)
    assert one["steps"] == 1 and two["steps"] == 2
    names = sorted(os.listdir(tmp_path / "one"))
    assert names == sorted(os.listdir(tmp_path / "two"))
    assert sum(os.path.getsize(tmp_path / "one" / n) for n in names) <= 64 << 20
    got = {}
    for n in names:
        a, b = np.load(tmp_path / "one" / n), np.load(tmp_path / "two" / n)
        assert a.dtype in (np.float32, np.float64) and a.dtype == b.dtype and a.shape == b.shape, n
        assert (a == b).all(), f"{n} differs between two runs of the same workload"
        got[n[:-4]] = a
    c = dict(zip(bench.DUMP_COUNTERS, got["counters"].astype(np.int64).tolist()))
    res = one["result"]
    assert c["n_points_inserted"] == res["n_points_inserted"] == one["config"]["points"]
    assert c["n_points_alive"] == res["n_points_alive"] and c["n_leaves"] == res["n_leaves"] and c["n_cells"] == res["n_cells"]
    assert got["pose_counts"].shape == (one["n_poses"], 3) and got["pose_counts"][:, 1].sum() == c["n_points_alive"]
    # a table is written whole when it is shorter than its sample, else as a sample of exactly DUMP_ROWS rows
    n_points = min(c["n_points_alive"], bench.DUMP_ROWS["point"])
    assert len(got["point_idx"]) == n_points and got["point_xyz"].shape == (n_points, 3) and np.isfinite(got["point_xyz"]).all()
    assert len(got["leaf_edge"]) == min(c["n_leaves"], bench.DUMP_ROWS["leaf"]) and (got["leaf_edge"] > 0).all()
    assert 0 < len(got["plane"]) == len(got["plane_size"]) <= bench.DUMP_ROWS["plane"]
    assert (got["plane_best_count"] <= got["plane_size"]).all()
