"""CPU: the benchmark's reference arm (`bench.py --impl reference`: the unmodified reference package from oracle/_ref on
the host cores, or the oracle port where that copy is absent) runs without a GPU and prints ONE JSON line with the keys the
driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


import pytest


@pytest.mark.parametrize("no_ref", ["0", "1"])
def test_reference_arm_json_line(no_ref):
    have_ref = no_ref == "0" and os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "octreelib"))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample", "120000"], capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, OL_NO_REFERENCE=no_ref))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("points/sec") and d["value"] > 0 and d["n_gpus"] == 1
    assert d["config"]["workload"] == "c4_street_100M"
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if have_ref else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "points" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _stub_grid(n_leaves, n_blocks, n_points):
    """the calls `bench.dump_outputs` makes on a grid, answered from seeded random tables"""
    from types import SimpleNamespace

    import numpy as np

    import bench

    rng = np.random.default_rng(5)
    leaves = dict(corner=rng.random((n_leaves, 3)), edge=rng.random(n_leaves), cell=rng.integers(0, 99, n_leaves, dtype=np.int32),
                  depth=rng.integers(0, 4, n_leaves, dtype=np.int32), parent_epoch=np.zeros(n_leaves, dtype=np.int32))
    planes = dict(plane=np.column_stack([np.arange(n_blocks), rng.random((n_blocks, 3))]).astype(np.float32),  # x = row number
                  **{k: rng.integers(0, 1000, n_blocks, dtype=np.int32) for k in ("pose", "leaf", "size", "best", "best_count")})
    points = dict(xyz=rng.random((n_points, 3)), idx=np.arange(n_points, dtype=np.int64), cell=np.zeros(n_points, dtype=np.int32))
    stats = {k: i + 1 for i, k in enumerate(bench.DUMP_COUNTERS)}
    forest = SimpleNamespace(stats=lambda light=False: stats, export_leaves=lambda: leaves,
                             export_ransac=lambda scored_only=False: planes,
                             export_points=lambda pose_index=-1, order=0: points)
    counts = rng.integers(0, 1000, (7, 3))
    return SimpleNamespace(_host=SimpleNamespace(forest=forest, counts=lambda: counts)), leaves, planes, points


def test_dump_outputs_is_a_fixed_float_sample_under_64_mb(tmp_path):
    import numpy as np

    import bench

    rows = bench.DUMP_ROWS
    grid, leaves, planes, points = _stub_grid(1000, rows["plane"] + 999, rows["point"] + 999)
    bench.dump_outputs(grid, str(tmp_path / "a"))
    bench.dump_outputs(grid, str(tmp_path / "b"))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert {"counters.npy", "pose_counts.npy", "leaf_corner.npy", "plane.npy", "plane_best_count.npy", "point_xyz.npy"} <= set(names)
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    got = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and a.dtype == b.dtype and (a == b).all(), n
        got[n[:-4]] = a
    assert got["counters"].tolist() == list(range(1, len(bench.DUMP_COUNTERS) + 1))
    # a table shorter than its sample is written whole, longer ones as a sorted sample of their rows
    assert (got["leaf_corner"] == leaves["corner"]).all() and (got["leaf_depth"] == leaves["depth"]).all()
    assert got["plane"].shape == (rows["plane"], 4) and len(got["point_idx"]) == rows["point"]
    sel = got["point_idx"].astype(np.int64)  # the stub's point index is the row number
    assert (np.diff(sel) > 0).all() and (got["point_xyz"] == points["xyz"][sel]).all()
    sel = got["plane"][:, 0].astype(np.int64)
    assert (np.diff(sel) > 0).all() and (got["plane"] == planes["plane"][sel]).all() and (got["plane_size"] == planes["size"][sel]).all()


def test_dump_outputs_is_refused_where_it_has_no_single_timed_grid():
    for extra, env in ((["--impl", "reference"], {}), (["--gpus", "2"], {"WORLD_SIZE": "2"})):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", "unused", *extra], capture_output=True,
                             text=True, timeout=120, cwd=ROOT, env=dict(os.environ, **env))
        assert out.returncode == 2 and "--dump-outputs" in out.stderr and not os.path.exists(os.path.join(ROOT, "unused"))
