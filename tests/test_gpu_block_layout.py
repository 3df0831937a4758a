"""The sort-free RANSAC batch layout (leaf spans from the run index of the block build, work list written by the ranking)
and the block of every position derived on demand must give what the sorted layout gives (OL_RANSAC_SORTED_LAYOUT=1, in
a subprocess) on the shapes where they are easiest to get wrong.  Run as a script, this file prints the digest of one
case."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

K = 6


def _blob(rng, n, lo, hi):
    return rng.uniform(lo, hi, size=(n, 3))


def _clouds(case):
    """(pose numbers in insertion order, clouds, MaxPoints of the subdivide)"""
    from octreelib_b200.synthetic import lidar64_scan

    rng = np.random.default_rng(17)
    if case == "one_block":  # one pose: every leaf holds exactly one block
        return [0], [lidar64_scan(0, seed=5)], 40
    if case == "straddle":  # 27 unsplit leaves of 300 blocks each: leaves cross 2048-position tiles and 4096-slot chunks
        return list(range(300)), [_blob(rng, 120, 0.0, 3.0) for _ in range(300)], 10**6
    if case == "all_small":  # about one point per (pose, cell): no block reaches K points, the work list is empty
        return list(range(3)), [_blob(rng, 2000, 0.0, 100.0) for _ in range(3)], 100
    if case == "ranks":  # poses inserted out of order: pose index != pose rank
        order = [4, 1, 6, 0, 3, 5, 2]
        return order, [lidar64_scan(p, seed=9, n_points=40000) for p in order], 60
    raise KeyError(case)


def digest(case):
    from octreelib_b200.criteria import MaxPoints, MinPoints
    from octreelib_b200.grid import Grid, GridConfig
    from octreelib_b200.ransac import CudaRansac

    numbers, clouds, max_points = _clouds(case)
    grid = Grid(GridConfig(voxel_edge_length=1.0))
    for p, c in zip(numbers, clouds):
        grid.insert_points(p, c)
    grid.subdivide([MaxPoints(max_points)])
    host = grid._host
    forest = host.forest
    pose_rank = [int(x) for x in host.pose_numbers]
    h = hashlib.sha256()

    def add(*arrays):
        for a in arrays:
            h.update(np.ascontiguousarray(a).tobytes())

    np.random.seed(5)
    table = CudaRansac(threshold=0.02, hypotheses_number=256, initial_points_number=K).random_hypotheses
    forest.ransac(table, 0.02, pose_rank, 3, apply=False)
    res = forest.export_ransac()
    add(*(res[k] for k in ("pose", "leaf", "size", "plane", "best", "best_count")))
    scored = forest.export_ransac(scored_only=True)
    if case == "all_small":
        assert len(scored["pose"]) == 0
    else:
        assert len(scored["pose"]) > 0
    pts = forest.export_points(-1, order=1, want_mask=True)  # block of every position, same block table as the fit
    add(pts["idx"], pts["xyz"])
    np.random.seed(7)
    grid.map_leaf_points_cuda_ransac(poses_per_batch=2, threshold=0.02, hypotheses_number=256, initial_points_number=K)
    res = forest.export_ransac(scored_only=True)
    add(*(res[k] for k in ("pose", "leaf", "size", "plane", "best", "best_count")))
    for p in numbers[:3]:
        for v in grid.get_leaf_points(p):
            add(v.get_points())
    grid.filter([MinPoints(3)])
    pts = forest.export_points(-1, order=0, pose_rank=pose_rank)
    add(pts["idx"], pts["xyz"])
    st = forest.stats()
    h.update(repr((st["n_points_alive"], st["n_leaves"], st["n_blocks"])).encode())
    return h.hexdigest()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["one_block", "straddle", "all_small", "ranks"])
def test_fast_layout_matches_sorted_layout(case):
    env = dict(os.environ, OL_RANSAC_SORTED_LAYOUT="1")
    out = subprocess.run([sys.executable, os.path.abspath(__file__), case], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    sorted_digest = [l for l in out.stdout.splitlines() if l.startswith("DIGEST ")][-1].split()[1]
    assert digest(case) == sorted_digest


if __name__ == "__main__":
    print("DIGEST", digest(sys.argv[1]))
