"""Digest of a grid after every declarative leaf map (tests/test_gpu_leaf_maps.py runs it under the library's debug
switches, in a subprocess of its own, the way tests/test_gpu_toggles.py does)."""
import hashlib
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from octreelib_b200.criteria import MaxPoints  # noqa: E402
from octreelib_b200.grid import Grid, GridConfig  # noqa: E402
from octreelib_b200.leaf_maps import Centroid, FirstPoints, Shrink  # noqa: E402


def clustered_clouds(seed, n_poses=3, n=1500):
    rng = np.random.default_rng(seed)
    out = {}
    for p in range(n_poses):
        centres = rng.uniform(-10, 14, (6, 3))
        pts = np.vstack([c + rng.normal(0, rng.uniform(0.2, 1.5), (n // 6, 3)) for c in centres])
        out[p] = np.vstack([pts, rng.uniform(-12, 16, (n // 5, 3))])
    return out


def digest():
    h = hashlib.sha256()
    for obj, poses in ((Shrink(0.5), None), (Centroid(), [2, 0]), (FirstPoints(2), None)):
        grid = Grid(GridConfig(voxel_edge_length=4.0))
        for p, c in clustered_clouds(11).items():
            grid.insert_points(p, c)
        grid.subdivide([MaxPoints(25)])
        grid.map_leaf_points(obj, poses)
        for p in range(3):
            e = grid._host.forest.export_points(grid._host.pose_index[p], order=0)
            h.update(np.ascontiguousarray(e["xyz"]).tobytes())
            h.update(np.ascontiguousarray(e["idx"]).tobytes())
            h.update(np.array([grid.n_leaves(p), grid.n_points(p), grid.n_nodes(p)], dtype=np.int64).tobytes())
    return h.hexdigest()


if __name__ == "__main__":
    print("DIGEST", digest())
