"""Helper of test_gpu_toggles.py (also runnable by hand): builds one grid on cuda:0 from seeded LiDAR scans, runs
subdivide + RANSAC and prints a SHA-256 over every exported table.  The digest must not depend on HOW the clouds were
handed over (pageable numpy / pinned numpy / CUDA tensors in small batches) nor on the size of the library's device
block cache (environment: OL_CACHE_BYTES)."""
import hashlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np


def digest(mode: str, n_poses: int = 11) -> str:
    import torch

    from octreelib_b200.criteria import MaxPoints
    from octreelib_b200.forest import Forest
    from octreelib_b200.grid import Grid, GridConfig
    from octreelib_b200.synthetic import lidar64_scan

    clouds = [lidar64_scan(p, seed=3) for p in range(n_poses)]  # ~120 k points each: > 2^20 in total (two-pass run segmentation)
    old = (Forest.FLUSH_EVERY, Forest.FLUSH_MIN_ROWS)
    try:
        if mode == "cuda_batches":
            Forest.FLUSH_EVERY, Forest.FLUSH_MIN_ROWS = 2, 0
            clouds = [torch.from_numpy(c).cuda() for c in clouds]
        elif mode == "pinned":
            pinned = []
            for c in clouds:
                t = torch.empty(c.shape, dtype=torch.float64, pin_memory=True)
                t.copy_(torch.from_numpy(c))
                pinned.append(t.numpy())
            clouds = pinned
        grid = Grid(GridConfig(voxel_edge_length=1.0))
        for p, c in enumerate(clouds):
            grid.insert_points(p, c)
        grid.subdivide([MaxPoints(60)])
        forest = grid._host.forest
        h = hashlib.sha256()
        leaves = forest.export_leaves()
        blocks = forest.export_blocks(list(range(n_poses)))
        for k in ("corner", "edge", "cell", "depth"):
            h.update(np.ascontiguousarray(leaves[k]).tobytes())
        for k in ("pose", "leaf", "size"):
            h.update(np.ascontiguousarray(blocks[k]).tobytes())
        np.random.seed(11)
        grid.map_leaf_points_cuda_ransac(poses_per_batch=4, threshold=0.02, hypotheses_number=128)
        res = forest.export_ransac(scored_only=True)
        for k in ("pose", "leaf", "size", "plane", "best", "best_count"):
            h.update(np.ascontiguousarray(res[k]).tobytes())
        pts = forest.export_points(-1, order=0, pose_rank=list(range(n_poses)))
        h.update(np.ascontiguousarray(pts["idx"]).tobytes())
        h.update(np.ascontiguousarray(pts["xyz"]).tobytes())
        st = forest.stats()
        h.update(repr((st["n_points_alive"], st["n_leaves"], st["n_cells"], st["n_blocks"])).encode())
        return h.hexdigest()
    finally:
        Forest.FLUSH_EVERY, Forest.FLUSH_MIN_ROWS = old


if __name__ == "__main__":
    print("DIGEST", digest(sys.argv[1] if len(sys.argv) > 1 else "numpy"))
