"""
`Grid` / `GridConfig`: the user entry point, same surface as the reference
(octreelib/grid/grid.py:21-36, 39-362), executed by the native B200 pipeline.

Mapping of the reference's per-cell Python machinery onto the device pipeline:
  insert_points  -> upload + bounding box; cell keys / sort / cell table are built lazily (K1-K3)
  subdivide      -> level-synchronous stable 8-way partition of all cells at once (K4)
  get_leaf_points-> leaf table in the reference's enumeration order (K5) + host views
  map_leaf_points_cuda_ransac -> one CTA per (pose, leaf) block (K6) + mask compaction (K7)
"""
from dataclasses import dataclass
import random
from typing import Callable, List, Optional

import numpy as np

from .._host import ForestHost
from ..internal.point import PointCloud
from ..internal.voxel import Voxel
from ..ransac.cuda_ransac import CudaRansac
from .grid_base import GridBase, GridConfigBase, GridVisualizationType, VisualizationConfig

__all__ = ["Grid", "GridConfig"]


@dataclass
class GridConfig(GridConfigBase):
    """See GridConfigBase."""


class Grid(GridBase):
    def __init__(self, grid_config: GridConfig):
        super().__init__(grid_config)
        edge = grid_config.voxel_edge_length
        corner = np.asarray(grid_config.corner, dtype=np.float64).reshape(3)
        self._host = ForestHost(edge, corner, single_cell=False)
        # the reference's cell corner is an int64 array (grid.py:72-81, 96-105); that is exact only for
        # integer-valued edges and a zero grid corner (SURVEY.md appendix A)
        self._integer_cells = float(edge) == float(int(edge)) and not corner.any()
        self.last_ransac = None

    # ---- grid.py:58-109 -------------------------------------------------------------------------
    def insert_points(self, pose_number: int, points: PointCloud):
        """Insert a pose's cloud: (n, 3) array-like (numpy, or a CUDA torch tensor to skip the upload).

        Ordinary (pageable) host arrays are consumed before the call returns, like in the reference.  A PAGE-LOCKED
        (pinned) host array is uploaded asynchronously: leave it unchanged until the next call that returns results
        (`subdivide`, `n_points`, `get_leaf_points`, ...)."""
        host = self._host
        pose_index = host.pose_index
        if pose_number in pose_index:
            raise ValueError(f"Cannot insert points to existing pose {pose_number}")
        forest = host._forest
        if forest is not None and getattr(points, "is_cuda", False) and type(points) is forest._Tensor:
            # CUDA tensors, one call per pose of a map (839 on the 100 M-point workload): the bookkeeping of
            # ForestHost.insert inline - a Python frame less per pose is 0.2 ms of host time in front of the first kernel
            idx = forest.insert(points)
            pose_index[pose_number] = idx
            host.pose_numbers.append(pose_number)
            host.pose_inserted.append(forest.last_insert_rows)
            host._pose_epoch[idx] = host._n_subdivides
            host._counts_cache = None
            return
        host.insert(pose_number, points if hasattr(points, "device") else np.asarray(points), allow_append=False)

    # ---- grid.py:111-122 ------------------------------------------------------------------------
    def map_leaf_points(self, function: Callable[[PointCloud], PointCloud], pose_numbers: Optional[List[int]] = None):
        """Host-callback compatibility path: see ForestHost.map_leaf_points (the function must return a selection of
        the leaf's own points).  The data-parallel equivalents are `filter` and `map_leaf_points_cuda_ransac`."""
        self._host.map_leaf_points(function, pose_numbers)

    # ---- grid.py:124-215 ------------------------------------------------------------------------
    def map_leaf_points_cuda_ransac(self, poses_per_batch: int = 10, threshold: float = 0.01,
                                    hypotheses_number: int = 1024, initial_points_number: int = 6):
        if threshold <= 0:
            raise ValueError("Threshold must be positive")
        if hypotheses_number < 1:
            raise ValueError("Number of RANSAC hypotheses must be positive")
        if hypotheses_number > 1024:
            raise ValueError("Number of RANSAC hypotheses must be <= 1024 because of the CUDA thread limit.")
        # same RNG draw as the reference (grid.py:160-164 -> cuda_ransac.py:39-41)
        ransac = CudaRansac(threshold=threshold, hypotheses_number=hypotheses_number,
                            initial_points_number=initial_points_number)
        host = self._host
        if host.empty:
            return
        # the reference batches pose NUMBERS range(0, P) (grid.py:149-157); any other numbering is a KeyError
        n_poses = len(host.pose_numbers)
        pose_rank = np.fromiter(host.pose_numbers, dtype=np.int64, count=n_poses)
        if pose_rank.min() < 0 or pose_rank.max() >= n_poses:  # numbers are unique: inside [0, P) means exactly range(P)
            raise KeyError(next(number for number in range(n_poses) if number not in host.pose_index))
        pose_rank = pose_rank.astype(np.int32)
        host.forest.ransac(ransac.random_hypotheses, threshold, pose_rank, poses_per_batch, apply=True)
        host._counts_cache = None

    # ---- grid.py:217-232 ------------------------------------------------------------------------
    def get_leaf_points(self, pose_number: int, non_empty: bool = True) -> List[Voxel]:
        host = self._host
        if pose_number not in host.pose_index:
            raise KeyError(pose_number)
        cells = None

        def root_corner(cell: int):
            nonlocal cells
            if cells is None:
                from .. import _views
                cells = _views.tables(host.forest)["cells"]
            if self._integer_cells:
                return (cells["q"][cell] * int(self._grid_config.voxel_edge_length)).astype(np.int64)
            return cells["corner"][cell].copy()

        return host.leaf_voxels(pose_number, non_empty, root_corner, self._grid_config.voxel_edge_length)

    def leaf_statistics(self, pose_number: Optional[int] = None) -> dict:
        """Point statistics of the non-empty leaves, computed on the GPU: a dict of numpy arrays `n` (B,), `mean` (B, 3),
        `covariance` (B, 3, 3, population), `extent` (B, 3, max - min per axis) and `pose` (B,, pose numbers).  With a
        pose number, row i belongs to `get_leaf_points(pose_number)[i]`; without, the rows cover every pose in the order
        of the RANSAC batches (pose numbers ascending, then the reference's leaf order).  An unknown pose is a KeyError.
        This is the per-(pose, leaf) hand-off of a plane-based back end (count, centroid, covariance)."""
        return self._host.leaf_statistics(pose_number)

    # ---- grid.py:234-242 ------------------------------------------------------------------------
    def get_points(self, pose_number: int) -> PointCloud:
        return self._host.points_dict_order(pose_number)

    # ---- grid.py:244-258 ------------------------------------------------------------------------
    def subdivide(self, subdivision_criteria: List[Callable[[PointCloud], bool]],
                  pose_numbers: Optional[List[int]] = None):
        host = self._host
        if pose_numbers is not None and not host.empty:
            # the reference raises KeyError as soon as a cell lacks a listed pose (octree_manager.py:56)
            from .. import _views
            cp = _views.tables(host.forest)["cell_poses"]
            n_cells = host.forest.stats()["n_cells"]
            for p in pose_numbers:
                idx = host.pose_index[p]
                if int((cp["pose"] == idx).sum()) != n_cells:
                    raise KeyError(p)
        host.subdivide(subdivision_criteria, pose_numbers)

    # ---- grid.py:260-267 ------------------------------------------------------------------------
    def filter(self, filtering_criteria: List[Callable[[PointCloud], bool]]):
        self._host.filter(filtering_criteria)

    # ---- grid.py:269-341 ------------------------------------------------------------------------
    def visualize(self, config: VisualizationConfig = VisualizationConfig()) -> None:
        """k3d HTML snapshot (host-side rendering; needs the optional `k3d` package)."""
        try:
            import k3d
        except ImportError as exc:  # pragma: no cover - k3d is not part of the GPU image
            raise ImportError("Grid.visualize needs the optional 'k3d' package") from exc
        plot = k3d.Plot()
        random.seed(config.seed)
        black = 0x000000
        colors = {}
        boxes = []
        by_pose = config.type is GridVisualizationType.POSE
        for pose_number in self._host.pose_numbers:
            # one colour per pose, or one per voxel id on its first appearance; the draws from `random` follow the
            # reference's sequence (grid.py:278-311: a voxel colour is drawn even when the voxel is then painted black)
            pose_color = random.randrange(0, 0xFFFFFF) if by_pose else None
            for leaf in self.get_leaf_points(pose_number):
                boxes.append(leaf.all_corners)
                if by_pose:
                    color = black if leaf.id in config.unused_voxels else pose_color
                else:
                    if leaf.id not in colors:
                        drawn = random.randrange(0, 0xFFFFFF)
                        colors[leaf.id] = black if leaf.id in config.unused_voxels else drawn
                    color = colors[leaf.id]
                plot += k3d.points(positions=leaf.get_points(), point_size=config.point_size, color=color)
        faces = [[0, 2, 2, 6, 6, 4, 4, 0], [0, 1, 1, 5, 5, 4, 4, 0], [0, 1, 1, 3, 3, 2, 2, 0],
                 [1, 3, 3, 7, 7, 5, 5, 1], [2, 3, 3, 7, 7, 6, 6, 2], [4, 5, 5, 7, 7, 6, 6, 4]]
        for corners in boxes:
            plot += k3d.lines(vertices=corners, indices=faces, width=config.line_width_size, color=config.line_color,
                              indices_type="segment")
        with open(config.filepath, "w") as f:
            f.write(plot.get_snapshot())

    # ---- grid.py:343-362 ------------------------------------------------------------------------
    def n_leaves(self, pose_number: int) -> int:
        return self._host.count(pose_number, 0)

    def n_points(self, pose_number: int) -> int:
        return self._host.count(pose_number, 1)

    def n_nodes(self, pose_number: int) -> int:
        return self._host.count(pose_number, 2)
