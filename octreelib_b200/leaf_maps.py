"""
Declarative leaf maps for `map_leaf_points`.

The reference's `map_leaf_points(function)` hands every non-empty (pose, leaf) block to a Python callable and replaces the
block's points with what it returns (grid/grid.py:111-122 -> octree_manager.py:68-83 -> octree/octree.py:114-123).  The
host path of this library does the same (`ForestHost._map_leaf_points_on_host`): one Python call per block.  The objects
below describe the maps users write most often, so that `map_leaf_points` runs them on the GPU
(`ol_forest_map_leaves`, csrc/leaf_maps.cuh) without calling Python per block:

  * `Centroid()`       voxel downsampling: `cloud.mean(axis=0, keepdims=True)`;
  * `Shrink(factor)`   pull the points towards their leaf centroid: `c + factor * (cloud - c)`, `c = cloud.mean(axis=0)`;
  * `FirstPoints(k)`   keep the first k points of every leaf: `cloud[:k]`.

They are also plain callables, so the reference, the CPU oracle and the host path accept the very same objects; the
device results equal them bit for bit (numpy's `mean(axis=0)` of a C-contiguous (n, 3) float64 array is a sequential
row sum divided by n, which tests/test_cpu_leaf_maps.py pins).  Any other callable keeps the host path.
"""
from __future__ import annotations

import numbers

import numpy as np

from . import _native as N

__all__ = ["LeafMap", "Centroid", "Shrink", "FirstPoints"]


class LeafMap:
    """Base class of the declarative leaf maps: `op` / `param` are the arguments of `ol_forest_map_leaves`."""

    op: int = -1

    @property
    def param(self) -> float:
        return 0.0

    def __call__(self, cloud):
        raise NotImplementedError


class Centroid(LeafMap):
    """Replace a leaf's points by their mean (one point per leaf and pose)."""

    op = N.OL_MAP_CENTROID

    def __call__(self, cloud):
        return cloud.mean(axis=0, keepdims=True)

    def __repr__(self):
        return "Centroid()"


class Shrink(LeafMap):
    """Move every point of a leaf towards the leaf's mean: `c + factor * (p - c)` (factor 0: onto the mean, 1: unchanged).
    A factor that pushes points out of their leaf is refused like any other out-of-leaf result (NotImplementedError)."""

    op = N.OL_MAP_SHRINK

    def __init__(self, factor: float):
        if isinstance(factor, bool) or not isinstance(factor, numbers.Real) or not np.isfinite(float(factor)):
            raise ValueError(f"the shrink factor must be a finite real number, got {factor!r}")
        self.factor = float(factor)

    @property
    def param(self) -> float:
        return self.factor

    def __call__(self, cloud):
        c = cloud.mean(axis=0)
        return c + self.factor * (cloud - c)

    def __repr__(self):
        return f"Shrink({self.factor!r})"


class FirstPoints(LeafMap):
    """Keep the first `k` points of every leaf (all of them if it holds fewer); k = 0 empties the leaves."""

    op = N.OL_MAP_FIRST

    def __init__(self, k: int):
        if isinstance(k, bool) or not isinstance(k, numbers.Integral):
            raise TypeError(f"the number of points to keep must be an int, got {k!r}")
        if k < 0:
            raise ValueError(f"the number of points to keep must be >= 0, got {k}")
        self.k = int(k)

    @property
    def param(self) -> float:
        return float(min(self.k, 1 << 53))  # (no block holds 2^31 points)

    def __call__(self, cloud):
        return cloud[:self.k]

    def __repr__(self):
        return f"FirstPoints({self.k})"
