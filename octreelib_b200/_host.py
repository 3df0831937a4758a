"""
`ForestHost`: the host-side logic shared by `Grid`, `OctreeManager` and `Octree` -- pose-number
bookkeeping, criteria folding, counters and object materialisation on top of one native forest.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import _views
from .criteria import CountCriterion, GeometricCriterion, NotCountOnly, as_threshold, fold_count_criteria, fold_levels
from .forest import Forest
from .leaf_maps import Centroid, FirstPoints, Shrink

__all__ = ["ForestHost"]

_TABLE_CAP = 1 << 20


class ForestHost:
    def __init__(self, edge, corner, single_cell: bool, max_depth: int = 21):
        self._edge = edge
        self._corner = corner
        self._single_cell = single_cell
        self._max_depth = max_depth
        self._forest: Optional[Forest] = None
        self.pose_index: Dict[int, int] = {}   # pose number -> dense pose index (insertion order)
        self.pose_numbers: List[int] = []      # pose index -> pose number
        self.pose_inserted: List[int] = []     # points inserted so far per pose index
        self._counts_cache = None
        # Leaf order across several subdivide calls: the reference's per-pose leaf lists grow across calls, so the order
        # depends on when a node was split and when a pose arrived.  The native forest tracks both (csrc/forest.cuh) and
        # exports blocks / points in that order; the host only needs the pose epochs for `non_empty=False` listings.
        self._n_subdivides = 0
        self._pose_epoch: Dict[int, int] = {}  # pose index -> subdivide calls made before the pose was created
        self._rows_cache = (-1, {})  # (forest version, {pose index: leaf -> row table on the device}) for locate

    # ---- plumbing --------------------------------------------------------------------------------
    @property
    def forest(self) -> Forest:
        if self._forest is None:
            corner = np.asarray(self._corner, dtype=np.float64).reshape(3)
            self._forest = Forest(float(self._edge), corner, single_cell=self._single_cell, max_depth=self._max_depth)
        return self._forest

    @property
    def empty(self) -> bool:
        return self._forest is None or not self.pose_numbers

    def _indices(self, pose_numbers: Optional[Sequence[int]]) -> Optional[List[int]]:
        if pose_numbers is None:
            return None
        return [self.pose_index[p] for p in pose_numbers]  # KeyError like the reference (octree_manager.py:56)

    # ---- insertion ------------------------------------------------------------------------------
    def insert(self, pose_number: int, points, allow_append: bool):
        # (called once per pose of a map: every attribute lookup here is host time the GPU waits for)
        pose_index = self.pose_index
        if pose_number in pose_index:
            if not allow_append:
                raise ValueError(f"Cannot insert points to existing pose {pose_number}")
            shape = getattr(points, "shape", None)
            n = int(shape[0]) if shape is not None and len(shape) == 2 else len(points)
            idx = pose_index[pose_number]
            self.forest.insert_segments(points, [n], [idx], [self.pose_inserted[idx]], len(self.pose_numbers))
            self.pose_inserted[idx] += n
        else:
            forest = self._forest or self.forest
            idx = forest.insert(points)
            assert idx == len(self.pose_numbers)
            pose_index[pose_number] = idx
            self.pose_numbers.append(pose_number)
            self.pose_inserted.append(forest.last_insert_rows)  # (the forest looked at the shape already)
            self._pose_epoch[idx] = self._n_subdivides
        self._counts_cache = None

    # ---- subdivision / filtering ----------------------------------------------------------------
    def subdivide(self, criteria: Sequence[Callable], pose_numbers: Optional[Sequence[int]] = None):
        if self.empty:
            return
        idx = self._indices(pose_numbers)
        criteria = list(criteria)
        if criteria and all(type(c).__call__ is CountCriterion.__call__ and c.op == ">" and not c.size_guarded for c in criteria):
            # any(len(points) > n_i) == len(points) > min(n_i): nothing to probe (the common case, and the host time of
            # a subdivide call is time the GPU waits)
            self.forest.subdivide(max(min(c.n for c in criteria), -1), idx)
            self._n_subdivides += 1
            self._counts_cache = None
            return
        guarded = any(isinstance(c, CountCriterion) and c.size_guarded for c in criteria)
        # [(first level, table, beyond, count criteria active from that level on, geometric terms)]; one entry unless
        # node-size guards are used
        if any(isinstance(c, GeometricCriterion) for c in criteria):
            try:
                levels = fold_levels(criteria, float(self._edge), 1024)  # (the geometric objects are not probed)
            except NotCountOnly:
                # an opaque criterion next to the geometric ones: the whole list is evaluated on the host
                self._subdivide_on_host(criteria, idx)
                self._counts_cache = None
                return
        else:
            levels = fold_levels(criteria, float(self._edge), 1024) if guarded else None
        if levels is None:
            try:
                table, beyond = fold_count_criteria(criteria, "any", 1024)
            except NotCountOnly:
                # opaque criteria (they look at coordinates): the scheme is worked out on the host, node by node like the
                # reference does, and imposed on the device (the partition itself still runs there)
                # (the native forest does not count an imposed scheme as a subdivide call: the history-dependent leaf
                # order of a SECOND subdivide, DESIGN.md section 8, is only tracked for device-evaluated criteria)
                self._subdivide_on_host(criteria, idx)
                self._counts_cache = None
                return
            levels = [(0, table, beyond, criteria, [])]
        thresholds = [as_threshold(t, b, active) if active else (1 << 62) for _, t, b, active, _ in levels]
        firsts = [lv[0] for lv in levels]
        terms = [lv[4] for lv in levels]
        if all(t is not None for t in thresholds):
            if any(terms):
                self.forest.subdivide_geometric(firsts, terms, thresholds=thresholds, pose_indices=idx)
            elif len(levels) == 1:
                self.forest.subdivide(thresholds[0], idx)
            else:
                self.forest.subdivide_levels(firsts, thresholds=thresholds, pose_indices=idx)
        else:
            n_alive = self.forest.stats()["n_points_alive"]
            upto = min(n_alive + 1, _TABLE_CAP)
            tables, beyonds = [], []
            for _, _, _, active, _ in levels:
                if active:
                    table, beyond = fold_count_criteria(active, "any", upto)
                else:
                    table, beyond = np.zeros(upto + 1, dtype=np.uint8), False
                if beyond is None:
                    if upto <= n_alive:
                        raise NotImplementedError("count criterion without a settled answer for very large nodes")
                    beyond = False
                tables.append(table)
                beyonds.append(beyond)
            if any(terms):
                self.forest.subdivide_geometric(firsts, terms, tables=tables, beyonds=beyonds, pose_indices=idx)
            elif len(levels) == 1:
                self.forest.subdivide_table(tables[0], beyonds[0], idx)
            else:
                self.forest.subdivide_levels(firsts, tables=tables, beyonds=beyonds, pose_indices=idx)
        self._n_subdivides += 1
        self._counts_cache = None

    def filter(self, criteria: Sequence[Callable], pose_numbers: Optional[Sequence[int]] = None):
        if self.empty:
            return
        idx = self._indices(pose_numbers)
        if any(isinstance(c, (CountCriterion, GeometricCriterion)) and c.size_guarded for c in criteria):
            raise NotImplementedError("node-size guards (max_depth / min_edge) apply to subdivision criteria, not to filters")
        geometric = [c for c in criteria if isinstance(c, GeometricCriterion)]
        counted = [c for c in criteria if not isinstance(c, GeometricCriterion)] if geometric else criteria
        max_block = self.forest.stats()["max_block_size"]
        upto = min(max_block + 1, _TABLE_CAP)
        try:
            table, beyond = fold_count_criteria(counted, "all", upto)
        except NotCountOnly:
            self._filter_on_host(list(criteria), idx)
            self._counts_cache = None
            return
        if upto <= max_block:  # blocks larger than the table share its last entry
            if beyond is None:
                raise NotImplementedError("count criterion without a settled answer for very large leaves")
            table[-1] = 1 if beyond else 0
        # an EMPTY leaf is also "filtered" by the reference, which changes nothing
        if geometric:
            self.forest.filter_geometric(table, [c.term() for c in geometric], idx)
        else:
            self.forest.filter(table, idx)
        self._counts_cache = None

    # ---- opaque (coordinate-dependent) criteria: evaluated on the host like the reference does -------------------------
    _HOST_SCHEME_MAX_DEPTH = 9  # what ol_forest_impose_shape can replay

    def _subdivide_on_host(self, criteria: Sequence[Callable], idx: Optional[List[int]]):
        """OctreeManager.subdivide with criteria the device cannot evaluate (octree_manager.py:36-66): per cell a scheme
        octree over the points of the listed poses (pose after pose, input order: octree_manager.py:57-61), split while any
        criterion holds (octree.py:20-32) with the reference's own routing arithmetic (octree.py:73-75, 94-97, 181-190),
        and the resulting set of split nodes imposed on the forest (`ol_forest_impose_shape`)."""
        forest = self.forest
        poses = list(range(len(self.pose_numbers))) if idx is None else list(idx)
        rows = []
        for p in poses:
            e = forest.export_points(p, order=1)
            if len(e["idx"]):
                rows.append((e["cell"].astype(np.int64), np.full(len(e["idx"]), poses.index(p), dtype=np.int64), e["idx"], e["xyz"]))
        if not rows:
            forest.impose_shape(dict(q=np.zeros((0, 3), np.int64), depth=np.zeros(0, np.uint32), path=np.zeros(0, np.uint64)))
            return
        cell = np.concatenate([r[0] for r in rows])
        order = np.lexsort((np.concatenate([r[2] for r in rows]), np.concatenate([r[1] for r in rows]), cell))
        cell, xyz = cell[order], np.vstack([r[3] for r in rows])[order]
        cells = _views.tables(forest)["cells"]
        out_q, out_depth, out_path = [], [], []

        def split(points, corner, edge, q, depth, path):
            if not any([criterion(points) for criterion in criteria]):
                return
            if depth >= self._HOST_SCHEME_MAX_DEPTH:
                raise RecursionError(f"subdivision criterion still true {depth} levels below the grid cell "
                                     "(host-evaluated criteria are limited to 9 levels)")
            out_q.append(q)
            out_depth.append(depth)
            out_path.append(path)
            half = edge / np.float64(2)
            sub = ((points - corner) // half).astype(int)
            if ((sub < 0) | (sub > 1)).any():
                raise IndexError("point outside of its octree node (reference: octree.py:98)")
            child = sub[:, 0] * 4 + sub[:, 1] * 2 + sub[:, 2]
            for c in range(8):
                off = np.array([(c >> 2) & 1, (c >> 1) & 1, c & 1]) * half
                split(points[child == c], corner + off, half, q, depth + 1, (path << 3) | c)

        bounds = np.flatnonzero(np.diff(cell)) + 1
        for lo, hi in zip(np.concatenate([[0], bounds]), np.concatenate([bounds, [len(cell)]])):
            k = int(cell[lo])
            if self._single_cell:
                corner, q = np.asarray(self._corner, dtype=np.float64).reshape(3), (0, 0, 0)
            else:
                corner, q = np.asarray(cells["corner"][k], dtype=np.float64), tuple(int(v) for v in cells["q"][k])
            split(xyz[lo:hi], corner, np.float64(self._edge), q, 0, 0)
        forest.impose_shape(dict(q=np.array(out_q, dtype=np.int64).reshape(-1, 3), depth=np.array(out_depth, dtype=np.uint32),
                                 path=np.array(out_path, dtype=np.uint64)))

    def _filter_on_host(self, criteria: Sequence[Callable], idx: Optional[List[int]]):
        """filter with opaque criteria (octree.py:102-112): every non-empty (pose, leaf) block goes to the host, the
        blocks for which not all criteria hold are emptied (keep-mask per pose -> K7 compaction)."""
        poses = list(range(len(self.pose_numbers))) if idx is None else list(idx)
        blocks = _views.tables(self.forest)["blocks"]
        plan = []
        for p in poses:
            sizes = blocks["size"][blocks["pose"] == p].astype(np.int64)
            if sizes.sum() == 0:
                continue
            xyz = self.forest.export_points(p, order=0, n_hint=int(sizes.sum()))["xyz"]
            mask = np.zeros(len(xyz), dtype=bool)
            start = 0
            for n in sizes:
                mask[start:start + n] = all([criterion(xyz[start:start + n].copy()) for criterion in criteria])
                start += n
            plan.append((p, mask))
        for p, mask in plan:
            self.forest.apply_pose_mask(p, mask)

    # ---- generic per-leaf callback (grid.py:111-122 -> octree_manager.py:68-83 -> octree.py:114-123) -----
    _DEVICE_LEAF_MAPS = (Centroid, Shrink, FirstPoints)

    def map_leaf_points(self, function: Callable, pose_numbers: Optional[Sequence[int]] = None):
        """`Centroid`, `Shrink` and `FirstPoints` (leaf_maps.py) run on the device (`ol_forest_map_leaves`) with the
        result of the host path below; any other callable - subclasses of those included, which may redefine `__call__` -
        takes the host path."""
        if type(function) not in self._DEVICE_LEAF_MAPS:
            self._map_leaf_points_on_host(function, pose_numbers)
            return
        if self.empty:
            return
        if pose_numbers is None:
            idx = None
        else:
            # unknown numbers are ignored like on the host path; a pose listed twice is mapped once
            idx = list(dict.fromkeys(self.pose_index[p] for p in pose_numbers if p in self.pose_index))
            if not idx:
                return
        rows = np.zeros(max(len(self.pose_numbers), 1), dtype=np.int64)
        try:
            self.forest.map_leaves(function.op, function.param, idx, rows)
        finally:  # (a failed post-rebuild check raises with the rows appended, like the host path)
            for p in np.flatnonzero(rows[:len(self.pose_inserted)]):
                self.pose_inserted[p] += int(rows[p])
            self._counts_cache = None

    def _map_leaf_points_on_host(self, function: Callable, pose_numbers: Optional[Sequence[int]] = None):
        """Host-callback compatibility path (SURVEY 8(f) rank 1): every non-empty (pose, leaf) block is copied to the
        host, handed to the opaque Python `function`, and the result replaces the block's points
        (grid.py:111-122 -> octree_manager.py:68-83 -> octree.py:114-123).  Like the reference, empty leaves are skipped
        and unknown poses are ignored.

        * A result that is a SELECTION of the leaf's own rows (the reference's tests use `lambda cloud: [cloud[0]]`)
          becomes a keep-mask on the device (K7 compaction).
        * Any other result (new coordinates, more or fewer points: centroids, projections onto a fitted plane, ...)
          replaces the block: its old points are removed and the new ones are appended to the same pose, after which the
          grid is rebuilt with the SAME shape (the scheme replay that also serves poses inserted after a subdivision,
          octree_manager.py:171).  Every new point must lie inside the leaf it was produced from - the forest finds a
          point's leaf from its coordinates, whereas the reference would keep a stray point in the old leaf object until
          the next subdivide mis-routes it (octree.py:94-98); a result that leaves its leaf raises NotImplementedError
          before anything is changed."""
        if self.empty:
            return
        numbers = list(self.pose_numbers) if pose_numbers is None else [p for p in pose_numbers if p in self.pose_index]
        tabs = _views.tables(self.forest)
        blocks, leaves = tabs["blocks"], tabs["leaves"]
        plan = []
        for number in numbers:
            idx = self.pose_index[number]
            sel = np.flatnonzero(blocks["pose"] == idx)
            sizes = blocks["size"][sel].astype(np.int64)
            if sizes.sum() == 0:
                continue
            xyz = self.forest.export_points(idx, order=0, n_hint=int(sizes.sum()))["xyz"]
            mask = np.zeros(len(xyz), dtype=bool)
            fresh, expect = [], []   # replacement clouds in block order / what the pose must hold afterwards
            start = 0
            for b, n in zip(sel, sizes):
                block = xyz[start:start + n]
                res = np.asarray(function(block.copy()), dtype=np.float64).reshape(-1, 3)
                keep = self._as_selection(block, res)
                if keep is not None:
                    mask[start:start + n] = keep
                    expect.append((False, block[keep]))
                else:
                    leaf = int(blocks["leaf"][b])
                    if leaves["depth"][leaf] == 0 and not self._single_cell:
                        cell = int(leaves["cell"][leaf])
                        lo = np.asarray(tabs["cells"]["corner"][cell], dtype=np.float64)
                        edge = float(self._edge)
                    elif leaves["depth"][leaf] == 0:
                        lo, edge = np.asarray(self._corner, dtype=np.float64).reshape(3), float(self._edge)
                    else:
                        lo, edge = np.asarray(leaves["corner"][leaf], dtype=np.float64), float(leaves["edge"][leaf])
                    if not np.isfinite(res).all() or ((res < lo) | (res >= lo + edge)).any():
                        raise NotImplementedError(
                            "map_leaf_points: the function returned points outside the leaf they were computed from; the "
                            "native grid locates a point by its coordinates (DESIGN.md section 8)")
                    fresh.append(res)
                    expect.append((True, res))
                start += n
            plan.append((idx, mask, fresh, expect))
        for idx, mask, fresh, expect in plan:
            self.forest.apply_pose_mask(idx, mask)
            if fresh:
                new = np.ascontiguousarray(np.vstack(fresh))
                if len(new):
                    self.forest.insert_segments(new, [len(new)], [idx], [self.pose_inserted[idx]], len(self.pose_numbers))
                    self.pose_inserted[idx] += len(new)
        self._counts_cache = None
        for idx, mask, fresh, expect in plan:
            if not fresh:
                continue
            # the rebuilt grid must hold, leaf by leaf, exactly what the reference would hold
            want = np.vstack([np.empty((0, 3))] + [pts for _, pts in expect])
            got = self.forest.export_points(idx, order=0)["xyz"]
            if got.shape != want.shape or not (got == want).all():
                raise RuntimeError("map_leaf_points: a replaced point changed its leaf during the rebuild (a point on a leaf "
                                   "boundary); the grid no longer matches the reference's result")

    @staticmethod
    def _as_selection(block: np.ndarray, res: np.ndarray):
        """keep-mask if `res` is a subsequence of the rows of `block` (bit-equal rows, in order), else None"""
        keep = np.zeros(len(block), dtype=bool)
        j, n = 0, len(block)
        for row in res:
            while j < n and not (block[j] == row).all():
                j += 1
            if j == n:
                return None
            keep[j] = True
            j += 1
        return keep

    # ---- per-leaf point statistics ------------------------------------------------------------------
    def leaf_statistics(self, pose_number: Optional[int] = None) -> dict:
        """n, mean, covariance (population, (B,3,3)), extent (per axis) and pose number of the non-empty (pose, leaf)
        blocks: of one pose in `get_leaf_points` order, or of all poses in the RANSAC batch order (pose numbers
        ascending, then the reference's leaf order).  Computed on the device (ol_forest_export_block_stats)."""
        if pose_number is not None and pose_number not in self.pose_index:
            raise KeyError(pose_number)
        if self.empty:
            return dict(n=np.zeros(0, np.int64), mean=np.zeros((0, 3)), covariance=np.zeros((0, 3, 3)), extent=np.zeros((0, 3)),
                        pose=np.zeros(0, np.int64))
        numbers = np.asarray(self.pose_numbers, dtype=np.int64)
        rank = np.empty(len(numbers), dtype=np.int32)
        rank[np.argsort(numbers, kind="stable")] = np.arange(len(numbers), dtype=np.int32)
        s = self.forest.export_block_stats(-1 if pose_number is None else self.pose_index[pose_number], rank)
        cov = np.asarray(s["cov"], dtype=np.float64)[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(-1, 3, 3)
        return dict(n=np.asarray(s["n"], dtype=np.int64), mean=np.array(s["mean"], dtype=np.float64), covariance=cov,
                    extent=np.array(s["extent"], dtype=np.float64), pose=numbers[np.asarray(s["pose"], dtype=np.int64)])

    # ---- point location ------------------------------------------------------------------------------
    def locate(self, points, pose_number: Optional[int] = None):
        """Leaf of every query point of an (n, 3) array (Grid.locate_points): its index in the leaf table, or with a pose
        number its row of `get_leaf_points(pose_number)`; -1 where there is none.  numpy in -> numpy out, a CUDA tensor
        in -> int64 CUDA tensor out."""
        if pose_number is not None and pose_number not in self.pose_index:
            raise KeyError(pose_number)
        on_device = bool(getattr(points, "is_cuda", False))
        if not on_device:
            points = np.asarray(points)
        shape = tuple(points.shape)
        if len(shape) != 2 or shape[1] != 3:
            raise ValueError(f"points must have shape (n, 3), got {shape}")
        n = shape[0]
        if self.empty or n == 0:
            if on_device:
                import torch

                return torch.full((n,), -1, dtype=torch.int64, device=points.device)
            return np.full(n, -1, dtype=np.int64)
        rows = None if pose_number is None else self._leaf_rows(self.pose_index[pose_number])
        return self.forest.locate(points, rows)

    def _leaf_rows(self, pose_index: int):
        """leaf-table index -> row of the pose's non-empty leaves (-1: no point of the pose there), from the block table
        of the current forest version; uploaded once per (version, pose)"""
        forest = self.forest
        version, cache = self._rows_cache
        if version != forest.version:
            cache = {}
            self._rows_cache = (forest.version, cache)
        rows = cache.get(pose_index)
        if rows is None:
            t = _views.tables(forest)
            blocks = t["blocks"]
            table = np.full(len(t["leaves"]["edge"]), -1, dtype=np.int32)
            sel = np.flatnonzero(blocks["pose"] == pose_index)
            table[blocks["leaf"][sel]] = np.arange(len(sel), dtype=np.int32)
            rows = cache[pose_index] = forest.upload(table)
        return rows

    # ---- counters (grid.py:343-362) --------------------------------------------------------------
    def counts(self) -> np.ndarray:
        if self._counts_cache is None or self._counts_cache[0] != self.forest.version:
            self._counts_cache = (self.forest.version, self.forest.pose_counts(len(self.pose_numbers)))
        return self._counts_cache[1]

    def count(self, pose_number: int, which: int) -> int:
        if self.empty or pose_number not in self.pose_index:
            return 0
        return int(self.counts()[self.pose_index[pose_number], which])

    # ---- materialisation -------------------------------------------------------------------------
    def leaf_voxels(self, pose_number: int, non_empty: bool, root_corner, root_edge):
        idx = self.pose_index[pose_number]
        return _views.leaf_voxels(self.forest, idx, non_empty, root_corner, root_edge, self._n_subdivides >= 2,
                                  self._pose_epoch.get(idx, 0))

    def points_dfs(self, pose_number: int) -> np.ndarray:
        if self.empty or pose_number not in self.pose_index:
            return np.empty((0, 3), dtype=float)
        return self.forest.export_points(self.pose_index[pose_number], order=1)["xyz"]

    def points_dict_order(self, pose_number: int) -> np.ndarray:
        if self.empty or pose_number not in self.pose_index:
            return np.empty((0, 3), dtype=float)
        return _views.points_dict_order(self.forest, self.pose_index[pose_number])
