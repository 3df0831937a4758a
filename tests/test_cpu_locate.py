"""`Grid.locate_points` / `Grid.leaf_table` on the CPU.

1. `oracle_locate` walks the CPU oracle's trees with the reference's own routing; against every structure fixture
   recorded from the real reference, the points of row j of `get_leaf_points(k)` locate to row j of pose k, and the
   leaf-table entry they locate to without a pose has that row's corner and edge.
2. The host layer (`ForestHost.locate`: pose rows from the block table, argument checks, empty cases) runs on the
   oracle-backed fake forest (`LocatingFakeForest`).  The same scenarios run against the CUDA forest in
   test_gpu_locate.py.
"""
import numpy as np
import pytest

from conftest import golden
from fake_forest import FakeForest
from octreelib_b200.criteria import MaxPoints, MinPoints
from octreelib_b200.grid import Grid, GridConfig
from oracle.structure import OracleGrid, max_points_criterion
from test_cpu_oracle_golden import STRUCTURE_CASES, build_oracle


def leaf_order(og, key):
    """Leaves of a cell's scheme in the one-call order of the native leaf table: for every internal node in depth-first
    pre-order, its leaf children by child id (an unsplit root is the only leaf)."""
    root = og.cells[key].scheme.root
    if root.children is None:
        return [root]
    out, stack = [], [root]
    while stack:
        node = stack.pop()
        out += [ch for ch in node.children if ch.children is None]
        stack += [ch for ch in reversed(node.children) if ch.children is not None]
    return out


def oracle_locate(og, points, pose=None):
    """Where `insert_points` of a new pose would put every point of an `OracleGrid`, with the reference's own routing
    (grid.py:72-76 for the cell, octree.py:73-97 level by level below it), without inserting anything.  pose None: the
    index of the leaf in the leaf table (cells lexicographic, `leaf_order` inside a cell); pose p: the row of the leaf in
    `og.get_leaf_points(p)`.  -1: non-finite point, no such cell, the pose has no points in the leaf, or the point
    leaves its node at a split node (insertion raises IndexError, octree.py:98)."""
    points = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    out = np.full(len(points), -1, dtype=np.int64)
    index = {}
    if pose is None:
        for key in sorted(og.cells):
            for leaf in leaf_order(og, key):
                index[(key, id(leaf))] = len(index)
    else:  # the rows of get_leaf_points(pose)
        for key in og.pose_cells[pose]:
            for leaf in og.cells[key].trees[pose].cache.values():
                if len(leaf.idx):
                    index[(key, id(leaf))] = len(index)
    for i, p in enumerate(points):
        if not np.isfinite(p).all():
            continue
        with np.errstate(invalid="ignore"):  # a coordinate beyond the int64 range names no cell
            key = tuple(int(v) for v in ((p - og.corner) // og.edge * og.edge).astype(int))
        cell = og.cells.get(key)
        if cell is None:
            continue
        if pose is None:
            node = cell.scheme.root
        elif pose in cell.trees:
            node = cell.trees[pose].root
        else:
            continue
        while node is not None and node.children is not None:
            sub = ((p - node.corner) // (node.edge / 2)).astype(int)
            node = None if ((sub < 0) | (sub > 1)).any() else node.children[sub[0] * 4 + sub[1] * 2 + sub[2]]
        if node is not None:
            out[i] = index.get((key, id(node)), -1)
    return out


class LocatingFakeForest(FakeForest):
    """The oracle-backed fake forest with `ol_forest_locate`: the oracle's leaf-table index (its leaf order is the
    one-call order of `FakeForest._shape`), mapped through leaf_to_row"""

    def locate(self, points, leaf_to_row=None):
        leaf = oracle_locate(self.og, points)
        if leaf_to_row is None:
            return leaf
        out = np.full(len(leaf), -1, dtype=np.int64)
        out[leaf >= 0] = np.asarray(leaf_to_row)[leaf[leaf >= 0]]
        return out

    def upload(self, table):
        return np.array(table)


def _grid(edge):
    grid = Grid(GridConfig(voxel_edge_length=edge))
    grid._host._forest = LocatingFakeForest(edge)
    return grid


def _check_rows(og, grid, g, poses, prefix):
    """the stored points of every recorded row locate to that row (oracle and host layer), and without a pose to a leaf
    with the row's geometry"""
    table = grid.leaf_table()
    for p in poses:
        sizes = np.asarray(g[f"{prefix}p{p}_size"], dtype=np.int64)
        pts = g[f"cloud{p}"][g[f"{prefix}p{p}_idx"]]
        want = np.repeat(np.arange(len(sizes)), sizes)
        assert (oracle_locate(og, pts, p) == want).all(), (prefix, p)
        assert (grid.locate_points(pts, p) == want).all(), (prefix, p)
        leaf = grid.locate_points(pts)
        assert (leaf >= 0).all()
        assert (table["corner"][leaf] == np.repeat(g[f"{prefix}p{p}_corner"], sizes, axis=0)).all()
        assert (table["edge"][leaf] == np.repeat(g[f"{prefix}p{p}_edge"], sizes)).all()


def _both_insert(og, grid, g, p):
    og.insert_points(p, g[f"cloud{p}"])
    grid.insert_points(p, g[f"cloud{p}"])


@pytest.mark.parametrize("name", STRUCTURE_CASES)
def test_stored_points_locate_to_their_reference_rows(name):
    g = golden(name)
    og, poses = build_oracle(g)
    grid = _grid(og.edge)
    for p in poses:
        grid.insert_points(p, g[f"cloud{p}"])
    _check_rows(og, grid, g, poses, "pre_")
    sub = [int(x) for x in g["subdivide_poses"]] or None
    og.subdivide([max_points_criterion(int(g["max_points"]))], sub)
    grid.subdivide([MaxPoints(int(g["max_points"]))], sub)
    if int(g["filter_min"]) >= 0:
        og.filter([lambda pts, n=int(g["filter_min"]): len(pts) >= n])
        grid.filter([MinPoints(int(g["filter_min"]))])
    _check_rows(og, grid, g, poses, "")


def test_late_poses_locate_to_their_reference_rows():
    g = golden("late_poses_edge2")
    late = [int(p) for p in g["late"]]
    poses = [int(p) for p in g["poses"]]
    og, grid = OracleGrid(int(g["edge"])), _grid(int(g["edge"]))
    for p in poses:
        if p not in late:
            _both_insert(og, grid, g, p)
    og.subdivide([max_points_criterion(int(g["max_points"]))])
    grid.subdivide([MaxPoints(int(g["max_points"]))])
    for p in late:
        _both_insert(og, grid, g, p)
    _check_rows(og, grid, g, poses, "")


def test_history_order_rows_match_the_reference():
    """two subdivides with a pose in between: rows follow the history-dependent leaf order"""
    g = golden("resubdivide_deepen_edge4")
    late = [int(p) for p in g["late"]]
    poses = [int(p) for p in g["poses"]]
    early = [p for p in poses if p not in late]
    og, grid = OracleGrid(int(g["edge"])), _grid(int(g["edge"]))
    for p in early:
        _both_insert(og, grid, g, p)
    og.subdivide([max_points_criterion(int(g["first_max"]))])
    grid.subdivide([MaxPoints(int(g["first_max"]))])
    _check_rows(og, grid, g, early, "s1_")
    for p in late:
        _both_insert(og, grid, g, p)
    _check_rows(og, grid, g, poses, "s2_")
    og.subdivide([max_points_criterion(int(g["second_max"]))])
    grid.subdivide([MaxPoints(int(g["second_max"]))])
    _check_rows(og, grid, g, poses, "")


@pytest.mark.parametrize("seed", range(6))
def test_pose_rows_follow_random_call_sequences(seed):
    """inserts, subdivides of decreasing capacity and filters in random order; after every call the stored points of
    every pose locate to their rows and random queries agree with the oracle (the pose-row tables are cached per forest
    version, so a stale table would show here)"""
    rng = np.random.default_rng(300 + seed)
    edge = int(rng.choice([2, 4]))
    grid = _grid(edge)
    og = grid._host._forest.og
    centers = rng.random((6, 3)) * 8
    n_poses, capacity = 0, int(rng.integers(40, 120))
    for _ in range(int(rng.integers(5, 9))):
        r = rng.random()
        if n_poses == 0 or r < 0.45:
            n = int(rng.integers(100, 400))
            pts = centers[rng.integers(0, 6, n)] + rng.normal(0, 0.4, (n, 3)) + (rng.random(3) * 6 if rng.random() < 0.3 else 0)
            grid.insert_points(n_poses, pts.astype(np.float32).astype(np.float64))
            n_poses += 1
        elif r < 0.8:
            grid.subdivide([MaxPoints(capacity)])
            capacity = max(3, int(capacity * rng.uniform(0.3, 0.9)))
        else:
            grid.filter([MinPoints(int(rng.integers(2, 6)))])
        queries = np.vstack([rng.uniform(-3, 13, (300, 3)), centers[rng.integers(0, 6, 300)] + rng.normal(0, 0.4, (300, 3))])
        for p in range(n_poses):
            vox = grid.get_leaf_points(p)
            stored = np.vstack([np.empty((0, 3))] + [v.get_points() for v in vox])
            want = np.repeat(np.arange(len(vox)), [v.n_points for v in vox])
            for _ in range(2):  # the second call reads the cached table
                assert (grid.locate_points(stored, p) == want).all(), p
            assert (grid.locate_points(queries, p) == oracle_locate(og, queries, p)).all(), p
        assert (grid.locate_points(queries) == oracle_locate(og, queries)).all()


def test_errors_and_empty_cases():
    grid = _grid(2)
    # an empty grid: all -1, no forest call
    assert grid.locate_points(np.zeros((3, 3))).tolist() == [-1, -1, -1]
    table = grid.leaf_table()
    assert {k: v.shape for k, v in table.items()} == dict(corner=(0, 3), edge=(0,), depth=(0,), cell=(0, 3))
    with pytest.raises(KeyError):
        grid.locate_points(np.zeros((1, 3)), 0)
    rng = np.random.default_rng(1)
    grid.insert_points(7, rng.random((200, 3)) * 6)
    grid.subdivide([MaxPoints(20)])
    with pytest.raises(KeyError):
        grid.locate_points(np.zeros((1, 3)), 0)
    for bad in (np.zeros(3), np.zeros((2, 2)), np.zeros((2, 3, 1)), np.zeros((0,))):
        with pytest.raises(ValueError):
            grid.locate_points(bad)
        with pytest.raises(ValueError):
            grid.locate_points(bad, 7)

    def no_call(*args, **kwargs):
        raise AssertionError("locate reached the forest for zero queries")

    forest = grid._host.forest
    forest.locate = no_call
    for pose in (None, 7):
        out = grid.locate_points(np.zeros((0, 3)), pose)
        assert out.shape == (0,) and out.dtype == np.int64
    del forest.locate
    # non-finite rows, missing cells, a float32 list input; numpy int64 out
    q = [[np.nan, 1, 1], [1, np.inf, 1], [-np.inf, 1, 1], [1, 1, 1], [100, 100, 100], [-1, 1, 1]]
    out = grid.locate_points(np.asarray(q, dtype=np.float32))
    assert out.dtype == np.int64 and out.tolist()[:3] == [-1, -1, -1] and out[3] >= 0 and out[4] == -1 and out[5] == -1
    assert (grid.locate_points(q, 7) == oracle_locate(grid._host._forest.og, q, 0)).all()


def test_leaf_table_matches_the_leaf_list_of_a_one_call_grid():
    rng = np.random.default_rng(4)
    grid = _grid(4)
    grid.insert_points(0, rng.random((1500, 3)) * 12 - 4)
    grid.subdivide([MaxPoints(25)])
    table = grid.leaf_table()
    vox = grid.get_leaf_points(0, non_empty=False)
    assert len(vox) == len(table["edge"])  # one pose: it owns every cell
    assert (np.array([np.asarray(v.corner_min, dtype=np.float64) for v in vox]) == table["corner"]).all()
    assert (np.array([float(v.edge_length) for v in vox]) == table["edge"]).all()
    assert (table["depth"] == np.round(np.log2(4 / table["edge"]))).all()
    assert (table["cell"] == np.floor_divide(table["corner"], 4).astype(np.int64)).all()
    assert table["depth"].dtype == np.int32 and table["cell"].dtype == np.int64
