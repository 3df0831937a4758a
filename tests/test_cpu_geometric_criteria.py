"""Geometric criteria (MaxExtent / MaxThickness / Planar) on the CPU: the objects as plain callables against numpy, their
node-size guards through the oracle, the level folding, and the host dispatch of `Grid.subdivide` / `filter` on a
forest stand-in that answers the new native calls with the oracle."""
import numpy as np
import pytest

from fake_forest import FakeForest
from octreelib_b200 import criteria as crit_mod
from octreelib_b200.criteria import (NO_LEVEL_LIMIT, GeometricCriterion, MaxExtent, MaxPoints, MaxThickness, MinPoints, Planar,
                                     _edge_of_node_under_test, as_threshold, extent, fold_levels, halvings, thickness)
from octreelib_b200.grid import Grid, GridConfig
from oracle.structure import OracleGrid


def _np_thickness(p):
    c = np.cov(np.asarray(p, dtype=np.float64).T, bias=True)
    return float(np.sqrt(max(np.linalg.eigvalsh(c)[0], 0.0)))


def _term_holds(term, pts):
    stat, op, min_points, value = term
    if len(pts) < min_points:
        return False
    v = extent(pts) if stat == 0 else thickness(pts)
    return v > value if op == 0 else v <= value


class GeomFakeForest(FakeForest):
    """FakeForest plus the geometric forest calls (restated from the native semantics), recording every mutating call."""

    def __init__(self, edge):
        super().__init__(edge)
        self.calls = []

    def subdivide(self, *a, **k):
        self.calls.append("subdivide")
        super().subdivide(*a, **k)

    def subdivide_table(self, *a, **k):
        self.calls.append("subdivide_table")
        super().subdivide_table(*a, **k)

    def subdivide_levels(self, *a, **k):
        self.calls.append("subdivide_levels")
        super().subdivide_levels(*a, **k)

    def impose_shape(self, *a, **k):
        self.calls.append("impose_shape")
        super().impose_shape(*a, **k)

    def filter(self, *a, **k):
        self.calls.append("filter")
        super().filter(*a, **k)

    def apply_pose_mask(self, *a, **k):
        self.calls.append("apply_pose_mask")
        super().apply_pose_mask(*a, **k)

    def subdivide_geometric(self, first_levels, terms, thresholds=None, tables=None, beyonds=None, pose_indices=None):
        self.calls.append("subdivide_geometric")
        firsts = [int(f) for f in first_levels]

        def rule(pts):
            level = halvings(self.edge, _edge_of_node_under_test())
            e = max(i for i, f in enumerate(firsts) if f <= level)
            if tables is None:
                count = len(pts) > int(thresholds[e])
            else:
                t = np.asarray(tables[e])
                count = bool(t[len(pts)]) if len(pts) < len(t) else bool(beyonds[e])
            return count or any(_term_holds(t, pts) for t in terms[e])

        self.og.subdivide([rule], pose_indices)
        self._after_subdivide()

    def filter_geometric(self, keep_table, terms, pose_indices=None):
        self.calls.append("filter_geometric")
        table = np.asarray(keep_table)
        self.og.filter([lambda pts: bool(table[min(len(pts), len(table) - 1)]) and all(_term_holds(t, pts) for t in terms)],
                       pose_indices)
        self.version += 1


def _scene(seed=3, n=600):
    """two poses: a tilted plane with noise plus a cluster, inside cells of edge 4"""
    rng = np.random.default_rng(seed)
    clouds = []
    for p in range(2):
        uv = rng.random((n, 2)) * 7.9
        z = 0.3 * uv[:, 0] + 0.1 * uv[:, 1] + rng.normal(0, 0.02, n) + 0.5
        blob = rng.normal([2.0, 6.0, 2.0], 0.3, (n // 3, 3))
        clouds.append(np.vstack([np.column_stack([uv, np.clip(z, 0, 7.9)]), np.clip(blob, 0.01, 7.9)]))
    return clouds


def _grid(edge, clouds):
    grid = Grid(GridConfig(voxel_edge_length=edge))
    grid._host._forest = GeomFakeForest(edge)
    for p, c in enumerate(clouds):
        grid.insert_points(p, c)
    return grid


def _oracle(edge, clouds):
    og = OracleGrid(edge)
    for p, c in enumerate(clouds):
        og.insert_points(p, c)
    return og


def _same(grid, og, poses):
    for p in poses:
        vox = grid.get_leaf_points(p)
        want = og.get_leaf_points(p)
        assert len(vox) == len(want)
        for v, w in zip(vox, want):
            assert (np.asarray(v.corner_min, dtype=np.float64) == np.asarray(w.corner, dtype=np.float64)).all()
            assert float(v.edge_length) == float(w.edge)
            assert (v.get_points() == w.points).all()
        assert [grid.n_leaves(p), grid.n_points(p), grid.n_nodes(p)] == [og.n_leaves(p), og.n_points(p), og.n_nodes(p)]


# ---- the objects as plain callables ----------------------------------------------------------------------------------
def test_statistics_match_numpy_definitions():
    rng = np.random.default_rng(0)
    flat = np.column_stack([rng.random((50, 2)) * 3, np.full(50, 2.5)])
    assert thickness(flat) == 0.0
    tilted = np.column_stack([flat[:, :2], 0.5 * flat[:, 0] - 0.25 * flat[:, 1]])
    assert thickness(tilted) < 1e-7
    slab = np.column_stack([rng.random((20000, 2)) * 10, rng.normal(0, 0.05, 20000)])
    assert thickness(slab) == pytest.approx(_np_thickness(slab), rel=1e-12)
    assert thickness(slab) == pytest.approx(0.05, rel=0.05)
    assert extent(slab) == float(np.ptp(slab, axis=0).max())
    empty = np.empty((0, 3))
    assert extent(empty) == 0.0 and thickness(empty) == 0.0 and thickness(slab[:2]) == 0.0
    assert not MaxExtent(0.0)(empty) and MaxExtent(9.0)(slab) and not MaxExtent(10.0)(slab)
    assert MaxThickness(0.04)(slab) and not MaxThickness(0.06)(slab)
    assert not MaxThickness(0.0, min_points=4)(slab[:3])  # n < min_points
    assert Planar(0.06)(slab) and not Planar(0.04)(slab)
    assert not Planar(1.0, min_points=3)(slab[:2]) and Planar(1.0, min_points=3)(slab[:3])
    assert MaxThickness(0.01).term() == (1, 0, 4, 0.01) and Planar(0.02).term() == (1, 1, 3, 0.02)
    assert MaxExtent(2.0).term() == (0, 0, 1, 2.0)


def test_arguments_are_validated():
    for bad in (lambda: MaxExtent(-1.0), lambda: MaxThickness(-0.1), lambda: Planar(0.1, min_points=0),
                lambda: MaxThickness(0.1, min_points=0), lambda: MaxThickness(float("nan")), lambda: MaxExtent(1.0, min_edge=0.0),
                lambda: GeometricCriterion("linearity", ">", 1.0), lambda: GeometricCriterion("extent", "<", 1.0)):
        with pytest.raises(ValueError):
            bad()
    for name in ("GeometricCriterion", "MaxExtent", "MaxThickness", "Planar"):
        assert name in crit_mod.__all__


def test_guards_reuse_the_count_guard_logic_through_the_oracle():
    clouds = _scene()
    c = MaxThickness(0.0, min_edge=0.5)
    assert c.level_limit(4.0) == MaxPoints(0, min_edge=0.5).level_limit(4.0) == 3
    assert MaxExtent(1.0, max_depth=2).level_limit(4.0) == 2 and MaxExtent(1.0).level_limit(4.0) == NO_LEVEL_LIMIT
    og = _oracle(4, clouds)
    og.subdivide([c])
    leaves = og.get_leaf_points(0)
    assert min(float(l.edge) for l in leaves) == 0.5  # thickness > 0 everywhere: split down to the guard
    with pytest.raises(NotImplementedError):  # a guarded criterion called outside a subdivision has no node to look at
        c(clouds[0])


# ---- level folding ----------------------------------------------------------------------------------------------------
def test_fold_levels_of_a_mixed_list():
    lv = fold_levels([MaxPoints(100), MaxThickness(0.05, min_edge=0.25)], 1.0, 64)
    assert [l[0] for l in lv] == [0, 2]
    assert lv[0][4] == [(1, 0, 4, 0.05)] and lv[1][4] == []
    assert as_threshold(lv[0][1], lv[0][2], lv[0][3]) == 100 and as_threshold(lv[1][1], lv[1][2], lv[1][3]) == 100
    lv = fold_levels([MaxExtent(0.5)], 1.0, 64)
    assert len(lv) == 1 and lv[0][3] == [] and lv[0][4] == [(0, 0, 1, 0.5)] and not lv[0][1].any()


# ---- host dispatch ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("make", [
    lambda: [MaxThickness(0.05, min_points=6)],
    lambda: [MaxPoints(100), MaxThickness(0.05, min_edge=0.5)],
    lambda: [MaxExtent(1.5), lambda p: len(p) > 300],
    lambda: [MaxExtent(0.7, max_depth=2, voxel_edge_length=4), MaxPoints(50, min_edge=1.0)],
])
def test_geometric_lists_reach_the_device_call_without_probing(make, monkeypatch):
    clouds = _scene()
    og = _oracle(4, clouds)
    og.subdivide(make())
    grid = _grid(4, clouds)

    def no_probe(self, points):
        raise AssertionError("a geometric criterion was probed")

    monkeypatch.setattr(GeometricCriterion, "on_points", no_probe)
    grid.subdivide(make())
    monkeypatch.undo()
    assert grid._host._forest.calls == ["subdivide_geometric"]
    assert grid._host._n_subdivides == 1
    _same(grid, og, [0, 1])


def test_geometric_subdivide_with_pose_subset_and_a_second_call():
    clouds = _scene()
    og = _oracle(4, clouds)
    grid = _grid(4, clouds)
    for crits, poses in (([MaxExtent(2.0)], [1]), ([MaxExtent(0.9)], None)):
        og.subdivide(crits, poses)
        grid.subdivide(crits, poses)
    assert grid._host._forest.calls == ["subdivide_geometric"] * 2
    _same(grid, og, [0, 1])


def test_opaque_lambda_next_to_a_geometric_criterion_takes_the_host_path():
    clouds = _scene()
    og = _oracle(4, clouds)
    crits = [MaxThickness(0.05), lambda p: len(p) > 3 and p[:, 0].mean() > 3.0]
    og.subdivide(crits)
    grid = _grid(4, clouds)
    grid.subdivide(crits)
    assert grid._host._forest.calls == ["impose_shape"]
    _same(grid, og, [0, 1])


@pytest.mark.parametrize("crits, calls", [
    ([MaxPoints(40)], ["subdivide"]),
    ([lambda p: len(p) > 40], ["subdivide"]),
    ([lambda p: len(p) > 40 and len(p) % 2 == 0], ["subdivide_table"]),
    ([MaxPoints(40, max_depth=2)], ["subdivide_levels"]),
])
def test_count_only_lists_make_the_calls_they_always_made(crits, calls):
    grid = _grid(4, _scene())
    grid.subdivide(crits)
    assert grid._host._forest.calls == calls


def test_filter_dispatch():
    clouds = _scene()
    og = _oracle(4, clouds)
    grid = _grid(4, clouds)
    og.subdivide([MaxPoints(40)])
    grid.subdivide([MaxPoints(40)])
    og.filter([Planar(0.03), MinPoints(5)])
    grid.filter([Planar(0.03), MinPoints(5)])
    assert grid._host._forest.calls == ["subdivide", "filter_geometric"]
    _same(grid, og, [0, 1])
    grid.filter([MinPoints(7)])
    assert grid._host._forest.calls[-1] == "filter"
    grid.filter([Planar(0.02), lambda p: len(p) > 0 and p[:, 2].mean() > 1.0])  # opaque: every block goes to the host
    assert grid._host._forest.calls[-1] == "apply_pose_mask"
    with pytest.raises(NotImplementedError):
        grid.filter([MaxThickness(0.1, min_edge=0.5)])
