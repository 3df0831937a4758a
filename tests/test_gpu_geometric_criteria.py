"""Geometric criteria and per-leaf statistics on the GPU: the device-evaluated MaxExtent / MaxThickness / Planar against the
CPU oracle (handed the very same objects) and against the host compatibility path, and Grid.leaf_statistics against
numpy.  Thickness decisions are compared only where no node's numpy thickness lies within the bound documented in
csrc/geometry.cuh of the threshold (asserted first); extent decisions and statistics n / extent are exact."""
import math

import numpy as np
import pytest

from conftest import golden
from gpu_util import compare_grid_with_oracle
from octreelib_b200.criteria import MaxExtent, MaxPoints, MaxThickness, MinPoints, Planar, extent, thickness
from octreelib_b200.grid import Grid, GridConfig
from oracle.structure import OracleGrid

pytestmark = pytest.mark.gpu
U = 2.0 ** -53
FIXTURES = ["indoor_1pose_edge1", "lidar_2pose_edge1", "far_offset_edge1", "clustered_2pose_edge4", "random_3pose_edge2"]


def lambda_bound(p):
    """|lambda_min(device) - lambda_min(numpy)| for the points p: the bound of csrc/geometry.cuh"""
    p = np.asarray(p, dtype=np.float64)
    n, E, M = len(p), extent(p), float(np.abs(p).max()) if len(p) else 0.0
    d0 = (n + 2) * U * (M + E)
    return 9 * (n + 8) * U * E * E + 3 * (2 * (E + d0) * d0 + (n + 3) * U * (E + d0) ** 2) + 24 * U * (E + d0) ** 2


def thickness_margin(p):
    dl = lambda_bound(p)
    t = thickness(p)
    return min(math.sqrt(dl), dl / t) if t > 0 else math.sqrt(dl)


def _inputs(name):
    g = golden(name)
    edge = float(g["edge"])
    edge = int(edge) if edge == int(edge) else edge
    return edge, {int(p): g[f"cloud{int(p)}"] for p in g["poses"]}


def _synthetic():
    from octreelib_b200.synthetic import indoor_scene

    return 1, {0: indoor_scene(20000, seed=5), 1: indoor_scene(20000, seed=6)}


def _build(edge, clouds):
    grid = Grid(GridConfig(voxel_edge_length=edge))
    og = OracleGrid(edge)
    for p, c in clouds.items():
        grid.insert_points(p, c)
        og.insert_points(p, c)
    return grid, og


def _oracle_subdivide_recording(og, criteria, pose_numbers=None):
    """subdivide the oracle with the given objects; returns the point sets of every node a criterion was evaluated on"""
    seen = []

    def rec(points):
        seen.append(np.array(points))
        return False

    og.subdivide([rec] + list(criteria), pose_numbers)
    return seen


def _assert_clear_of_threshold(point_sets, t, min_points):
    for p in point_sets:
        if len(p) >= min_points:
            assert abs(thickness(p) - t) > thickness_margin(p), "a node lies within the documented margin of the threshold"


@pytest.mark.parametrize("name", FIXTURES + ["synthetic_indoor"])
@pytest.mark.parametrize("kind", ["extent", "thickness", "mixed"])
def test_device_criteria_match_the_oracle(name, kind):
    edge, clouds = _synthetic() if name == "synthetic_indoor" else _inputs(name)
    crits = {"extent": [MaxExtent(edge / 5)],
             "thickness": [MaxThickness(0.031, min_points=6, min_edge=edge / 64)],
             "mixed": [MaxPoints(100), MaxThickness(0.031, min_edge=edge / 16)]}[kind]
    grid, og = _build(edge, clouds)
    seen = _oracle_subdivide_recording(og, crits)
    if kind != "extent":
        _assert_clear_of_threshold(seen, 0.031, 4)
    grid.subdivide(crits)
    compare_grid_with_oracle(grid, og, list(clouds))


def test_device_matches_the_host_path():
    edge, clouds = _inputs("lidar_2pose_edge1")
    for crit in (MaxExtent(0.2), MaxThickness(0.03, min_points=5)):
        a, og = _build(edge, clouds)
        b, _ = _build(edge, clouds)
        if isinstance(crit, MaxThickness):
            _assert_clear_of_threshold(_oracle_subdivide_recording(og, [crit]), 0.03, 5)
        a.subdivide([crit])
        b.subdivide([lambda p: crit(p)])  # opaque to the probe: the host path
        sa, sb = a._host.forest.export_shape(), b._host.forest.export_shape()
        assert max(sa["depth"].tolist() or [0]) <= 8
        for k in ("q", "depth", "path"):
            assert (sa[k] == sb[k]).all()
        for p in clouds:
            va, vb = a.get_leaf_points(p), b.get_leaf_points(p)
            assert len(va) == len(vb) and all((x.get_points() == y.get_points()).all() for x, y in zip(va, vb))
        # filter: keep planar leaves of at least 5 points
        blocks = [v.get_points() for p in clouds for v in a.get_leaf_points(p)]
        _assert_clear_of_threshold(blocks, 0.01, 3)
        planar = Planar(0.01)
        a.filter([planar, MinPoints(5)])
        b.filter([lambda p: planar(p) and len(p) >= 5])
        for p in clouds:
            assert (a._host.forest.export_points(a._host.pose_index[p])["xyz"] ==
                    b._host.forest.export_points(b._host.pose_index[p])["xyz"]).all()
            assert a.n_points(p) == b.n_points(p) and a.n_leaves(p) == b.n_leaves(p)


def test_pose_subsets_history_and_late_inserts():
    edge, clouds = _inputs("random_3pose_edge2")
    late = clouds.pop(2)
    grid, og = _build(edge, clouds)
    og.subdivide([MaxExtent(0.6)], [1])
    grid.subdivide([MaxExtent(0.6)], [1])  # the scheme from pose 1's points only
    compare_grid_with_oracle(grid, og, [0, 1])
    og.subdivide([MaxExtent(0.3), MaxPoints(40)])
    grid.subdivide([MaxExtent(0.3), MaxPoints(40)])  # second call: the history-dependent leaf order
    compare_grid_with_oracle(grid, og, [0, 1])
    og.insert_points(2, late)
    grid.insert_points(2, late)  # a late pose follows the scheme
    compare_grid_with_oracle(grid, og, [0, 1, 2])


def test_depth_beyond_the_host_path_and_the_cap():
    rng = np.random.default_rng(4)
    pts = np.vstack([[0.3, 0.3, 0.3] + rng.random((40, 3)) * 2e-3, rng.random((40, 3))])
    grid, og = _build(1, {0: pts})
    crit = MaxExtent(2e-4)
    og.subdivide([crit])
    grid.subdivide([crit])
    compare_grid_with_oracle(grid, og, [0])
    assert grid._host.forest.stats()["max_depth_reached"] > 9  # deeper than the host path can replay
    host, _ = _build(1, {0: pts})
    with pytest.raises(RecursionError):
        host.subdivide([lambda p: crit(p)])
    never, _ = _build(1, {0: pts[:5]})
    with pytest.raises(RecursionError):
        never.subdivide([Planar(1.0, min_points=1)])  # true on every non-empty node: never stops


def _adversarial_grid():
    rng = np.random.default_rng(9)
    cells = [
        1e5 + 0.2 + rng.random((300, 3)) * 0.5,                                        # 1e5 m from the origin
        np.array([3.5, 0.5, 0.5]) + rng.random((50, 3)) * 1e-4,                        # 1e-4 m extent
        np.column_stack([5.1 + rng.random((80, 2)) * 0.8, np.full(80, 0.25)]),         # exactly planar
        np.array([7.2, 0.1, 0.1]) + np.outer(rng.random(60), [0.5, 0.25, 0.125]),      # collinear
        np.repeat(np.array([[9.5, 0.5, 0.5]]), 17, axis=0),                            # duplicated point
        np.array([[11.5, 0.5, 0.5]]),                                                  # n = 1
        np.array([[13.1, 0.2, 0.3], [13.7, 0.9, 0.4]]),                                # n = 2
        -2e5 - rng.random((500, 3)) * 0.9,                                             # far on the other side
    ]
    grid = Grid(GridConfig(voxel_edge_length=1.0))
    clouds = {5: np.vstack(cells[:5]), 2: np.vstack(cells[5:])}
    for p, c in clouds.items():
        grid.insert_points(p, c)
    return grid, clouds


def _check_stats(stats, voxels):
    assert len(stats["n"]) == len(voxels)
    for i, v in enumerate(voxels):
        p = np.asarray(v.get_points(), dtype=np.float64)
        n = len(p)
        assert stats["n"][i] == n
        assert (stats["extent"][i] == p.max(axis=0) - p.min(axis=0)).all()
        E, M = extent(p), float(np.abs(p).max())
        assert np.abs(stats["mean"][i] - p.mean(axis=0)).max() <= 4 * (n + 4) * U * (M + E)
        d = p - p.mean(axis=0)
        assert np.abs(stats["covariance"][i] - d.T @ d / n).max() <= lambda_bound(p)
        assert (stats["covariance"][i] == stats["covariance"][i].T).all()


def test_leaf_statistics_adversarial_leaves_and_row_order():
    grid, clouds = _adversarial_grid()
    for p in clouds:
        _check_stats(grid.leaf_statistics(p), grid.get_leaf_points(p))
    every = grid.leaf_statistics()
    assert every["pose"].tolist() == sorted(every["pose"].tolist())  # pose numbers ascending (2 before 5)
    order = [v for p in sorted(clouds) for v in grid.get_leaf_points(p)]
    _check_stats(every, order)
    with pytest.raises(KeyError):
        grid.leaf_statistics(3)
    # after a geometric subdivision and a geometric filter as well
    grid.subdivide([MaxExtent(0.2)])
    grid.filter([Planar(0.05)])
    for p in clouds:
        _check_stats(grid.leaf_statistics(p), grid.get_leaf_points(p))


def test_leaf_statistics_on_a_lidar_map():
    edge, clouds = _inputs("lidar_2pose_edge1")
    grid, _ = _build(edge, clouds)
    grid.subdivide([MaxPoints(2000)])  # leaves of several thousand points: more than one chunk per leaf
    for p in clouds:
        _check_stats(grid.leaf_statistics(p), grid.get_leaf_points(p))


def _digest():
    import hashlib

    from octreelib_b200.synthetic import lidar64_scan

    grid = Grid(GridConfig(voxel_edge_length=1.0))
    for p in range(4):
        grid.insert_points(p, lidar64_scan(p, seed=3))
    grid.subdivide([MaxPoints(500), MaxThickness(0.02, min_edge=0.125)])
    h = hashlib.sha256()
    for k, v in sorted(grid.leaf_statistics().items()):
        h.update(k.encode())
        h.update(np.ascontiguousarray(v).tobytes())
    grid.filter([Planar(0.03)])
    h.update(grid._host.forest.export_points(0)["xyz"].tobytes())
    return h.hexdigest()


def test_statistics_are_bit_identical_across_runs():
    assert _digest() == _digest()


def test_single_cell_octree_manager():
    from octreelib_b200.octree import Octree, OctreeConfig
    from octreelib_b200.octree_manager import OctreeManager

    rng = np.random.default_rng(2)
    c0 = np.column_stack([rng.random((300, 2)) * 7.9, 0.2 * rng.random(300) + 3.0])
    c1 = rng.random((200, 3)) * 7.9
    mp = OctreeManager(Octree, OctreeConfig(), np.array([0, 0, 0]), 8)
    mp.insert_points(0, c0)
    mp.insert_points(1, c1)
    mp.subdivide([MaxExtent(2.5)])
    # restate with the oracle's tree on the same single cell
    from oracle.structure import _Tree

    scheme = _Tree(np.array([0, 0, 0]), 8)
    scheme.insert(scheme.root, np.arange(500), np.vstack([c0, c1]))
    scheme.subdivide(scheme.root, [MaxExtent(2.5)])
    want_nodes = scheme.n_nodes()
    assert mp.n_nodes(0) == mp.n_nodes(1) == want_nodes
    for p, c in ((0, c0), (1, c1)):
        t = _Tree(np.array([0, 0, 0]), 8)
        t.insert(t.root, np.arange(len(c)), c)
        t.subdivide_as(t.root, scheme.root)
        assert mp.n_leaves(p) == sum(1 for l in t.cache.values() if len(l.idx))
        assert mp.n_points(p) == len(c)

