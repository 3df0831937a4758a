"""GPU: declarative leaf maps of `map_leaf_points` (Centroid, Shrink, FirstPoints; csrc/leaf_maps.cuh) against the
reference fixture and against the host path, which calls the equivalent plain function once per (pose, leaf) block.
Every comparison is bit for bit: points, leaf corners and edges, counters, and the point indices of export_points."""
import hashlib

import numpy as np
import pytest

from conftest import golden
from octreelib_b200.criteria import MaxExtent, MaxPoints, MinPoints
from octreelib_b200.grid import Grid, GridConfig
from octreelib_b200.leaf_maps import Centroid, FirstPoints, Shrink
from test_gpu_key_regimes import REGIMES, box_cells, cluster, expected_key_bits
from test_gpu_map_leaf_points import _check

pytestmark = pytest.mark.gpu

OBJECTS = [Centroid(), Shrink(0.5), Shrink(0.0), Shrink(0.9), FirstPoints(0), FirstPoints(1), FirstPoints(3),
           FirstPoints(1 << 40)]


def clustered_clouds(seed, n_poses=3, n=1500):
    rng = np.random.default_rng(seed)
    out = {}
    for p in range(n_poses):
        centres = rng.uniform(-10, 14, (6, 3))
        pts = np.vstack([c + rng.normal(0, rng.uniform(0.2, 1.5), (n // 6, 3)) for c in centres])
        out[p] = np.vstack([pts, rng.uniform(-12, 16, (n // 5, 3))])
    return out


def plain(obj):
    """the same map as a plain function: the host path"""
    if isinstance(obj, Centroid):
        return lambda c: c.mean(axis=0, keepdims=True)
    if isinstance(obj, Shrink):
        f = obj.factor
        return lambda c: c.mean(axis=0) + f * (c - c.mean(axis=0))
    k = obj.k
    return lambda c: c[:k]


def _grid(clouds, edge, subdivide=None):
    g = Grid(GridConfig(voxel_edge_length=float(edge)))
    for p, c in clouds.items():
        g.insert_points(p, c)
    if subdivide:
        g.subdivide(subdivide)
    return g


def _state(grid):
    host = grid._host
    out = {"inserted": list(host.pose_inserted)}
    for p in host.pose_numbers:
        for non_empty in (True, False):
            leaves = grid.get_leaf_points(p, non_empty=non_empty)
            out[p, non_empty, "corner"] = np.array([np.asarray(v.corner_min, dtype=np.float64) for v in leaves]).reshape(-1, 3)
            out[p, non_empty, "edge"] = np.array([float(v.edge_length) for v in leaves])
            out[p, non_empty, "pts"] = [np.asarray(v.get_points(), dtype=np.float64).reshape(-1, 3) for v in leaves]
        out[p, "points"] = np.asarray(grid.get_points(p), dtype=np.float64)
        out[p, "counts"] = [grid.n_leaves(p), grid.n_points(p), grid.n_nodes(p)]
        e = host.forest.export_points(host.pose_index[p], order=0)
        out[p, "xyz"], out[p, "idx"] = e["xyz"].copy(), e["idx"].copy()
    return out


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, list) and x and isinstance(x[0], np.ndarray):
            assert len(x) == len(y) and all(u.shape == v.shape and (u == v).all() for u, v in zip(x, y)), k
        else:
            x, y = np.asarray(x), np.asarray(y)
            assert x.shape == y.shape and (x == y).all(), k


def _both(ga, gb, method, *args):
    """the same call on both grids: both raise the same exception type, or both succeed"""
    errs = []
    for g in (ga, gb):
        try:
            getattr(g, method)(*args)
            errs.append(None)
        except Exception as e:  # noqa: BLE001
            errs.append(type(e))
    assert errs[0] == errs[1], errs
    return errs[0]


def _map_both(ga, gb, obj, poses=None):
    """ga: the device path (the object), gb: the host path (the plain function); True when both succeeded"""
    errs = []
    for g, fn in ((ga, obj), (gb, plain(obj))):
        try:
            g.map_leaf_points(fn, poses)
            errs.append(None)
        except Exception as e:  # noqa: BLE001
            errs.append(type(e))
    assert errs[0] == errs[1], errs
    return errs[0] is None


def _follow_up(ga, gb):
    """later operations see the same grid"""
    for method, args in (("subdivide", ([MaxPoints(6)],)), ("filter", ([MinPoints(2)],))):
        if _both(ga, gb, method, *args) is not None:
            return
        _same(_state(ga), _state(gb))
    sa, sb = ga.leaf_statistics(), gb.leaf_statistics()
    for k in sa:
        assert sa[k].shape == sb[k].shape and (sa[k] == sb[k]).all(), k
    for g in (ga, gb):
        np.random.seed(9)
        g.map_leaf_points_cuda_ransac(poses_per_batch=2, threshold=0.05, hypotheses_number=64)
    _same(_state(ga), _state(gb))


def _pair(clouds, edge, subdivide):
    return _grid(clouds, edge, subdivide), _grid(clouds, edge, subdivide)


# ---- 1. the reference's own fixture -------------------------------------------------------------------------------
def test_golden_fixture():
    g = golden("map_leaf_points_edge4")
    grid = _grid({0: g["cloud0"], 1: g["cloud1"]}, float(g["edge"]), [lambda pts: len(pts) > int(g["max_points"])])
    grid.map_leaf_points(Shrink(0.5))
    _check(grid, g, "s1")
    grid.map_leaf_points(Centroid(), [1])
    _check(grid, g, "s2")
    before = [grid.n_points(p) for p in (0, 1)]
    np.random.seed(3)
    grid.map_leaf_points_cuda_ransac(poses_per_batch=2, threshold=0.05, hypotheses_number=64)
    assert all(grid.n_points(p) <= b for p, b in zip((0, 1), before))


# ---- 2. device path == host path ----------------------------------------------------------------------------------
@pytest.mark.parametrize("obj", OBJECTS, ids=repr)
def test_clustered_map_matches_the_host_path(obj):
    ga, gb = _pair(clustered_clouds(1), 4.0, [MaxPoints(30)])
    assert _map_both(ga, gb, obj)
    _same(_state(ga), _state(gb))
    _follow_up(ga, gb)


@pytest.mark.parametrize("obj", OBJECTS, ids=repr)
def test_history_dependent_order_and_late_pose(obj):
    clouds = clustered_clouds(2, n_poses=4)
    first = {p: c for p, c in list(clouds.items())[:2]}
    ga, gb = _pair(first, 3.0, [MaxPoints(60)])
    p2, c2 = list(clouds.items())[2]
    for g in (ga, gb):
        g.insert_points(p2, c2)
        g.subdivide([MaxPoints(20)])  # second call: the leaf order depends on when a node was split and a pose came
    assert _map_both(ga, gb, obj)
    _same(_state(ga), _state(gb))
    p3, c3 = list(clouds.items())[3]
    for g in (ga, gb):
        g.insert_points(p3, c3)  # a late pose after the map: the rebuilt grid replays the shape again
    _same(_state(ga), _state(gb))
    _follow_up(ga, gb)


@pytest.mark.parametrize("obj", OBJECTS, ids=repr)
def test_pose_subsets_with_unknown_numbers(obj):
    ga, gb = _pair(clustered_clouds(3, n_poses=4), 4.0, [MaxPoints(25)])
    assert _map_both(ga, gb, obj, [2, 999, 0])
    _same(_state(ga), _state(gb))
    assert _map_both(ga, gb, obj, [3, 2])  # a second map on a pose that already holds appended rows
    _same(_state(ga), _state(gb))
    assert _map_both(ga, gb, obj, [12345])
    _same(_state(ga), _state(gb))


@pytest.mark.parametrize("obj", OBJECTS, ids=repr)
def test_deep_subdivision(obj):
    rng = np.random.default_rng(4)
    clouds = {0: np.vstack([rng.uniform(0, 8, (400, 3)), [3.1, 2.2, 5.3] + 1e-3 * rng.random((300, 3))]),
              1: rng.uniform(0, 8, (300, 3))}
    ga, gb = _pair(clouds, 8.0, [MaxExtent(4e-4)])
    assert ga._host.forest.stats()["max_depth_reached"] > 10
    # replacing rows needs a replay of the shape, which holds 9 levels: both paths refuse that the same way
    if _map_both(ga, gb, obj):
        _same(_state(ga), _state(gb))


@pytest.mark.parametrize("key_bits", [22, 23, 32, 33, 64])
@pytest.mark.parametrize("obj", [Centroid(), Shrink(0.5), FirstPoints(2)], ids=repr)
def test_key_regimes(key_bits, obj):
    edge, qmin, bits, _ = REGIMES[key_bits]
    rng = np.random.default_rng(key_bits)
    cells = box_cells(qmin, bits)
    clouds = {p: np.vstack([cluster(rng, q, edge, 50) for q in cells[p::2]]) for p in range(2)}
    assert expected_key_bits(clouds.values(), edge) == key_bits
    ga, gb = _pair(clouds, edge, [MaxPoints(20)])
    assert ga._host.forest.stats()["key_bits"] == key_bits
    assert _map_both(ga, gb, obj, [1])
    _same(_state(ga), _state(gb))
    _follow_up(ga, gb)


# ---- 3. refusal -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("factor", [3.0, -2.0])
def test_a_shrink_out_of_the_leaf_is_refused_before_anything_changes(factor):
    ga, gb = _pair(clustered_clouds(5), 4.0, [MaxPoints(30)])
    before = _state(ga)
    with pytest.raises(NotImplementedError):
        ga.map_leaf_points(Shrink(factor))
    with pytest.raises(NotImplementedError):
        gb.map_leaf_points(plain(Shrink(factor)))
    _same(_state(ga), before)
    assert ga._host.forest.stats()["n_points_inserted"] == sum(len(c) for c in clustered_clouds(5).values())
    assert _map_both(ga, gb, Shrink(0.5))
    _same(_state(ga), _state(gb))


@pytest.mark.parametrize("factor", [1.0, 1.0 - 2.0 ** -52, 1.0 + 2.0 ** -52, 1.0 + 1e-9, 0.999999])
def test_points_one_ulp_inside_the_leaf(factor):
    lo, hi = np.nextafter(0.0, 1.0), np.nextafter(2.0, 0.0)
    rng = np.random.default_rng(6)
    inner = rng.uniform(0.0, 2.0, (200, 3))
    faces = np.array([[lo, 1.0, 1.0], [hi, 1.0, 1.0], [1.0, lo, hi], [hi, hi, hi], [lo, lo, lo], [np.nextafter(1.0, 0.0), 1.0, 1.0]])
    clouds = {0: np.vstack([inner, faces]), 1: np.vstack([faces[::-1], inner[:50]])}
    for subdivide in (None, [MaxPoints(40)]):
        ga, gb = _pair(clouds, 2.0, subdivide)
        if _map_both(ga, gb, Shrink(factor)):
            _same(_state(ga), _state(gb))


# ---- 4. a large block -----------------------------------------------------------------------------------------------
def test_centroid_of_a_large_unsplit_leaf():
    rng = np.random.default_rng(8)
    pts = 99400.0 + rng.uniform(0, 900, ((1 << 18) + 77, 3))
    grid = _grid({0: pts}, 1024.0)
    grid.map_leaf_points(Centroid())
    got = np.asarray(grid.get_points(0))
    want = pts.mean(axis=0, keepdims=True)
    assert got.shape == (1, 3) and (got.view(np.uint64) == want.view(np.uint64)).all()


# ---- 5. single cell -------------------------------------------------------------------------------------------------
def _single_cell_state(obj):
    from octreelib_b200.octree import Octree, OctreeConfig
    from octreelib_b200.octree_manager import OctreeManager

    rng = np.random.default_rng(10)
    c0, c1 = rng.random((400, 3)) * 7.9, rng.random((250, 3)) * 7.9
    out = []
    for fn in (obj, plain(obj)):
        mp = OctreeManager(Octree, OctreeConfig(), np.array([0.0, 0.0, 0.0]), 8.0)
        mp.insert_points(0, c0)
        mp.insert_points(1, c1)
        mp.subdivide([MaxPoints(30)])
        mp.map_leaf_points(fn, [1, 0])
        tree = Octree(OctreeConfig(), np.array([0.0, 0.0, 0.0]), 8.0)
        tree.insert_points(c0)
        tree.subdivide([MaxPoints(30)])
        tree.map_leaf_points(fn)
        st = [[mp.n_leaves(p), mp.n_points(p), mp.n_nodes(p)] for p in (0, 1)] + [[tree.n_leaves, tree.n_points, tree.n_nodes]]
        pts = [np.asarray(mp.get_points(p)) for p in (0, 1)] + [np.asarray(tree.get_points())]
        leaves = [(tuple(np.asarray(v.corner_min, dtype=float)), float(v.edge_length), np.asarray(v.get_points()).tobytes())
                  for v in tree.get_leaf_points()]
        out.append((st, pts, leaves, list(mp._host.pose_inserted)))
    return out


@pytest.mark.parametrize("obj", OBJECTS, ids=repr)
def test_single_cell_manager_and_octree(obj):
    (sa, pa, la, ia), (sb, pb, lb, ib) = _single_cell_state(obj)
    assert sa == sb and ia == ib and la == lb
    assert all(x.shape == y.shape and (x == y).all() for x, y in zip(pa, pb))


# ---- 6. no Python call per block ------------------------------------------------------------------------------------
def test_no_per_block_python(monkeypatch):
    from octreelib_b200.octree import Octree, OctreeConfig
    from octreelib_b200.octree_manager import OctreeManager

    def refuse(self, cloud):
        raise AssertionError("called per block")

    for cls in (Centroid, Shrink, FirstPoints):
        monkeypatch.setattr(cls, "__call__", refuse)
    for obj in (Shrink(0.5), Centroid(), FirstPoints(1)):
        grid = _grid(clustered_clouds(7), 4.0, [MaxPoints(30)])
        grid.map_leaf_points(obj)
        mp = OctreeManager(Octree, OctreeConfig(), np.array([-20.0, -20.0, -20.0]), 64.0)
        tree = Octree(OctreeConfig(), np.array([-20.0, -20.0, -20.0]), 64.0)
        for p, c in clustered_clouds(7).items():
            mp.insert_points(p, c)
        tree.insert_points(clustered_clouds(7)[1])
        mp.subdivide([MaxPoints(30)])
        tree.subdivide([MaxPoints(30)])
        mp.map_leaf_points(obj)
        tree.map_leaf_points(obj)
        assert grid.n_points(1) > 0 and mp.n_points(1) > 0 and tree.n_points > 0


# ---- 7. repeatability -----------------------------------------------------------------------------------------------
def _digest():
    """digest of a grid after every declarative leaf map"""
    h = hashlib.sha256()
    for obj, poses in ((Shrink(0.5), None), (Centroid(), [2, 0]), (FirstPoints(2), None)):
        grid = _grid(clustered_clouds(11), 4.0, [MaxPoints(25)])
        grid.map_leaf_points(obj, poses)
        for p in range(3):
            e = grid._host.forest.export_points(grid._host.pose_index[p], order=0)
            h.update(np.ascontiguousarray(e["xyz"]).tobytes())
            h.update(np.ascontiguousarray(e["idx"]).tobytes())
            h.update(np.array([grid.n_leaves(p), grid.n_points(p), grid.n_nodes(p)], dtype=np.int64).tobytes())
    return h.hexdigest()


def test_leaf_maps_are_bit_identical_across_runs():
    assert _digest() == _digest()
