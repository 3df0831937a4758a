"""`Grid.locate_points` / `Grid.leaf_table` on the B200.

A query lands where `insert_points` of a new pose would have put it.  Checked two ways:
  * self-location: every stored point of every pose (`export_points(order=0)`), located with its pose, gives the row of
    the block that holds it (and without a pose, that block's leaf) - for any edge, corner, key width and depth;
  * against the CPU oracle, which walks its trees with the reference's routing (integer edges, zero corner: the
    reference's own cell keys), for random queries, points on leaf faces and one ulp on either side of them, missing
    cells, cells beyond the packed key range and non-finite rows.
"""
import hashlib

import numpy as np
import pytest

from gpu_util import torch_cuda
from octreelib_b200 import _native as N
from octreelib_b200.criteria import MaxPoints, MinPoints
from octreelib_b200.grid import Grid, GridConfig
from octreelib_b200.leaf_maps import Centroid
from oracle.structure import OracleGrid, max_points_criterion
from test_cpu_locate import oracle_locate
from test_gpu_key_regimes import REGIMES, _regime_map, cluster

pytestmark = pytest.mark.gpu


def _self_location(grid, poses):
    host = grid._host
    forest = host.forest
    blocks = forest.export_blocks()
    for p in poses:
        pi = host.pose_index[p]
        sel = blocks["pose"] == pi
        sizes = blocks["size"][sel].astype(np.int64)
        xyz = forest.export_points(pi, order=0)["xyz"]
        assert len(sizes) == len(grid.get_leaf_points(p))
        got = grid.locate_points(xyz, p)
        assert (got == np.repeat(np.arange(len(sizes)), sizes)).all(), f"pose {p}: a stored point locates to another row"
        leaf = grid.locate_points(xyz)
        assert (leaf == np.repeat(blocks["leaf"][sel], sizes)).all(), f"pose {p}: a stored point locates to another leaf"


def _build(edge, clouds, corner=(0.0, 0.0, 0.0), oracle=True):
    grid = Grid(GridConfig(voxel_edge_length=edge, corner=np.asarray(corner, dtype=np.float64)))
    og = OracleGrid(edge) if oracle else None
    for p, c in clouds.items():
        grid.insert_points(p, c)
        if og:
            og.insert_points(p, c)
    return grid, og


def _face_queries(grid, rng, n_leaves=400):
    """corners, face centres and edge midpoints of random leaves, and one ulp on either side of every coordinate"""
    t = grid.leaf_table()
    pick = rng.choice(len(t["edge"]), size=min(n_leaves, len(t["edge"])), replace=False)
    offs = np.array([(i, j, k) for i in (0, 1, 2) for j in (0, 1, 2) for k in (0, 1, 2)], dtype=np.float64) / 2
    pts = (t["corner"][pick][:, None, :] + offs[None] * t["edge"][pick][:, None, None]).reshape(-1, 3)
    return np.vstack([pts, np.nextafter(pts, np.inf), np.nextafter(pts, -np.inf)])


def _against_oracle(grid, og, poses, queries):
    assert (grid.locate_points(queries) == oracle_locate(og, queries)).all()
    for p in poses:
        assert (grid.locate_points(queries, p) == oracle_locate(og, queries, p)).all(), p


def _odd_queries(rng, edge):
    big = 2.0 ** 60
    return np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [np.nan] * 3, [big, 0, 0], [-big, 0, 0], [0, big, big],
                     [1e300, 1e300, 1e300], [-1e6 * edge, 5, 5]] + (rng.random((20, 3)) * 1e4 * edge - 5e3 * edge).tolist())


@pytest.mark.parametrize("key_bits", sorted(REGIMES))
def test_every_key_regime(key_bits):
    edge, qmin, bits, cells, clouds, rng = _regime_map(key_bits)
    grid, og = _build(edge, clouds)
    for crit in (40, 25):
        grid.subdivide([MaxPoints(crit)])
        og.subdivide([max_points_criterion(crit)])
        _self_location(grid, [0, 1])
        near = np.vstack([cluster(rng, q, edge, 30) for q in cells]) + rng.normal(0, 0.3 * edge, (30 * len(cells), 3))
        _against_oracle(grid, og, [0, 1], np.vstack([near, _face_queries(grid, rng), _odd_queries(rng, edge)]))
    # a late pose that widens the key where the regime says so: located before anything else reads the grid
    wider = REGIMES[key_bits][3]
    late = [cells[0]] + ([(qmin[0] + (1 << bits[0]), qmin[1], qmin[2])] if wider else [])
    clouds[2] = np.vstack([cluster(rng, q, edge, 40) for q in late])
    grid.insert_points(2, clouds[2])
    og.insert_points(2, clouds[2])
    _against_oracle(grid, og, [0, 1, 2], np.vstack([clouds[2], _face_queries(grid, rng), _odd_queries(rng, edge)]))
    _self_location(grid, [0, 1, 2])


@pytest.mark.parametrize("edge", [1.0, 0.25, 0.3, 5.0])
def test_edges_and_grid_corner(edge):
    """non-pow2 edges (a true floor division for the cell, depth-0 points of unsplit cells) and a grid corner that is
    not zero; with pow2 edges many points on node faces"""
    rng = np.random.default_rng(int(edge * 100))
    corner = np.array([0.375, -2.5, 11.125])
    clouds = {}
    for p in range(3):
        pts = corner + rng.random((3000, 3)) * 6 * edge - 2 * edge
        if edge in (1.0, 0.25):
            # exact node faces down to depth 3 (a dyadic corner and edge: every routing operation is exact; with a
            # non-pow2 edge a point on a face may leave its node by an ulp, which insertion itself rejects)
            on_face = rng.random(len(pts)) < 0.3
            pts[on_face] = corner + np.round((pts[on_face] - corner) / edge * 8) * edge / 8
        clouds[p] = pts
    grid, _ = _build(edge, clouds, corner, oracle=False)
    _self_location(grid, [0, 1, 2])  # unsplit cells
    grid.subdivide([MaxPoints(30)])
    _self_location(grid, [0, 1, 2])
    grid.subdivide([MaxPoints(8)])
    clouds[3] = corner + rng.random((500, 3)) * 4 * edge
    grid.insert_points(3, clouds[3])
    _self_location(grid, [0, 1, 2, 3])


def test_depth_21():
    """two points 2^-21 apart split down to the deepest level: 63 path bits"""
    base = np.array([0.5, 0.25, 0.75])
    pts = np.vstack([base, base + [2.0 ** -21, 0, 0], base + [0, 2.0 ** -21, 2.0 ** -21], [[0.1, 0.1, 0.1], [3.5, 0.5, 0.5]]])
    grid, og = _build(1, {0: pts})
    grid.subdivide([MaxPoints(1)])
    og.subdivide([max_points_criterion(1)])
    assert grid._host.forest.stats()["max_depth_reached"] == 21
    assert grid.leaf_table()["depth"].max() == 21
    _self_location(grid, [0])
    rng = np.random.default_rng(21)
    q = np.vstack([pts, np.nextafter(pts, np.inf), np.nextafter(pts, -np.inf), base + rng.random((500, 3)) * 2.0 ** -19,
                   _face_queries(grid, rng), rng.random((500, 3)) * 5 - 0.5])
    _against_oracle(grid, og, [0], q)


def _clusters(rng, n_poses, edge):
    centers = rng.random((12, 3)) * 6 * edge
    return {p: (centers[rng.integers(0, 12, 4000)] + rng.normal(0, 0.2 * edge, (4000, 3))).astype(np.float32).astype(np.float64)
            for p in range(n_poses)}


def test_history_filter_ransac_and_leaf_maps():
    rng = np.random.default_rng(7)
    clouds = _clusters(rng, 3, 2)
    grid, og = _build(2, {p: clouds[p] for p in (0, 1)})
    grid.subdivide([MaxPoints(60)])
    og.subdivide([max_points_criterion(60)])
    grid.insert_points(2, clouds[2])  # a late pose: a pending scheme replay, resolved by the locate call itself
    og.insert_points(2, clouds[2])
    _against_oracle(grid, og, [0, 1, 2], np.vstack([clouds[2][:500], rng.random((2000, 3)) * 16 - 2]))
    grid.subdivide([MaxPoints(15)])  # a second, deeper subdivide: history-dependent rows
    og.subdivide([max_points_criterion(15)])
    queries = np.vstack([clouds[0][:2000], rng.random((2000, 3)) * 16 - 2, _face_queries(grid, rng)])
    _self_location(grid, [0, 1, 2])
    _against_oracle(grid, og, [0, 1, 2], queries)
    grid.filter([MinPoints(6)])
    og.filter([lambda pts: len(pts) >= 6])
    _self_location(grid, [0, 1, 2])
    _against_oracle(grid, og, [0, 1, 2], queries)
    grid.map_leaf_points_cuda_ransac(poses_per_batch=2, threshold=0.05, hypotheses_number=64)
    _self_location(grid, [0, 1, 2])
    grid.map_leaf_points(Centroid())
    _self_location(grid, [0, 1, 2])
    t = grid.leaf_table()
    for p in (0, 1, 2):  # a pose's rows are the leaves that still hold its points
        rows = grid.locate_points(t["corner"] + t["edge"][:, None] / 2, p)
        assert sorted(set(rows[rows >= 0].tolist())) == list(range(len(grid.get_leaf_points(p))))


def test_leaf_table_matches_get_leaf_points():
    rng = np.random.default_rng(3)
    grid, _ = _build(4, {0: rng.random((5000, 3)) * 20 - 6}, oracle=False)
    grid.subdivide([MaxPoints(30)])
    t = grid.leaf_table()
    vox = grid.get_leaf_points(0, non_empty=False)
    assert len(vox) == len(t["edge"])
    assert (np.array([np.asarray(v.corner_min, dtype=np.float64) for v in vox]) == t["corner"]).all()
    assert (np.array([float(v.edge_length) for v in vox]) == t["edge"]).all()
    assert (t["edge"] == 4 * 0.5 ** t["depth"]).all()
    assert (t["cell"] == np.floor_divide(t["corner"], 4).astype(np.int64)).all()


def _street(rng, n=200_000):
    grid, _ = _build(1.0, _clusters(rng, 2, 1.0), oracle=False)
    grid.subdivide([MaxPoints(20)])
    q = rng.random((n, 3)) * 8 - 1
    return grid, q


def test_input_forms():
    torch = torch_cuda()
    rng = np.random.default_rng(11)
    grid, q = _street(rng)
    want, want_p = grid.locate_points(q), grid.locate_points(q, 1)
    assert want.dtype == np.int64 and (want >= 0).any() and (want == -1).any()
    dev = grid._host.forest.device
    t = torch.from_numpy(q).to(dev)
    got = grid.locate_points(t)
    assert got.is_cuda and got.device == t.device and got.dtype == torch.int64
    assert (got.cpu().numpy() == want).all() and (grid.locate_points(t, 1).cpu().numpy() == want_p).all()
    q32 = q.astype(np.float32)
    w32 = grid.locate_points(q32.astype(np.float64))
    assert (grid.locate_points(q32) == w32).all()
    assert (grid.locate_points(torch.from_numpy(q32).to(dev)).cpu().numpy() == w32).all()
    wide = torch.zeros((len(q), 5), dtype=torch.float64, device=dev)
    wide[:, 1:4] = t
    assert not wide[:, 1:4].is_contiguous()
    assert (grid.locate_points(wide[:, 1:4]).cpu().numpy() == want).all()
    assert (grid.locate_points(np.asfortranarray(q)) == want).all()
    assert (grid.locate_points(torch.from_numpy(q)) == want).all()  # a CPU tensor is an array-like: numpy out
    with pytest.raises(ValueError):
        grid.locate_points(t.reshape(-1))
    # a query count that is not a multiple of the block size
    n = (1 << 24) + 17
    big = torch.rand((n, 3), dtype=torch.float64, device=dev) * 8 - 1
    got = grid.locate_points(big)
    assert got.shape == (n,)
    idx = torch.randint(0, n, (100_000,), device=dev)
    assert (got[idx].cpu().numpy() == grid.locate_points(big[idx].cpu().numpy())).all()
    assert (got[-17:].cpu().numpy() == grid.locate_points(big[-17:].cpu().numpy())).all()
    # empty inputs
    assert grid.locate_points(t[:0]).shape == (0,)
    empty = Grid(GridConfig(voxel_edge_length=1.0))
    e = empty.locate_points(t[:5])
    assert e.is_cuda and (e == -1).all()


def _digest(grid, poses):
    forest = grid._host.forest
    h = hashlib.sha256()
    for part in (forest.export_cells(), forest.export_leaves(), forest.export_blocks(), forest.export_cell_poses()):
        for k in sorted(part):
            h.update(np.ascontiguousarray(part[k]).tobytes())
    for p in poses:
        e = forest.export_points(grid._host.pose_index[p], order=0)
        h.update(e["xyz"].tobytes())
        h.update(e["idx"].tobytes())
        s = grid.leaf_statistics(p)
        h.update(s["mean"].tobytes())
    stats = {k: v for k, v in forest.stats().items() if k != "device_bytes_peak"}
    return h.hexdigest(), [[grid.n_leaves(p), grid.n_points(p), grid.n_nodes(p)] for p in poses], stats


def test_no_side_effects_and_one_launch():
    torch = torch_cuda()
    rng = np.random.default_rng(5)
    grid, q = _street(rng)
    forest = grid._host.forest
    lib = N.lib()
    t = torch.from_numpy(q).to(forest.device)
    grid.locate_points(t[:10], 1)  # tables and the pose-row table of pose 1 current
    before, version = _digest(grid, [0, 1]), forest.version
    for pose in (None, 1):
        for src in (t, q):
            c0 = lib.ol_launch_count()
            grid.locate_points(src, pose)
            assert lib.ol_launch_count() - c0 <= 2, (pose, type(src))
    torch.cuda.synchronize()
    assert forest.version == version
    assert _digest(grid, [0, 1]) == before
    # a later subdivide gives what it gives on a twin grid that never located anything
    twin, _ = _street(np.random.default_rng(5))
    for g in (grid, twin):
        g.subdivide([MaxPoints(5)])
    assert _digest(grid, [0, 1]) == _digest(twin, [0, 1])


def test_profiler_stage_and_cuda_tensor_inserts():
    """deferred CUDA-tensor inserts are flushed first; the call is timed as stage `locate`"""
    torch = torch_cuda()
    rng = np.random.default_rng(9)
    clouds = _clusters(rng, 2, 1.0)
    grid, og = Grid(GridConfig(voxel_edge_length=1.0)), OracleGrid(1)
    dev = torch.device("cuda", torch.cuda.current_device())
    for p, c in clouds.items():
        grid.insert_points(p, torch.from_numpy(c).to(dev))
        og.insert_points(p, c)
    q = np.vstack([clouds[1], rng.random((3000, 3)) * 8 - 1])
    assert (grid.locate_points(q, 1) == oracle_locate(og, q, 1)).all()
    forest = grid._host.forest
    forest.profile(True)
    grid.locate_points(torch.from_numpy(clouds[0]).to(dev))
    prof = forest.profile_read()
    assert prof["locate"][0] == 1 and prof["locate"][2] == len(clouds[0])
