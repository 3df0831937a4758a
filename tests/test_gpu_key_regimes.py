"""Wide maps against the CPU oracle: every sort-key regime of the grid build.

The build packs a point's cell coordinates (and, for out-of-order pose segments, the pose index) into one sort key of
`key_bits` bits, and picks its code path from that width:
  <= 22    32-bit key with min(8, (31 - key_bits) // 3) Morton levels embedded in its low bits
  23 .. 32 32-bit key, Morton codes in a separate array
  33 .. 64 64-bit key
  > 64     refused (ValueError)
Each map here is a few small point clusters placed so that the cell span along every axis is exactly chosen.  The
clusters sit on adversarial cells: neighbours in the packed key that differ in the top bit of one field and the bottom
bit of the next, a negative minimum cell, an axis of zero width, and cell edges 1, 2 and 3 (3 is not a power of two, so
the cell coordinate is a true floor division).  Edges stay >= 1: below 1 the reference truncates cell keys."""
import numpy as np
import pytest

from gpu_util import compare_grid_with_oracle
from octreelib_b200.criteria import MaxExtent, MaxPoints, MinPoints, extent
from octreelib_b200.grid import Grid, GridConfig
from oracle import ransac as oransac
from oracle.structure import OracleGrid

pytestmark = pytest.mark.gpu
U = 2.0 ** -53
SLAB = 416 / 1024  # a face of depth-10 nodes


def expected_key_bits(clouds, edge, pose_bits=0):
    """cell bits of the bounding box of all points (numpy floor_divide, like the reference's cell key) + pose bits"""
    q = np.floor_divide(np.vstack(list(clouds)), float(edge))
    return sum(int(hi - lo).bit_length() for lo, hi in zip(q.min(axis=0), q.max(axis=0))) + pose_bits


def cluster(rng, q, edge, n, tight=0):
    """n points over cell q, clear of its faces, half of them on a thin slab (a floor for RANSAC to find); plus `tight`
    points in one node of depth 10 on that slab"""
    u = 0.02 + 0.96 * rng.random((n, 3))
    u[: n // 2, 2] = SLAB + 4e-3 * rng.random(n // 2)
    if tight:
        u = np.vstack([u, [0.5, 0.5, SLAB] + 5e-4 * rng.random((tight, 3))])
    return (np.asarray(q, dtype=np.float64) + u) * edge


def box_cells(qmin, bits):
    """cells that make the span along axis a exactly `bits[a]` bits: the corners of the box, and pairs of cells whose
    packed keys are neighbours across a field boundary, (0, 2^by - 1, 2^bz - 1) | (1, 0, 0) and (0, 0, 2^bz - 1) | (0, 1, 0)"""
    top = [(1 << b) - 1 for b in bits]
    rel = [(x, y, z) for x in {0, top[0]} for y in {0, top[1]} for z in {0, top[2]}]
    if bits[0]:
        rel += [(0, top[1], top[2]), (1, 0, 0)]
    if bits[1]:
        rel += [(0, 0, top[2]), (0, 1, 0)]
    rel = sorted(set(rel))
    return [tuple(int(m + r) for m, r in zip(qmin, c)) for c in rel]


# (key bits, edge, minimum cell, bits per axis, the late pose's extra x bit: the width after it)
REGIMES = {
    7: (1, (0, 0, 0), (3, 2, 2), 8),                              # 8 embedded Morton levels
    22: (3, (-5, 7, -300), (8, 7, 7), 23),                        # 3 embedded levels -> 23: non-embedded 32-bit key
    23: (2, (-1000, 0, 12), (12, 11, 0), None),                   # z of zero width
    32: (1, (-3, -1 << 10, 5), (11, 11, 10), 33),                 # 32-bit -> 33: 64-bit key
    33: (3, (0, -7, 2), (11, 11, 11), None),
    64: (2, (-1 << 21, 3, -1 << 20), (22, 21, 21), None),         # every bit of the 64-bit key
}


def _regime_map(key_bits):
    edge, qmin, bits, _ = REGIMES[key_bits]
    rng = np.random.default_rng(key_bits)
    cells = box_cells(qmin, bits)
    order = rng.permutation(len(cells))
    pose0 = np.vstack([cluster(rng, cells[i], edge, 90, tight=12 if k == 0 else 0) for k, i in enumerate(order)])
    pose1 = np.vstack([cluster(rng, cells[i], edge, 50) for i in order[::2]])
    clouds = {0: pose0[rng.permutation(len(pose0))], 1: pose1}
    return edge, qmin, bits, cells, clouds, rng


def _build(edge, clouds):
    grid, og = Grid(GridConfig(voxel_edge_length=edge)), OracleGrid(edge)
    for p, c in clouds.items():
        grid.insert_points(p, c)
        og.insert_points(p, c)
    return grid, og


def _both(grid, og, call, *args):
    getattr(grid, call)(*args)
    getattr(og, call)(*args)


def lambda_bound(p):
    """|covariance(device) - covariance(numpy)| for the points p: the bound derived in csrc/geometry.cuh"""
    p = np.asarray(p, dtype=np.float64)
    n, E, M = len(p), extent(p), float(np.abs(p).max()) if len(p) else 0.0
    d0 = (n + 2) * U * (M + E)
    return 9 * (n + 8) * U * E * E + 3 * (2 * (E + d0) * d0 + (n + 3) * U * (E + d0) ** 2) + 24 * U * (E + d0) ** 2


def _check_leaf_statistics(grid, og, poses):
    for p in poses:
        stats, want = grid.leaf_statistics(p), og.get_leaf_points(p)
        assert len(stats["n"]) == len(want)
        for i, leaf in enumerate(want):
            pts = leaf.points
            n, E, M = len(pts), extent(pts), float(np.abs(pts).max())
            assert stats["n"][i] == n
            assert (stats["extent"][i] == pts.max(axis=0) - pts.min(axis=0)).all()
            assert np.abs(stats["mean"][i] - pts.mean(axis=0)).max() <= 4 * (n + 4) * U * (M + E)
            d = pts - pts.mean(axis=0)
            assert np.abs(stats["covariance"][i] - d.T @ d / n).max() <= lambda_bound(pts)


@pytest.mark.parametrize("key_bits", sorted(REGIMES))
def test_regime_matches_the_oracle(key_bits):
    edge, qmin, bits, cells, clouds, rng = _regime_map(key_bits)
    assert sum(bits) == key_bits == expected_key_bits(clouds.values(), edge)
    grid, og = _build(edge, clouds)
    # 1. one subdivision
    _both(grid, og, "subdivide", [MaxPoints(40)])
    assert grid._host.forest.stats()["key_bits"] == key_bits
    compare_grid_with_oracle(grid, og, [0, 1])
    # 2. a second one (history-dependent leaf order: the recorded shape is replayed under this key)
    _both(grid, og, "subdivide", [MaxPoints(25)])
    assert grid._host.forest.stats()["max_depth_reached"] <= 9
    compare_grid_with_oracle(grid, og, [0, 1])
    # 3. a late pose: the rebuild replays the shape; where the case says so it widens the key across a class boundary
    wider = REGIMES[key_bits][3]
    late = [cells[0], cells[-1]]
    if wider:
        late.append((qmin[0] + (1 << bits[0]), qmin[1], qmin[2]))
    clouds[2] = np.vstack([cluster(rng, q, edge, 40) for q in late])
    _both(grid, og, "insert_points", 2, clouds[2])
    want = expected_key_bits(clouds.values(), edge)
    assert want == (wider or key_bits)
    assert grid._host.forest.stats()["key_bits"] == want
    compare_grid_with_oracle(grid, og, [0, 1, 2])
    # 4. filter, then another late pose
    _both(grid, og, "filter", [MinPoints(4)])
    clouds[3] = np.vstack([cluster(rng, q, edge, 30) for q in cells[1:3]])
    _both(grid, og, "insert_points", 3, clouds[3])
    compare_grid_with_oracle(grid, og, [0, 1, 2, 3])
    _check_leaf_statistics(grid, og, [0, 1, 2, 3])
    # 5. RANSAC on the leaves: the hypothesis table is drawn from the global RNG like the reference does
    np.random.seed(42)
    table = oransac.make_table(256, 6)
    np.random.seed(42)
    grid.map_leaf_points_cuda_ransac(poses_per_batch=3, threshold=0.02, hypotheses_number=256)
    og.map_leaf_points_ransac(table, threshold=0.02, poses_per_batch=3)
    compare_grid_with_oracle(grid, og, [0, 1, 2, 3])
    assert grid.n_points(0) > len(clouds[0]) // 3
    # 6. a deep subdivision: Morton codes recomputed past depth 8 (32-bit words) and 10 (64-bit words)
    _both(grid, og, "subdivide", [MaxExtent(5e-5 * edge)])
    assert grid._host.forest.stats()["max_depth_reached"] > 10
    compare_grid_with_oracle(grid, og, [0, 1, 2, 3])
    _check_leaf_statistics(grid, og, [0, 1, 2, 3])


def test_more_than_64_key_bits_is_refused_and_leaves_no_error_behind():
    rng = np.random.default_rng(65)
    cells = box_cells((-1 << 21, 0, 5), (22, 22, 21))
    clouds = {0: np.vstack([cluster(rng, q, 2, 20) for q in cells])}
    assert expected_key_bits(clouds.values(), 2) == 65
    grid, _ = _build(2, clouds)
    with pytest.raises(ValueError, match="64"):
        grid.subdivide([MaxPoints(10)])  # the first build
    edge, _, _, _, clouds, _ = _regime_map(7)
    grid, og = _build(edge, clouds)
    _both(grid, og, "subdivide", [MaxPoints(40)])
    compare_grid_with_oracle(grid, og, [0, 1])


def _leaves_by_corner(grid, pose):
    """{(corner, edge): points} of the pose's non-empty leaves"""
    host = grid._host
    forest = host.forest
    pi = host.pose_index[pose]
    blocks, leaves = forest.export_blocks(), forest.export_leaves()
    sel = np.flatnonzero(blocks["pose"] == pi)
    xyz = forest.export_points(pi, order=0)["xyz"]
    out, start = {}, 0
    for b in sel:
        leaf, n = blocks["leaf"][b], int(blocks["size"][b])
        out[tuple(float(v) for v in leaves["corner"][leaf]) + (float(leaves["edge"][leaf]),)] = xyz[start:start + n]
        start += n
    assert start == len(xyz)
    return out


def _midpoint_appended(block):
    """new coordinates inside the block's leaf: the block plus the midpoint of its first and last point (never a
    selection of the block's rows, so every block of the pose is replaced)"""
    return np.vstack([block, (block[:1] + block[-1:]) * 0.5])


def test_pose_bits_turn_an_embedded_key_into_a_wide_one():
    rng = np.random.default_rng(21)
    edge, qmin, bits = 1, (-64, 0, 10), (7, 7, 7)
    cells = box_cells(qmin, bits)
    clouds = {p: np.vstack([cluster(rng, q, edge, 60) for q in cells[p::2]]) for p in range(3)}
    grid, og = _build(edge, clouds)
    _both(grid, og, "subdivide", [MaxPoints(30)])
    assert grid._host.forest.stats()["key_bits"] == 21 == expected_key_bits(clouds.values(), edge)
    compare_grid_with_oracle(grid, og, [0, 1, 2])
    before = og.get_leaf_points(0)
    # pose 0 now has a segment after pose 2's: 2 pose bits, 23 key bits, no embedded Morton levels
    grid.map_leaf_points(_midpoint_appended, [0])
    assert grid._host.forest.stats()["key_bits"] == 23 == expected_key_bits(clouds.values(), edge, pose_bits=2)
    got = _leaves_by_corner(grid, 0)
    assert list(got) == [tuple(float(v) for v in l.corner) + (float(l.edge),) for l in before]
    for leaf, pts in zip(before, got.values()):
        assert (pts == _midpoint_appended(leaf.points)).all()
    assert grid.n_nodes(0) == og.n_nodes(0) and grid.n_leaves(0) == og.n_leaves(0)
    compare_grid_with_oracle(grid, og, [1, 2])
    # a fresh subdivision of the rebuilt grid, against an oracle that got pose 0's mapped points in block order; the
    # native grid has one more subdivide call in its history, so leaves are matched by (corner, edge), not by position
    mapped = {0: np.vstack([_midpoint_appended(l.points) for l in before]), 1: clouds[1], 2: clouds[2]}
    _, og2 = _build(edge, mapped)
    _both(grid, og2, "subdivide", [MaxPoints(20)])
    for p in range(3):
        got = _leaves_by_corner(grid, p)
        want = {tuple(float(v) for v in l.corner) + (float(l.edge),): l.points for l in og2.get_leaf_points(p)}
        assert sorted(got) == sorted(want), f"pose {p}: leaves differ"
        for k, pts in want.items():
            assert (got[k] == pts).all(), f"pose {p}: points of leaf {k} differ"
        assert [grid.n_leaves(p), grid.n_points(p), grid.n_nodes(p)] == [og2.n_leaves(p), og2.n_points(p), og2.n_nodes(p)]


# ---- ol_forest_impose_shape ignores nodes of cells the forest does not hold -----------------------------------------

def _forest(cells, edge=1.0, n=40, seed=0):
    from octreelib_b200.forest import Forest

    rng = np.random.default_rng(seed)
    f = Forest(edge)
    f.insert(np.vstack([cluster(rng, q, edge, n) for q in cells]))
    return f


def _unsplit_state(f):
    leaves = f.export_leaves()
    st = f.stats()
    return (leaves["corner"].tolist(), leaves["edge"].tolist(), leaves["depth"].tolist(), st["n_leaves"], st["n_internal"],
            f.export_points(0)["idx"].tolist())


def _shape(rows):
    return dict(q=np.array([r[0] for r in rows], dtype=np.int64).reshape(-1, 3), depth=np.array([r[1] for r in rows], np.uint32),
                path=np.array([r[2] for r in rows], np.uint64))


def test_impose_shape_ignores_cells_whose_key_spills_into_another_field():
    a = _forest([(0, 0, 0), (0, 0, 1), (0, 1, 0), (0, 1, 1)])
    assert a.stats()["key_bits"] == 2
    fresh = _unsplit_state(a)
    # (0, 0, 2) and (0, 0, 3) pack to the keys of (0, 1, 0) and (0, 1, 1): the z field spills into y
    b = _forest([(0, 0, 2), (0, 0, 3)], seed=1)
    b.subdivide(5)
    shape = b.export_shape()
    assert {tuple(q) for q in shape["q"]} == {(0, 0, 2), (0, 0, 3)} and (shape["depth"] == 0).any()
    a.impose_shape(shape)
    assert len(a.export_shape()["depth"]) == 0
    assert _unsplit_state(a) == fresh
    # a node below the minimum cell is ignored too; a node of a held cell is split
    a.impose_shape(_shape([((-1, 1, 0), 0, 0), ((0, 0, 1), 0, 0)]))
    got = a.export_shape()
    assert got["q"].tolist() == [[0, 0, 1]] and a.stats()["n_leaves"] == 4 - 1 + 8


def test_impose_shape_ignores_cells_whose_key_runs_past_bit_63():
    top = (1 << 20) - 1
    a = _forest([(0, 0, 0), (top, top, top), (5, 0, top)], n=20)
    assert a.stats()["key_bits"] == 60
    fresh = _unsplit_state(a)
    # x = 2^24 is shifted by 40 bits: its key wraps to 0, the key of (0, 0, 0)
    a.impose_shape(_shape([((1 << 24, 0, 0), 0, 0), ((1 << 24, 0, 0), 1, 3)]))
    assert len(a.export_shape()["depth"]) == 0
    assert _unsplit_state(a) == fresh
    a.impose_shape(_shape([((1 << 24, 0, 0), 0, 0), ((-1, top, top), 0, 0), ((top, top, top), 0, 0)]))
    assert a.export_shape()["q"].tolist() == [[top, top, top]]
