"""GPU (single device): the device side of the multi-GPU path - owner partition kernel, run-based
insertion - checked by emulating the ranks one after the other in one process, then comparing the
union of the per-rank results with a plain single-GPU Grid and with the oracle."""
import ctypes as C

import numpy as np
import pytest

from octreelib_b200 import _native as N
from octreelib_b200.criteria import MaxPoints
from octreelib_b200.forest import Forest, TorchAllocator
from octreelib_b200.grid import Grid, GridConfig
from octreelib_b200.parallel import routing_layout, segments_from_counts
from octreelib_b200.synthetic import lidar64_scan

pytestmark = pytest.mark.gpu


def _partition(points_list, edge, world, bounds=None):
    import torch

    lib = N.lib()
    dev = torch.device("cuda", 0)
    local = torch.from_numpy(np.vstack(points_list)).to(dev)
    sizes = np.array([len(p) for p in points_list], dtype=np.int64)
    send = torch.empty_like(local)
    counts = np.zeros((world, len(points_list)), dtype=np.int64)
    alloc = TorchAllocator(dev)
    corner = (C.c_double * 3)(0.0, 0.0, 0.0)
    b = None if bounds is None else np.ascontiguousarray(bounds, dtype=np.int64)
    N.check(lib.ol_partition_by_owner(C.c_void_p(torch.cuda.current_stream(dev).cuda_stream), C.c_void_p(local.data_ptr()),
                                      len(local), sizes.ctypes.data_as(C.c_void_p), len(sizes), float(edge), C.byref(corner),
                                      world, None if b is None else b.ctypes.data_as(C.c_void_p), C.c_void_p(send.data_ptr()),
                                      counts.ctypes.data_as(C.c_void_p), alloc.alloc_cb, alloc.free_cb, None))
    return send.cpu().numpy(), counts


def test_slab_histogram_boundaries_and_owner():
    """Slab partition: the device histogram of the leading cell coordinate, the quantile boundaries every rank derives
    from the gathered histograms, and the owner rule of the partition kernel (owner = number of boundaries <= ix)."""
    import torch

    from octreelib_b200.parallel import SLAB_BINS, slab_boundaries

    lib = N.lib()
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(4)
    world = 4
    clouds = [(rng.normal(0, 40, (20000, 3)) + np.array([60.0 * r, 0, 0])).astype(np.float32).astype(np.float64) for r in range(world)]
    gathered = np.zeros((world, 2 + SLAB_BINS), dtype=np.int64)
    for r, c in enumerate(clouds):
        t = torch.from_numpy(c).to(dev)
        out = torch.empty(2 + SLAB_BINS, dtype=torch.int64, device=dev)
        N.check(lib.ol_slab_histogram(C.c_void_p(torch.cuda.current_stream(dev).cuda_stream), C.c_void_p(t.data_ptr()), len(c), 2.0, 0.0,
                                      SLAB_BINS, C.c_void_p(out.data_ptr())))
        gathered[r] = out.cpu().numpy()
        ix = np.floor_divide(c[::8, 0], 2.0).astype(np.int64)  # the kernels look at every 8th point
        assert gathered[r, 0] == ix.min() and gathered[r, 1] == ix.max() and gathered[r, 2:].sum() == len(ix)
        width = max(1, -(-(ix.max() - ix.min() + 1) // SLAB_BINS))
        assert (gathered[r, 2:] == np.bincount((ix - ix.min()) // width, minlength=SLAB_BINS)).all()
    bounds = slab_boundaries(gathered, world)
    assert len(bounds) == world - 1 and (np.diff(bounds) >= 0).all()
    allpts = np.vstack(clouds)
    owner = np.searchsorted(bounds, np.floor_divide(allpts[:, 0], 2.0).astype(np.int64), side="right")
    share = np.bincount(owner, minlength=world) / len(allpts)
    assert share.min() > 0.2 and share.max() < 0.3, share
    send, counts = _partition(clouds, 2.0, world, bounds)
    run = np.concatenate([np.full(len(c), j) for j, c in enumerate(clouds)])
    order = np.lexsort((np.arange(len(allpts)), run, owner))
    assert (send == allpts[order]).all()
    exp = np.zeros_like(counts)
    np.add.at(exp, (owner, run), 1)
    assert (counts == exp).all()


def test_emulated_slab_ranks_reproduce_the_single_gpu_batch_layout():
    """Three 'ranks' with slab ownership, processed one after the other: with `pose_start` from the gathered pose sizes
    every rank's RANSAC uses the reference's batch-global block starts, so planes / winners / masks are bit-identical to
    the single-GPU grid at poses_per_batch = 2 - and the rank-major concatenation of the plane tables, sorted stably by
    pose, is the single-GPU table row for row.  The emulated ranks run twice: with the dense pose ranks (sort-free batch
    layout) and with the ranks shifted by 2048, a whole number of batches of at least REFSTART_MAX_RANKS (sorted layout)."""
    from octreelib_b200.parallel import pose_starts
    from octreelib_b200.ransac import CudaRansac

    world, P, ppb = 3, 5, 2
    clouds = {p: lidar64_scan(p, seed=7)[::8] for p in range(P)}
    ref = Grid(GridConfig(voxel_edge_length=1.0))
    for p in range(P):
        ref.insert_points(p, clouds[p])
    ref.subdivide([MaxPoints(40)])
    np.random.seed(9)
    table = CudaRansac(0.02, 128, 6).random_hypotheses
    ref._host.forest.ransac(table, 0.02, list(range(P)), ppb, apply=False)
    want = ref._host.forest.export_ransac(scored_only=True)
    want_leaves = ref._host.forest.export_leaves()
    # slab boundaries from the true quantiles of ix
    ix_all = np.concatenate([np.floor_divide(c[:, 0], 1.0).astype(np.int64) for c in clouds.values()])
    bounds = np.quantile(ix_all, [1 / 3, 2 / 3]).astype(np.int64)
    forests, sizes = [], np.zeros((world, P), dtype=np.int64)
    for r in range(world):
        f = Forest(1.0)
        seg_sizes, seg_pose, pts = [], [], []
        for p in range(P):
            own = np.searchsorted(bounds, np.floor_divide(clouds[p][:, 0], 1.0).astype(np.int64), side="right") == r
            if own.any():
                pts.append(clouds[p][own])
                seg_sizes.append(int(own.sum()))
                seg_pose.append(p)
        f.insert_segments(np.vstack(pts), seg_sizes, seg_pose, [0] * len(seg_sizes), P)
        f.subdivide(40)
        sizes[r] = f.pose_point_counts(P)
        forests.append(f)
    assert (sizes.sum(axis=0) == [len(clouds[p]) for p in range(P)]).all()
    for rank_offset in (0, 2048):
        rows = []
        leaf_base = 0
        for r, f in enumerate(forests):
            f.ransac(table, 0.02, [p + rank_offset for p in range(P)], ppb, apply=False, pose_start=pose_starts(sizes, r, ppb))
            got = f.export_ransac(scored_only=True)
            lv = f.export_leaves()
            for i in range(len(got["best"])):
                rows.append((int(got["pose"][i]), r, i, tuple(lv["corner"][got["leaf"][i]]), float(lv["edge"][got["leaf"][i]]),
                             int(got["best"][i]), int(got["best_count"][i]), got["plane"][i].tobytes()))
            leaf_base += len(lv["edge"])
        rows.sort(key=lambda t: (t[0], t[1], t[2]))  # stable by pose over the rank-major concatenation
        assert len(rows) == len(want["best"]), rank_offset
        for i, row in enumerate(rows):
            assert row[0] == want["pose"][i] and row[3] == tuple(want_leaves["corner"][want["leaf"][i]]), rank_offset
            assert row[5] == want["best"][i] and row[6] == want["best_count"][i] and row[7] == want["plane"][i].tobytes(), rank_offset


def test_partition_by_owner_matches_host_rule():
    lib = N.lib()
    rng = np.random.default_rng(0)
    clouds = [(rng.random((3000 + 500 * k, 3)) * 20 - 10).astype(np.float32).astype(np.float64) for k in range(3)]
    world = 4
    send, counts = _partition(clouds, 1.0, world)
    allpts = np.vstack(clouds)
    q = np.floor_divide(allpts, 1.0).astype(np.int64)
    owner = np.array([lib.ol_host_cell_owner(int(a), int(b), int(c), world) for a, b, c in q])
    run = np.concatenate([np.full(len(c), j) for j, c in enumerate(clouds)])
    order = np.lexsort((np.arange(len(allpts)), run, owner))
    assert (send == allpts[order]).all()
    exp = np.zeros_like(counts)
    np.add.at(exp, (owner, run), 1)
    assert (counts == exp).all()


def test_emulated_two_rank_grid_equals_single_gpu_grid():
    """Two 'ranks' (processed one after the other on one GPU) each hold half of the poses; after the
    routing every cell lives on exactly one rank and the union of the per-rank leaf tables and leaf
    point sets equals the single-GPU grid's."""
    world, P = 2, 4
    clouds = {p: lidar64_scan(p, seed=3)[::12] for p in range(P)}
    held = {r: [p for p in range(P) if p % world == r] for r in range(world)}  # non-monotone arrival order
    sends, counts = {}, {}
    for r in range(world):
        s, c = _partition([clouds[p] for p in held[r]], 1.0, world)
        sends[r], counts[r] = s, routing_layout(c, held[r], P)
    ref = Grid(GridConfig(voxel_edge_length=1.0))
    for p in range(P):
        ref.insert_points(p, clouds[p])
    ref.subdivide([MaxPoints(50)])
    ref_leaves = ref._host.forest.export_leaves()
    ref_blocks = ref._host.forest.export_blocks()
    ref_pts = ref._host.forest.export_points(-1, order=0)["xyz"]
    ref_keys = set()
    off = 0
    for pose, leaf, size in zip(ref_blocks["pose"], ref_blocks["leaf"], ref_blocks["size"]):
        key = (int(pose), tuple(ref_leaves["corner"][leaf]), float(ref_leaves["edge"][leaf]), ref_pts[off:off + size].tobytes())
        ref_keys.add(key)
        off += size
    got_keys = set()
    total_leaves = 0
    for dst in range(world):
        # what rank dst receives: from src 0 its slice, then from src 1 its slice
        parts, rc = [], np.zeros((world, P), dtype=np.int64)
        for src in range(world):
            start = int(counts[src][:dst].sum())
            n = int(counts[src][dst].sum())
            parts.append(sends[src][start:start + n])
            rc[src] = counts[src][dst]
        recv = np.vstack(parts)
        sizes, poses, first = segments_from_counts(rc)
        f = Forest(1.0)
        f.insert_segments(recv, sizes, poses, first, P)
        f.subdivide(50)
        lv, bl = f.export_leaves(), f.export_blocks()
        pts = f.export_points(-1, order=0)["xyz"]
        off = 0
        for pose, leaf, size in zip(bl["pose"], bl["leaf"], bl["size"]):
            got_keys.add((int(pose), tuple(lv["corner"][leaf]), float(lv["edge"][leaf]), pts[off:off + size].tobytes()))
            off += size
        total_leaves += f.stats()["n_leaves"]
    assert got_keys == ref_keys
    assert total_leaves == ref._host.forest.stats()["n_leaves"]


def test_append_to_existing_pose_in_a_manager():
    from octreelib_b200.octree import Octree, OctreeConfig
    from octreelib_b200.octree_manager import OctreeManager
    from oracle.structure import OracleGrid, max_points_criterion

    rng = np.random.default_rng(1)
    a = (rng.random((300, 3)) * 8).astype(np.float32).astype(np.float64)
    b = (rng.random((200, 3)) * 8).astype(np.float32).astype(np.float64)
    c = (rng.random((250, 3)) * 8).astype(np.float32).astype(np.float64)
    mp = OctreeManager(Octree, OctreeConfig(), np.array([0, 0, 0]), 8)
    mp.insert_points(0, a)
    mp.insert_points(1, b)
    mp.insert_points(0, c)  # appended to pose 0 (octree_manager.py:161-171)
    mp.subdivide([lambda pts: len(pts) > 20])
    og = OracleGrid(8)
    og.insert_points(0, np.vstack([a, c]))
    og.insert_points(1, b)
    og.subdivide([max_points_criterion(20)])
    for p in (0, 1):
        want = og.get_leaf_points(p)
        got = mp.get_leaf_points(pose_number=p)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert (np.asarray(g.corner_min, dtype=float) == np.asarray(w.corner, dtype=float)).all()
            assert (g.get_points() == w.points).all()
        assert mp.n_nodes(p) == og.n_nodes(p) and mp.n_points(p) == og.n_points(p)


def test_fused_exchange_world1_equals_plain_grid(monkeypatch):
    """The fused exchange (csrc/exchange.cu: count pass, scatter pass, adopted receive buffer, cell range without a bounding
    box pass) with a single rank must reproduce a plain Grid: same blocks, same points in the same order, same planes, same
    counters - and so must the staged exchange it falls back to when `_FusedExchange.disabled_reason` is set.  Clouds are
    staged out of pose order and one pose arrives in two pieces."""
    import torch

    from octreelib_b200.parallel import ShardedGrid, _FusedExchange

    P = 5
    clouds = {p: lidar64_scan(p, seed=3)[::4] for p in range(P)}
    dev = torch.device("cuda", 0)
    for reason in (None, "RuntimeError: no symmetric memory"):  # the fused exchange, then the staged fallback
        with monkeypatch.context() as m:
            if reason is not None:
                m.setattr(_FusedExchange, "disabled_reason", reason)
            for partition in ("slab", "hash"):
                # the fused receive buffers alternate: the third grid reuses the first one's
                for repeat in range(3 if reason is None else 1):
                    g = ShardedGrid(GridConfig(voxel_edge_length=1.0), P, partition=partition)
                    for p in (3, 0, 4, 1):
                        g.insert_points(p, torch.from_numpy(clouds[p]).to(dev) if p % 2 else clouds[p])
                    half = len(clouds[2]) // 2
                    g.insert_points(2, clouds[2][:half])
                    g.insert_points(2, clouds[2][half:])
                    g.exchange()
                    assert g.last_exchange["mode"] == "local" and g.last_exchange["received"] == sum(len(c) for c in clouds.values())
                    assert g.last_exchange["disabled_reason"] == reason
                    g.subdivide([MaxPoints(50)])
                    ref = Grid(GridConfig(voxel_edge_length=1.0))
                    for p in range(P):
                        ref.insert_points(p, clouds[p])
                    ref.subdivide([MaxPoints(50)])
                    f_a, f_b = g._host.forest, ref._host.forest
                    la, lb = f_a.export_leaves(), f_b.export_leaves()
                    assert (la["corner"] == lb["corner"]).all() and (la["edge"] == lb["edge"]).all()
                    ba, bb = f_a.export_blocks(list(range(P))), f_b.export_blocks(list(range(P)))
                    for k in ("pose", "leaf", "size"):
                        assert (ba[k] == bb[k]).all()
                    pa = f_a.export_points(-1, order=0, pose_rank=list(range(P)))
                    pb = f_b.export_points(-1, order=0, pose_rank=list(range(P)))
                    assert (pa["xyz"] == pb["xyz"]).all() and (pa["idx"] == pb["idx"]).all()
                    np.random.seed(11)
                    g.map_leaf_points_cuda_ransac(poses_per_batch=2, threshold=0.02, hypotheses_number=128)
                    np.random.seed(11)
                    ref.map_leaf_points_cuda_ransac(poses_per_batch=2, threshold=0.02, hypotheses_number=128)
                    ra, rb = g._host.forest.export_ransac(scored_only=True), ref._host.forest.export_ransac(scored_only=True)
                    for k in ("pose", "leaf", "size", "best", "best_count"):
                        assert (ra[k] == rb[k]).all()
                    assert (ra["plane"].view(np.uint32) == rb["plane"].view(np.uint32)).all()
                    assert [g.n_points(p) for p in range(P)] == [ref.n_points(p) for p in range(P)]
                    if repeat == 0:
                        keep = g  # stays alive across the next two exchanges: must be told to copy its points out
            if reason is None:
                assert [keep.n_points(p) for p in range(P)] == [ref.n_points(p) for p in range(P)]
                pk = keep._host.forest.export_points(-1, order=0, pose_rank=list(range(P)))
                pr = ref._host.forest.export_points(-1, order=0, pose_rank=list(range(P)))
                assert (pk["xyz"] == pr["xyz"]).all()


def test_fused_exchange_rejects_nonfinite(monkeypatch):
    """Non-finite coordinates are rejected by the fused exchange and by the staged fallback alike."""
    from octreelib_b200.parallel import ShardedGrid, _FusedExchange

    for reason in (None, "RuntimeError: no symmetric memory"):  # the fused exchange, then the staged fallback
        with monkeypatch.context() as m:
            if reason is not None:
                m.setattr(_FusedExchange, "disabled_reason", reason)
            g = ShardedGrid(GridConfig(voxel_edge_length=1.0), 1)
            pts = np.random.default_rng(0).normal(0, 3, (1000, 3))
            pts[17, 1] = np.nan
            g.insert_points(0, pts)
            with pytest.raises(ValueError, match="NaN or infinite"):
                g.exchange()
