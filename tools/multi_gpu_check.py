"""Multi-GPU correctness check (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/multi_gpu_check.py

Every rank holds a slice of the poses of a synthetic multi-pose LiDAR map.  The sharded pipeline (routing by cell owner
-> local subdivide -> local RANSAC) runs on both exchange paths - the fused peer-to-peer exchange, and the staged NCCL
all-to-all it falls back to when `_FusedExchange.disabled_reason` is set - each with the slab and the hash partition, and
rank 0 compares the union of the per-rank leaf / plane tables with a plain single-GPU Grid built from ALL poses: same
leaves (corner, edge), same (pose, leaf) blocks with the same points in the same order, same fitted planes (bit
patterns), same per-pose counters.  poses_per_batch = 10 (the reference's default, 3 batches here): the slab runs
reproduce the reference's batch-global block starts across the ranks, and their gathered tables (`gather_tables`)
equal the single-GPU tables row for row.
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from octreelib_b200.criteria import MaxPoints
from octreelib_b200.grid import Grid, GridConfig
from octreelib_b200.parallel import ShardedGrid, _FusedExchange
from octreelib_b200.synthetic import lidar64_scan

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
P, H, THR, PPB = 24, 256, 0.02, 10
clouds = {p: lidar64_scan(p, seed=1)[::3] for p in range(P)}
mine = [p for p in range(P) if p % world == rank]  # interleaved: the received runs are not pose-monotone


def block_table(forest, n_poses):
    leaves = forest.export_leaves()
    blocks = forest.export_blocks(list(range(n_poses)))
    pts = forest.export_points(-1, order=0, pose_rank=list(range(n_poses)))["xyz"]
    out, off = {}, 0
    for pose, leaf, size in zip(blocks["pose"], blocks["leaf"], blocks["size"]):
        key = (int(pose), tuple(leaves["corner"][leaf]), float(leaves["edge"][leaf]))
        out[key] = pts[off:off + size].tobytes()
        off += size
    return out


def plane_table(forest):
    leaves = forest.export_leaves()
    r = forest.export_ransac(scored_only=True)
    return {(int(p), tuple(leaves["corner"][l]), float(leaves["edge"][l])): (r["plane"][i].tobytes(), int(r["best"][i]), int(r["best_count"][i]))
            for i, (p, l) in enumerate(zip(r["pose"], r["leaf"]))}


def sharded(path, partition):
    g = ShardedGrid(GridConfig(voxel_edge_length=1.0), P, partition=partition)
    for p in mine:
        g.insert_points(p, clouds[p])
    saved = _FusedExchange.disabled_reason
    if path == "fallback":  # the same on every rank: all of them take the staged exchange
        _FusedExchange.disabled_reason = "fallback run of multi_gpu_check"
    try:
        g.exchange()
    finally:
        _FusedExchange.disabled_reason = saved
    g.subdivide([MaxPoints(60)])
    before = block_table(g._host.forest, P)
    np.random.seed(5)
    # hash partition: the batch-global start index cannot be reproduced across ranks, one batch makes it irrelevant
    g.map_leaf_points_cuda_ransac(poses_per_batch=PPB if partition == "slab" else P, threshold=THR, hypotheses_number=H)
    planes = plane_table(g._host.forest)
    after = block_table(g._host.forest, P)
    counts = [[g.n_leaves(p), g.n_points(p), g.n_nodes(p)] for p in range(P)]
    tables = g.gather_tables(0)
    gathered = [None] * world
    dist.gather_object(dict(before=before, planes=planes, after=after, exch=g.last_exchange), gathered if rank == 0 else None, dst=0)
    return gathered, counts, tables


results = {(path, part): sharded(path, part) for path, part in (("fused", "slab"), ("fused", "hash"), ("fallback", "slab"),
                                                                  ("fallback", "hash"))}
if rank == 0:
    def single(ppb):
        ref = Grid(GridConfig(voxel_edge_length=1.0))
        for p in range(P):
            ref.insert_points(p, clouds[p])
        ref.subdivide([MaxPoints(60)])
        before = block_table(ref._host.forest, P)
        leaves = ref._host.forest.export_leaves()
        np.random.seed(5)
        ref.map_leaf_points_cuda_ransac(poses_per_batch=ppb, threshold=THR, hypotheses_number=H)
        return dict(before=before, planes=plane_table(ref._host.forest), after=block_table(ref._host.forest, P),
                    counts=[[ref.n_leaves(p), ref.n_points(p), ref.n_nodes(p)] for p in range(P)], leaves=leaves,
                    table=ref._host.forest.export_ransac(scored_only=True))

    refs = {PPB: single(PPB), P: single(P)}
    for (path, part), (gathered, counts, tables) in results.items():
        ref = refs[PPB if part == "slab" else P]
        union_before, union_after, union_planes = {}, {}, {}
        for g in gathered:
            assert not (set(g["before"]) & set(union_before)), "a (pose, leaf) block lives on two ranks"
            union_before.update(g["before"])
            union_after.update(g["after"])
            union_planes.update(g["planes"])
        assert union_before == ref["before"], f"{path}/{part}: blocks after subdivide differ from the single-GPU grid"
        assert set(union_planes) == set(ref["planes"]), f"{path}/{part}: fitted block sets differ"
        assert union_planes == ref["planes"], f"{path}/{part}: planes differ"
        assert union_after == ref["after"], f"{path}/{part}: inlier sets differ"
        assert counts == ref["counts"], f"{path}/{part}: counters differ"
        if part == "slab":  # the gathered tables are the single-GPU tables, row for row
            assert (tables["leaves"]["corner"] == ref["leaves"]["corner"]).all() and (tables["leaves"]["edge"] == ref["leaves"]["edge"]).all()
            for k in ("pose", "leaf", "size", "best", "best_count"):
                assert (tables["planes"][k] == ref["table"][k]).all(), f"{path}/{part}: gathered plane table column {k} differs"
            assert (tables["planes"]["plane"].view(np.uint32) == ref["table"]["plane"].view(np.uint32)).all()
        sent = sum(g["exch"]["sent"] for g in gathered)
        mode = "fused-p2p" if path == "fused" else "nccl"
        assert all(g["exch"]["mode"] == mode for g in gathered), [g["exch"]["mode"] for g in gathered]
        print(f"[multi_gpu_check] world {world} exchange {path} ({mode}) partition {part}: OK - {len(ref['before'])} blocks, "
              f"{len(ref['planes'])} fitted planes, {sent} points crossed ranks, shares {[g['exch']['received'] for g in gathered]}; "
              f"fused exchange disabled reason: {gathered[0]['exch']['disabled_reason']}", flush=True)
dist.barrier()
dist.destroy_process_group()
