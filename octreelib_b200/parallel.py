"""
Multi-GPU grid (SURVEY.md 8(e)): one process per GPU, `torch.distributed` (NCCL over NVLink) as the
plumbing.  Every grid cell is independent in the reference (`Grid.subdivide` / `filter` loop over
cells, grid/grid.py:255-258, 266-267; the scheme octree is per cell, octree_manager.py:50-66; RANSAC
is per (pose, leaf) block, cuda_ransac.py:94-97), so the grid shards by CELL, by a function of the cell key:

    partition="slab" (default)  owner(cell) = #{k : bound[k] <= ix}: an ORDER-PRESERVING hash of the cell key.  The
                                world - 1 boundaries are count quantiles of the leading cell coordinate over all ranks
                                (a sample histogram per rank), so the load is balanced, and because the reference
                                enumerates cells lexicographically (grid/grid.py:79-81) every cell of rank r precedes every
                                cell of rank r + 1.  That makes the two things that depend on the GLOBAL order exact: the
                                batch layout of the RANSAC kernel (`block_start_indices`, cuda_ransac.py:65-67: the sample
                                index is computed on the batch-global start) and the final leaf / plane tables
                                (`gather_tables`: rank-major concatenation = the reference's order).
    partition="hash"            owner(cell) = hash(ix, iy, iz) mod world (csrc/partition.cu, `ol_host_cell_owner`): the
                                layout north_star names; balanced whatever the geometry, but the global order - and with
                                it the sample index where `R n + start` sits within an ulp of an integer (p ~ 1e-8 per
                                draw) - would need a merge of all (cell, pose) tables.

`ShardedGrid.insert_points` stages a rank's local clouds; `exchange()` moves every point to the rank that owns its cell.
On one rank, or in an NCCL group whose ranks map each other's memory (torch symmetric memory), that is the fused exchange
of csrc/exchange.cu (`_FusedExchange`): owner rule, counting and peer stores over NVLink in one native call, after which
the receiving forest adopts the receive buffer.  Elsewhere - another backend, or no symmetric memory - the staged exchange
runs: `ol_partition_by_owner` (owner kernel + stable radix sort + gather), ONE all-to-all (counts first), and insertion of
what arrived as (source rank, pose) runs.  After that every operation is local to the rank - there is no further
data-path collective; only scalar counters and the final leaf / plane tables are reduced or gathered.

The routing helpers (`routing_layout`, `exchange_points`) are device independent so that the host
logic is covered by world_size-2 `gloo` tests on CPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N
from ._host import ForestHost
from .forest import TorchAllocator, require_cuda

__all__ = ["ShardedGrid", "routing_layout", "exchange_points", "segments_from_counts", "slab_boundaries", "pose_starts"]

SLAB_BINS = 1024


def slab_boundaries(gathered: np.ndarray, world: int) -> np.ndarray:
    """world - 1 ascending cell-x boundaries (owner = number of boundaries <= ix) that split the points of all ranks
    into equal shares.  gathered[r] = [min ix, max ix, counts of SLAB_BINS equal-width bins over that range] as written
    by `ol_slab_histogram` on rank r (min > max: the rank holds nothing).  Every rank computes the same answer from the
    same gathered array.  The bins are spread uniformly over their cells, which is exact for bins one cell wide."""
    g = np.asarray(gathered, dtype=np.int64)
    have = g[:, 0] <= g[:, 1]
    if not have.any() or world <= 1:
        return np.zeros(max(world - 1, 0), dtype=np.int64)
    lo, hi = int(g[have, 0].min()), int(g[have, 1].max())
    n_bins = g.shape[1] - 2
    # cumulative count at candidate boundaries: resolution = the finest rank bin width, at most 1 << 16 candidates
    span = hi - lo + 1
    step = max(1, -(-span // (1 << 16)))
    edges = lo + step * np.arange(-(-span // step) + 1, dtype=np.int64)  # candidate boundaries lo, lo + step, ...
    cum = np.zeros(len(edges), dtype=np.float64)
    for r in np.flatnonzero(have):
        rlo, rhi = int(g[r, 0]), int(g[r, 1])
        width = max(1, -(-(rhi - rlo + 1) // n_bins))
        c = np.concatenate([[0], np.cumsum(g[r, 2:], dtype=np.float64)])  # points of rank r with ix < rlo + k * width
        pos = (edges - rlo) / width
        cum += np.interp(pos, np.arange(n_bins + 1, dtype=np.float64), c)
    total = cum[-1]
    targets = total * np.arange(1, world, dtype=np.float64) / world
    idx = np.searchsorted(cum, targets, side="left")
    return edges[np.minimum(idx, len(edges) - 1)].astype(np.int64)


def pose_starts(pose_sizes: np.ndarray, rank: int, poses_per_batch: int) -> np.ndarray:
    """pose_sizes[r][p] = points of pose p held by rank r (slab partition: rank-major = the reference's cell order).
    Returns, per pose, the index inside its batch of `poses_per_batch` consecutive poses (grid.py:149-157) of the first
    point of that pose held by `rank`: points of the batch's earlier poses on all ranks + points of the pose on the
    lower ranks (cuda_ransac.py:65-67: block_start_indices is an exclusive cumulative sum over the batch)."""
    sizes = np.asarray(pose_sizes, dtype=np.int64)
    total = sizes.sum(axis=0)
    P = sizes.shape[1]
    excl = np.cumsum(total) - total                                  # points of all earlier poses
    batch_first = (np.arange(P) // poses_per_batch) * poses_per_batch
    before = excl - excl[batch_first]                                # ... of the earlier poses of the same batch
    return before + sizes[:rank].sum(axis=0)


def routing_layout(counts_local: np.ndarray, pose_numbers: Sequence[int], n_poses_total: int) -> np.ndarray:
    """counts_local[owner][local run] -> counts_global[owner][pose number] (runs of one pose add up)."""
    world = counts_local.shape[0]
    out = np.zeros((world, n_poses_total), dtype=np.int64)
    if len(pose_numbers):
        np.add.at(out, (slice(None), np.asarray(pose_numbers, dtype=np.int64)), counts_local[:, :len(pose_numbers)])
    return out


def exchange_points(send, send_counts: np.ndarray, group=None):
    """One all-to-all of point records.

    send: (n, 3) float64 tensor grouped by destination rank (then by pose); send_counts[dst][pose].
    Returns (recv tensor, recv_counts[src][pose]).  Works with any torch.distributed backend.
    """
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    dev = send.device
    sc = torch.from_numpy(np.ascontiguousarray(send_counts, dtype=np.int64)).to(dev)
    rc = torch.empty_like(sc)
    dist.all_to_all_single(rc, sc, group=group)  # row r of rc = what rank r sends to me, per pose
    recv_counts = rc.cpu().numpy()
    in_splits = [int(v) * 3 for v in recv_counts.sum(axis=1)]
    out_splits = [int(v) * 3 for v in send_counts.sum(axis=1)]
    recv = torch.empty((sum(in_splits) // 3, 3), dtype=send.dtype, device=dev)
    dist.all_to_all_single(recv.view(-1), send.reshape(-1), output_split_sizes=in_splits, input_split_sizes=out_splits,
                           group=group)
    assert len(in_splits) == world
    return recv, recv_counts


def segments_from_counts(recv_counts: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(source rank, pose) runs of the received buffer: sizes, pose numbers, and the index of each
    run's first point among the points of that pose received so far (keeps the original input order
    of a pose when its source ranks hold increasing index ranges)."""
    rc = np.asarray(recv_counts, dtype=np.int64)
    # index of a run's first point inside its pose = points of that pose received from lower source ranks
    before = np.cumsum(rc, axis=0) - rc
    src, pose = np.nonzero(rc)  # row-major: source rank, then pose -> the order of the received buffer
    return rc[src, pose].astype(np.int64), pose.astype(np.int32), before[src, pose].astype(np.int64)


class _FusedExchange:
    """Everything `ol_exchange_run` (csrc/exchange.cu) needs of one (group, world, pose count): the peer-mapped control
    blocks and receive buffers (torch.distributed._symmetric_memory; plain device tensors when world == 1) and the native
    exchange object.  Two receive buffers alternate, so the forest of one step may still be alive while the next step's
    exchange runs; a forest that outlives TWO exchanges is made to copy its points out first (`disown_points`)."""

    NBUF = 2
    _cache: Dict[Tuple[int, int, int], "_FusedExchange"] = {}
    disabled_reason: Optional[str] = None

    def __init__(self, world: int, rank: int, n_poses: int, rows_cap: int, device, group):
        import torch

        lib = N.lib()
        self.world, self.rank, self.n_poses, self.rows_cap = world, rank, n_poses, int(rows_cap)
        ctrl_words = int(lib.ol_exchange_ctrl_bytes(world, n_poses)) // 8 + 1
        if world > 1:
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm

            g = group if group is not None else dist.group.WORLD
            self.ctrl = symm.empty(ctrl_words, dtype=torch.int64, device=device)
            self.ctrl.zero_()
            hdl = symm.rendezvous(self.ctrl, g)
            ctrl_ptrs = [int(p) for p in hdl.buffer_ptrs]
            self.bufs, data_ptrs = [], []
            for _ in range(self.NBUF):
                t = symm.empty(max(self.rows_cap, 1) * 3, dtype=torch.float64, device=device)
                h = symm.rendezvous(t, g)
                self.bufs.append(t)
                data_ptrs += [int(p) for p in h.buffer_ptrs]
            torch.cuda.synchronize(device)
            hdl.barrier()  # every rank's flags are zero before anybody raises one
            torch.cuda.synchronize(device)
            self._hdl = hdl
        else:
            self.ctrl = torch.zeros(ctrl_words, dtype=torch.int64, device=device)
            self.bufs = [torch.empty(max(self.rows_cap, 1) * 3, dtype=torch.float64, device=device) for _ in range(self.NBUF)]
            ctrl_ptrs = [self.ctrl.data_ptr()]
            data_ptrs = [t.data_ptr() for t in self.bufs]
            torch.cuda.synchronize(device)
        self._h = C.c_void_p()
        N.check(lib.ol_exchange_create(world, rank, n_poses, self.rows_cap, self.NBUF, (C.c_void_p * world)(*ctrl_ptrs),
                                       (C.c_void_p * (self.NBUF * world))(*data_ptrs), device.index, C.byref(self._h)))
        self._next = 0
        self._holder = [None] * self.NBUF  # weak reference to the forest that adopted the buffer

    def __del__(self):
        try:
            if self._h:
                N.lib().ol_exchange_destroy(self._h)
                self._h = None
        except Exception:  # noqa: BLE001
            pass

    @classmethod
    def get(cls, world: int, rank: int, n_poses: int, n_local: int, device, group, dist, min_rows: int = 0) -> "_FusedExchange":
        """Collective.  Sized on first use from the total point count (one all-reduce): 1.25 x the mean share."""
        key = (id(group), world, n_poses)
        xc = cls._cache.get(key)
        if xc is not None and xc.rows_cap >= min_rows:
            return xc
        import torch

        total = n_local
        if world > 1:
            t = torch.tensor([n_local], dtype=torch.int64, device=device)
            dist.all_reduce(t, group=group)
            total = int(t.item())
        rows = max(int(1.25 * -(-total // world)) + 65536, int(1.25 * min_rows))
        cls._cache.pop(key, None)
        xc = cls(world, rank, n_poses, rows, device, group)
        cls._cache[key] = xc
        return xc

    def run(self, forest, tensors, numbers, slabs: bool):
        """Routes `tensors` (device float64 (n, 3), pose numbers ascending) and lets `forest` adopt what arrives.
        Returns (info[4], slab bounds, pose sizes [world][n_poses])."""
        import weakref

        lib = N.lib()
        b = self._next
        self._next = (b + 1) % self.NBUF
        prev = self._holder[b]() if self._holder[b] is not None else None
        if prev is not None and prev is not forest:
            prev.disown_points()  # still alive after two exchanges: it gets its own copy, the buffer is reused
        count = len(tensors)
        ptrs = (C.c_void_p * max(count, 1))(*[t.data_ptr() for t in tensors])
        sizes = (C.c_int64 * max(count, 1))(*[t.shape[0] for t in tensors])
        poses = (C.c_int32 * max(count, 1))(*numbers)
        info = np.zeros(4, dtype=np.int64)
        bounds = np.zeros(max(self.world - 1, 1), dtype=np.int64)
        psz = np.zeros((self.world, self.n_poses), dtype=np.uint32)
        self.last_info = info
        forest.adopt_exchange(self, self._h, ptrs, sizes, poses, count, 1 if slabs else 0, b, info, bounds, psz)
        self._holder[b] = weakref.ref(forest)
        return info, bounds[: self.world - 1], psz


class ShardedGrid:
    """The `Grid` operations of the hot path on a cell-sharded grid.  Pose numbers must be 0..P-1."""

    _identity_tables: Dict[int, tuple] = {}

    def __init__(self, grid_config, n_poses_total: int, group=None, partition: str = "slab"):
        import torch.distributed as dist

        if partition not in ("slab", "hash"):
            raise ValueError("partition must be 'slab' or 'hash'")
        self.partition = partition
        self.slab_bounds: Optional[np.ndarray] = None
        self._cfg = grid_config
        self._group = group
        self._dist = dist
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.n_poses_total = int(n_poses_total)
        corner = np.asarray(grid_config.corner, dtype=np.float64).reshape(3)
        self._corner = corner
        self._host = ForestHost(grid_config.voxel_edge_length, corner, single_cell=False)
        # the local forest knows every pose number (index == number)
        P = self.n_poses_total
        cached = ShardedGrid._identity_tables.get(P)
        if cached is None:
            cached = ShardedGrid._identity_tables[P] = (list(range(P)), {p: p for p in range(P)})
        self._host.pose_numbers = cached[0].copy()
        self._host.pose_index = cached[1].copy()
        self._host.pose_inserted = [0] * P
        self._staged: List[Tuple[int, object]] = []
        self.exchanged = False
        self.last_exchange = None
        self._pose_sizes: Optional[np.ndarray] = None  # [rank][pose] rows held after the exchange (fused path)
        self._removed = False                          # a filter / mask has removed points since

    # ---- staging + routing ----------------------------------------------------------------------
    def insert_points(self, pose_number: int, points):
        if not 0 <= pose_number < self.n_poses_total:
            raise KeyError(pose_number)
        if self.exchanged:
            raise RuntimeError("insert after exchange() is not supported")
        self._staged.append((int(pose_number), points))

    def exchange(self):
        """Route every staged point to the rank that owns its cell.  The fused exchange runs wherever it can: on a single
        rank, or in an NCCL group whose ranks map each other's memory.  Otherwise (another backend, or
        `_FusedExchange.disabled_reason` set because symmetric memory is unavailable) the staged all-to-all runs."""
        if any(a[0] > b[0] for a, b in zip(self._staged, self._staged[1:])):
            self._staged.sort(key=lambda s: s[0])  # stable: poses ascending, insertion order inside a pose
        dev = self._host.forest.device
        if (_FusedExchange.disabled_reason is None and not self.exchanged
                and (self.world == 1 or self._dist.get_backend(self._group) == "nccl")):
            if self._exchange_fused(dev):
                return
        self._exchange_staged(dev)

    def _exchange_fused(self, dev) -> bool:
        """The production path (csrc/exchange.cu): one native call, no library collective, one host wait.  Returns False
        when peer-mapped memory is not available (the caller falls back to `_exchange_staged`)."""
        torch = require_cuda()
        staged = self._staged
        numbers = [s[0] for s in staged]
        # the host time of this loop is time the GPU idles: one attribute test per cloud on the fast path
        tensors, f64, dev_index = [], torch.float64, dev.index
        for _, pts in staged:
            t = pts
            if not (type(t) is torch.Tensor and t.dtype is f64 and t.is_cuda and t.get_device() == dev_index and t.dim() == 2
                    and t.is_contiguous()):
                t = pts if isinstance(pts, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64))
                t = t.to(dev, dtype=torch.float64, non_blocking=True).contiguous().reshape(-1, 3)
            tensors.append(t)
        n_local = sum([t.shape[0] for t in tensors])
        forest = self._host.forest
        slabs = self.partition == "slab"
        min_rows = 0
        for _attempt in range(3):
            try:
                xc = _FusedExchange.get(self.world, self.rank, self.n_poses_total, n_local, dev, self._group, self._dist, min_rows)
            except Exception as exc:  # noqa: BLE001 - no symmetric memory on this system: the staged exchange still works
                _FusedExchange.disabled_reason = f"{type(exc).__name__}: {exc}"
                return False
            try:
                info, bounds, psz = xc.run(forest, tensors, numbers, slabs)
                break
            except N.ExchangeCapacityError:
                min_rows = int(xc.last_info[3])  # the same on every rank: everybody grows alike
        else:
            raise RuntimeError("exchange buffers could not be sized")
        if slabs and self.world > 1:
            self.slab_bounds = bounds.copy()
        self._pose_sizes = psz.astype(np.int64)
        self.last_exchange = dict(sent=int(info[0]), received=int(info[1]), kept=int(info[2]), mode="fused-p2p" if self.world > 1 else "local",
                                  partition=self.partition, disabled_reason=None, bytes=int(info[0]) * 24)
        self._staged = []
        self.exchanged = True
        return True

    def _exchange_staged(self, dev):
        """The fallback: an owner-grouped staging copy with counts on the host (`ol_partition_by_owner`), one all-to-all
        of any backend (`exchange_points`), and insertion of what arrived as (source rank, pose) runs."""
        torch = require_cuda()
        lib = N.lib()
        stream = torch.cuda.current_stream(dev)
        parts = []
        for _, pts in self._staged:
            t = pts if isinstance(pts, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64))
            parts.append(t.to(dev, dtype=torch.float64, non_blocking=True).reshape(-1, 3))
        numbers = [p for p, _ in self._staged]
        sizes = np.array([int(t.shape[0]) for t in parts] or [0], dtype=np.int64)
        local = torch.cat(parts) if parts else torch.empty((0, 3), dtype=torch.float64, device=dev)
        n, n_seg = int(local.shape[0]), max(len(parts), 1)
        bounds = None
        if self.partition == "slab" and self.world > 1:
            # count quantiles of the leading cell coordinate over all ranks: one small all-gather, one read-back
            hist = torch.empty(2 + SLAB_BINS, dtype=torch.int64, device=dev)
            N.check(lib.ol_slab_histogram(C.c_void_p(stream.cuda_stream), C.c_void_p(local.data_ptr()), n,
                                          float(self._cfg.voxel_edge_length), float(self._corner[0]), SLAB_BINS,
                                          C.c_void_p(hist.data_ptr())))
            allh = torch.empty((self.world, 2 + SLAB_BINS), dtype=torch.int64, device=dev)
            self._dist.all_gather_into_tensor(allh, hist, group=self._group)
            self.slab_bounds = slab_boundaries(allh.cpu().numpy(), self.world)
            bounds = np.ascontiguousarray(self.slab_bounds, dtype=np.int64)
        bounds_p = None if bounds is None else bounds.ctypes.data_as(C.c_void_p)
        send = torch.empty_like(local)
        counts = np.zeros((self.world, n_seg), dtype=np.int64)
        alloc = TorchAllocator(dev)
        corner = (C.c_double * 3)(*self._corner)
        N.check(lib.ol_partition_by_owner(C.c_void_p(stream.cuda_stream), C.c_void_p(local.data_ptr()), n,
                                          sizes.ctypes.data_as(C.c_void_p), n_seg, float(self._cfg.voxel_edge_length),
                                          C.byref(corner), self.world, bounds_p, C.c_void_p(send.data_ptr()),
                                          counts.ctypes.data_as(C.c_void_p), alloc.alloc_cb, alloc.free_cb, None))
        send_counts = routing_layout(counts[:, :len(parts)], numbers, self.n_poses_total)
        if self.world > 1:
            recv, recv_counts = exchange_points(send, send_counts, self._group)
        else:
            recv, recv_counts = send, send_counts
        seg_sizes, seg_pose, seg_first = segments_from_counts(recv_counts)
        if len(seg_sizes) == 0:
            seg_sizes, seg_pose, seg_first = np.array([0], np.int64), np.array([0], np.int32), np.array([0], np.int64)
        self._host.forest.insert_segments(recv, seg_sizes, seg_pose, seg_first, self.n_poses_total)
        sent, kept = int(send_counts.sum() - send_counts[self.rank].sum()), int(send_counts[self.rank].sum())
        self.last_exchange = dict(sent=sent, received=int(recv.shape[0]), kept=kept, mode="nccl" if self.world > 1 else "local",
                                  partition=self.partition, disabled_reason=_FusedExchange.disabled_reason,
                                  bytes=sent * 24)
        self._staged = []
        self.exchanged = True

    # ---- local pipeline -------------------------------------------------------------------------
    def subdivide(self, subdivision_criteria, pose_numbers: Optional[Sequence[int]] = None):
        self._require_exchanged()
        self._host.subdivide(subdivision_criteria, pose_numbers)

    def filter(self, filtering_criteria):
        self._require_exchanged()
        self._host.filter(filtering_criteria)
        self._removed = True

    def map_leaf_points_cuda_ransac(self, poses_per_batch: int = 10, threshold: float = 0.01, hypotheses_number: int = 1024,
                                    initial_points_number: int = 6):
        from .ransac.cuda_ransac import CudaRansac

        self._require_exchanged()
        if threshold <= 0:
            raise ValueError("Threshold must be positive")
        if hypotheses_number < 1:
            raise ValueError("Number of RANSAC hypotheses must be positive")
        if hypotheses_number > 1024:
            raise ValueError("Number of RANSAC hypotheses must be <= 1024 because of the CUDA thread limit.")
        # every rank draws the same table (same seed state is the caller's responsibility, as in the reference)
        ransac = CudaRansac(threshold=threshold, hypotheses_number=hypotheses_number, initial_points_number=initial_points_number)
        forest = self._host.forest
        start = None
        if self.world > 1 and self.partition == "slab" and self._pose_sizes is not None and not self._removed:
            # the fused exchange already told every rank how many rows of every pose every rank holds
            start = pose_starts(self._pose_sizes, self.rank, poses_per_batch)
        elif self.world > 1 and self.partition == "slab":
            # the reference's batch-global start index of every block (cuda_ransac.py:65-67) across the ranks: one
            # all-gather of the per-rank pose sizes (P integers per rank)
            import torch

            mine = torch.from_numpy(forest.pose_point_counts(self.n_poses_total)).to(forest.device)
            sizes = torch.empty((self.world, self.n_poses_total), dtype=torch.int64, device=forest.device)
            self._dist.all_gather_into_tensor(sizes, mine, group=self._group)
            start = pose_starts(sizes.cpu().numpy(), self.rank, poses_per_batch)
        forest.ransac(ransac.random_hypotheses, threshold, np.arange(self.n_poses_total, dtype=np.int32), poses_per_batch, apply=True,
                      pose_start=start)
        self._removed = True
        self._host._counts_cache = None

    def _require_exchanged(self):
        if not self.exchanged:
            self.exchange()

    # ---- global counters: sums over the ranks (cells are disjoint) --------------------------------
    def _global(self, which: int, pose_number: int) -> int:
        import torch

        local = self._host.count(pose_number, which)
        if self.world == 1:
            return local
        t = torch.tensor([local], dtype=torch.int64, device=self._host.forest.device)
        self._dist.all_reduce(t, group=self._group)
        return int(t.item())

    def n_leaves(self, pose_number: int) -> int:
        return self._global(0, pose_number)

    def n_points(self, pose_number: int) -> int:
        return self._global(1, pose_number)

    def n_nodes(self, pose_number: int) -> int:
        return self._global(2, pose_number)

    # ---- final gather of the leaf / plane tables ----------------------------------------------------
    def gather_tables(self, dst: int = 0) -> Optional[Dict[str, np.ndarray]]:
        """Leaf table (corner, edge, depth) and fitted-plane table of the whole grid on rank `dst`, in the REFERENCE's
        global order (slab partition): leaves = cells lexicographic x leaf order (grid.py:217-232) = the rank-major
        concatenation of the local tables; plane rows = (pose, then that leaf order), i.e. the rows of every rank sorted
        stably by pose.  `leaf` of a plane row indexes the gathered leaf table.  With partition="hash" the tables are
        concatenated by rank (no global order) and `rank_of_leaf` tells where a leaf lives."""
        forest = self._host.forest
        mine = dict(leaves=forest.export_leaves(), planes=forest.export_ransac(scored_only=True))
        if self.world == 1:
            return mine
        out = [None] * self.world if self.rank == dst else None
        self._dist.gather_object(mine, out, dst=dst, group=self._group)
        if self.rank != dst:
            return None
        n_leaves = [len(o["leaves"]["edge"]) for o in out]
        leaf_base = np.concatenate([[0], np.cumsum(n_leaves)])
        leaves = {k: np.concatenate([o["leaves"][k] for o in out]) for k in mine["leaves"]}
        planes = {k: np.concatenate([o["planes"][k] for o in out]) for k in mine["planes"]}
        planes["leaf"] = np.concatenate([o["planes"]["leaf"].astype(np.int64) + leaf_base[r] for r, o in enumerate(out)])
        rank_of_leaf = np.concatenate([np.full(n, r) for r, n in enumerate(n_leaves)])
        if self.partition == "slab":
            order = np.argsort(planes["pose"], kind="stable")  # rank-major inside a pose = lexicographic cells
            planes = {k: v[order] for k, v in planes.items()}
        return dict(leaves=leaves, planes=planes, rank_of_leaf=rank_of_leaf)
