"""
`Forest`: thin Python owner of one native `ol_forest` handle.

A forest is the device-resident state behind one `Grid` (many cells, many poses) or one
`OctreeManager` / `Octree` (a single fixed cell).  This class only moves arguments across the C
ABI, lends torch's caching allocator to the library (PyTorch tensors are used purely as device
buffers) and turns status codes into the exceptions the reference raises.  All arithmetic happens
in the CUDA library; nothing here falls back to the CPU.
"""
from __future__ import annotations

import contextlib
import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _native as N

__all__ = ["Forest", "TorchAllocator", "require_cuda", "release_cached_memory"]


_NULL_SCOPE = contextlib.nullcontext()


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError(
            "octreelib_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback for the grid pipeline")
    return torch


class TorchAllocator:
    """Device allocator callbacks backed by torch's caching allocator.

    The ctypes callbacks close over a plain dict, NOT over `self`: a bound-method callback would make
    allocator -> callback -> allocator a reference cycle, so a dropped Forest (gigabytes of device buffers) would
    only be released by Python's cyclic garbage collector, several steps later and all at once - measured as
    100-300 ms stalls (cudaMalloc of new multi-GB blocks while the dead forests still held theirs)."""

    _per_device: dict = {}

    def __new__(cls, device):
        # ONE allocator per device for the life of the process: the native library keeps released blocks in a process-wide
        # cache and hands them to the next forest (csrc/common.cuh, BlockCache), so the callbacks - and the tensors behind
        # the cached blocks - must outlive every single forest.  `release_cached_memory()` returns the blocks to torch.
        torch = require_cuda()
        device = torch.device(device)
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self = cls._per_device.get(device.index)
        if self is None:
            self = super().__new__(cls)
            self._setup(torch, device)
            cls._per_device[device.index] = self
        return self

    def _setup(self, torch, device):
        self.device = device
        live = {}
        self.live = live

        def _alloc(_user, nbytes):
            try:
                t = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
                ptr = t.data_ptr()
                live[ptr] = t
                return ptr
            except Exception:  # noqa: BLE001 - must not propagate through the C frame
                return None

        def _free(_user, ptr):
            live.pop(ptr, None)

        self.alloc_cb = N.ALLOC_FN(_alloc)
        self.free_cb = N.FREE_FN(_free)


def release_cached_memory() -> int:
    """Return the device blocks the native library caches between forests to torch's allocator (bytes released)."""
    return int(N.lib().ol_release_cached_memory())


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _i32_array(values: Optional[Sequence[int]]):
    if values is None:
        return None, 0
    arr = np.ascontiguousarray(values if isinstance(values, np.ndarray) else list(values), dtype=np.int32)
    return arr, len(arr)


class Forest:
    FLUSH_EVERY = 128           # deferred CUDA-tensor inserts are handed over in batches of this many poses ...
    FLUSH_MIN_ROWS = 1 << 20    # ... once they hold at least this many points (small grids: one batch at the end)

    def __init__(self, edge: float, corner=(0.0, 0.0, 0.0), single_cell: bool = False, max_depth: int = N.OL_MAX_DEPTH,
                 device=None):
        torch = require_cuda()
        self._lib = N.lib()
        self._torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._stream = torch.cuda.current_stream(self.device)
        self._raw_stream = self._stream.cuda_stream
        self._allocator = TorchAllocator(self.device)
        cfg = N.ForestConfig()
        cfg.voxel_edge_length = float(edge)
        cfg.corner = (C.c_double * 3)(*[float(v) for v in corner])
        cfg.single_cell = 1 if single_cell else 0
        cfg.max_depth = int(max_depth)
        cfg.device = self.device.index
        cfg.stream = C.c_void_p(self._stream.cuda_stream)
        cfg.alloc = self._allocator.alloc_cb
        cfg.free = self._allocator.free_cb
        cfg.alloc_user = None
        self._pending_sources = []  # sources of inserts that may still be in flight
        self._batch = []            # CUDA tensors whose insert is deferred (one native call for all of them)
        self._batch_rows = 0
        self._batch_sizes = []      # rows of every deferred tensor
        self.last_insert_rows = 0   # rows of the cloud handed to the last insert() call
        self._first_flush = max(self.FLUSH_EVERY // 4, 1)
        self._Tensor, self._f64 = torch.Tensor, torch.float64
        self._n_poses_native = 0    # poses the native forest knows about
        self._h = C.c_void_p()
        with self._scope():
            N.check(self._lib.ol_forest_create(C.byref(cfg), C.byref(self._h)))
        self.version = 0  # bumped by every mutating call; hosts cache exports per version
        self.extra_ransac_flags = 0  # OR-ed into every RANSAC launch (bench.py: OL_RANSAC_STATS for its profiled step)

    def _scope(self, flush: bool = True):
        """Context in which torch's current stream is the forest's stream (the allocator callbacks allocate
        on the current stream).  Entering torch.cuda.stream() costs ~12 us, so it is skipped when the
        caller already is on that stream - the common case.  Every native call except the batched insert itself
        first flushes the deferred CUDA-tensor inserts, so the native side always sees the poses in insertion order."""
        if flush and self._batch:
            self._flush()
        try:
            if self._torch._C._cuda_getCurrentRawStream(self.device.index) == self._raw_stream:
                return _NULL_SCOPE
        except AttributeError:  # private torch API moved: fall back to the public, slower path
            pass
        return self._torch.cuda.stream(self._stream)

    def close(self):
        self._batch = []
        self._batch_sizes = []
        if getattr(self, "_h", None) is not None and self._h:
            with self._scope():
                self._lib.ol_forest_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    # ---- mutation ------------------------------------------------------------------------------
    def insert(self, points) -> int:
        """Append one pose's cloud: numpy (n,3) array or a CUDA float64 tensor.  Returns pose index.

        CUDA tensors are not copied right away: they are collected (by reference) and handed to the native side in ONE
        call before the next grid operation (`ol_forest_insert_batch`: one growth of the point array, one copy kernel
        instead of a driver call per pose).  Do not modify such a tensor in place between `insert_points` and the next
        operation on the grid."""
        # (one call per pose of a map, 839 on the bench workload: every attribute access here is host time in front of the
        # first kernel - `t.device.type` alone costs as much as six of the tests below)
        if type(points) is self._Tensor and points.is_cuda:
            t = points
            shape = t.shape
            if t.dtype is not self._f64 or len(shape) != 2 or shape[1] != 3 or not t.is_contiguous():
                t = t.to(self._f64).contiguous().reshape(-1, 3)
                shape = t.shape
            rows = shape[0]
            self.last_insert_rows = rows
            batch = self._batch
            batch.append(t)
            self._batch_sizes.append(rows)
            self._batch_rows += rows
            self.version += 1
            index = self._n_poses_native + len(batch) - 1
            # (the FIRST batch goes out after a quarter of FLUSH_EVERY poses, so that the GPU starts early)
            if len(batch) >= (self.FLUSH_EVERY if self._n_poses_native else self._first_flush) and self._batch_rows >= self.FLUSH_MIN_ROWS:
                self._flush()  # the copy kernel runs while the caller is still inserting the following poses
            return index
        out = C.c_int32(-1)
        src, n, on_dev, keep = self._as_source(points)
        self.last_insert_rows = n
        with self._scope():
            N.check(self._lib.ol_forest_insert(self._h, src, n, on_dev, C.byref(out)))
        # a pinned host source is read asynchronously (csrc/forest_host.inl): keep it alive until the next synchronising call
        self._pending_sources.append(keep)
        self._n_poses_native += 1
        self.version += 1
        return out.value

    def _flush(self):
        """Hand the deferred CUDA-tensor inserts to the native forest (one call)."""
        batch, self._batch = self._batch, []
        rows, self._batch_sizes = self._batch_sizes, []
        self._batch_rows = 0
        if not batch:
            return
        count = len(batch)
        ptrs = (C.c_void_p * count)(*[t.data_ptr() for t in batch])
        sizes = (C.c_int64 * count)(*rows)
        first = C.c_int32(-1)
        with self._scope(flush=False):
            N.check(self._lib.ol_forest_insert_batch(self._h, ptrs, sizes, count, C.byref(first)))
        assert first.value == self._n_poses_native, (first.value, self._n_poses_native)
        self._n_poses_native += count

    def insert_segments(self, points, seg_sizes, seg_pose, seg_first, n_poses_total: int):
        src, n, on_dev, keep = self._as_source(points)
        ss = np.ascontiguousarray(seg_sizes, dtype=np.int64)
        sp = np.ascontiguousarray(seg_pose, dtype=np.int32)
        sf = np.ascontiguousarray(seg_first, dtype=np.int64)
        with self._scope():
            N.check(self._lib.ol_forest_insert_segments(self._h, src, n, on_dev, _ptr(ss), _ptr(sp), _ptr(sf), len(ss),
                                                        int(n_poses_total)))
        self._pending_sources.append(keep)
        self._n_poses_native = max(self._n_poses_native, int(n_poses_total))
        self.version += 1

    def adopt_exchange(self, exchange, handle, ptrs, sizes, poses, count, slabs, buffer, info, bounds, pose_sizes):
        """Collective multi-GPU exchange into this (empty) forest: parallel.py `_FusedExchange.run`.  The forest keeps the
        exchange object (and with it the receive buffer it adopted) alive."""
        with self._scope():
            N.check(self._lib.ol_exchange_run(handle, self._h, ptrs, sizes, poses, int(count), int(slabs), int(buffer),
                                              _ptr(info), _ptr(bounds), _ptr(pose_sizes)))
        self._adopted = exchange
        self._n_poses_native = max(self._n_poses_native, int(exchange.n_poses))
        self.version += 1

    def disown_points(self):
        """Copy an adopted receive buffer into memory of the forest's own (the exchange is about to reuse the buffer)."""
        if getattr(self, "_h", None) is not None and self._h:
            with self._scope():
                N.check(self._lib.ol_forest_disown_points(self._h))
        self._adopted = None

    def _as_source(self, points):
        torch = self._torch
        if isinstance(points, torch.Tensor):
            t = points
            if t.device.type != "cuda":
                return self._as_source(t.numpy())
            if t.dtype != torch.float64 or not t.is_contiguous():
                t = t.to(torch.float64).contiguous()
            if t.dim() != 2 or t.shape[1] != 3:
                t = t.reshape(-1, 3)
            return C.c_void_p(t.data_ptr()), t.shape[0], 1, t
        a = np.ascontiguousarray(np.asarray(points), dtype=np.float64)
        if a.size == 0:
            a = a.reshape(0, 3)
        if a.ndim != 2 or a.shape[1] != 3:
            raise ValueError(f"points must have shape (n, 3), got {a.shape}")
        return _ptr(a), a.shape[0], 0, a

    def subdivide(self, max_points: int, pose_indices: Optional[Sequence[int]] = None):
        arr, n = _i32_array(pose_indices)
        with self._scope():
            N.check(self._lib.ol_forest_subdivide(self._h, int(max_points), _ptr(arr), n))
        self._pending_sources.clear()  # the build read every inserted cloud and synchronised
        self.version += 1

    def subdivide_table(self, table: np.ndarray, beyond: bool, pose_indices: Optional[Sequence[int]] = None):
        arr, n = _i32_array(pose_indices)
        tab = np.ascontiguousarray(table, dtype=np.uint8)
        with self._scope():
            N.check(self._lib.ol_forest_subdivide_table(self._h, _ptr(tab), len(tab), 1 if beyond else 0, _ptr(arr), n))
        self.version += 1

    def subdivide_levels(self, first_levels: Sequence[int], thresholds: Optional[Sequence[int]] = None, tables=None,
                         beyonds: Optional[Sequence[bool]] = None, pose_indices: Optional[Sequence[int]] = None):
        """Level-dependent split rule (node-size thresholds, criteria.py): entry e applies from octree level
        first_levels[e] on.  Either `thresholds` (split iff count > thresholds[e]) or `tables` + `beyonds`."""
        arr, n = _i32_array(pose_indices)
        fl = np.ascontiguousarray(list(first_levels), dtype=np.int32)
        with self._scope():
            if tables is None:
                th = np.ascontiguousarray([min(int(t), 1 << 62) for t in thresholds], dtype=np.int64)
                N.check(self._lib.ol_forest_subdivide_levels(self._h, _ptr(fl), len(fl), _ptr(th), None, 0, None, _ptr(arr), n))
            else:
                tab = np.ascontiguousarray(np.stack([np.asarray(t, dtype=np.uint8) for t in tables]), dtype=np.uint8)
                by = np.ascontiguousarray([1 if b else 0 for b in beyonds], dtype=np.int32)
                N.check(self._lib.ol_forest_subdivide_levels(self._h, _ptr(fl), len(fl), None, _ptr(tab), tab.shape[1], _ptr(by),
                                                             _ptr(arr), n))
        self._pending_sources.clear()
        self.version += 1

    def subdivide_geometric(self, first_levels: Sequence[int], terms: Sequence[Sequence[tuple]],
                            thresholds: Optional[Sequence[int]] = None, tables=None, beyonds: Optional[Sequence[bool]] = None,
                            pose_indices: Optional[Sequence[int]] = None):
        """`subdivide_levels` whose entries also carry geometric terms (stat, op, min_points, value), OR-ed with the
        count rule: terms[e] belongs to the entry that starts at first_levels[e] (`ol_forest_subdivide_geometric`)."""
        arr, n = _i32_array(pose_indices)
        fl = np.ascontiguousarray(list(first_levels), dtype=np.int32)
        flat = [t for entry in terms for t in entry]
        term_arr = (N.GeomTerm * max(len(flat), 1))(*[N.GeomTerm(int(s), int(o), int(m), float(v)) for s, o, m, v in flat])
        counts = np.ascontiguousarray([len(entry) for entry in terms], dtype=np.int32)
        with self._scope():
            if tables is None:
                th = np.ascontiguousarray([min(int(t), 1 << 62) for t in thresholds], dtype=np.int64)
                N.check(self._lib.ol_forest_subdivide_geometric(self._h, _ptr(fl), len(fl), _ptr(th), None, 0, None, term_arr,
                                                                _ptr(counts), _ptr(arr), n))
            else:
                tab = np.ascontiguousarray(np.stack([np.asarray(t, dtype=np.uint8) for t in tables]), dtype=np.uint8)
                by = np.ascontiguousarray([1 if b else 0 for b in beyonds], dtype=np.int32)
                N.check(self._lib.ol_forest_subdivide_geometric(self._h, _ptr(fl), len(fl), None, _ptr(tab), tab.shape[1], _ptr(by),
                                                                term_arr, _ptr(counts), _ptr(arr), n))
        self._pending_sources.clear()
        self.version += 1

    def export_shape(self) -> dict:
        """The split nodes of the forest: cell coordinates, depth and Morton path (`ol_forest_export_shape`)."""
        n = C.c_int64(0)
        with self._scope():
            N.check(self._lib.ol_forest_export_shape(self._h, None, None, None, C.byref(n)))
        q = np.zeros((n.value, 3), dtype=np.int64)
        depth = np.zeros(n.value, dtype=np.uint32)
        path = np.zeros(n.value, dtype=np.uint64)
        if n.value:
            with self._scope():
                N.check(self._lib.ol_forest_export_shape(self._h, _ptr(q), _ptr(depth), _ptr(path), C.byref(n)))
        return dict(q=q, depth=depth, path=path)

    def impose_shape(self, shape: dict):
        """Make exactly the listed nodes the split nodes of this forest (`ol_forest_impose_shape`)."""
        q = np.ascontiguousarray(shape["q"], dtype=np.int64).reshape(-1, 3)
        depth = np.ascontiguousarray(shape["depth"], dtype=np.uint32)
        path = np.ascontiguousarray(shape["path"], dtype=np.uint64)
        with self._scope():
            N.check(self._lib.ol_forest_impose_shape(self._h, _ptr(q), _ptr(depth), _ptr(path), len(depth)))
        self.version += 1

    def filter(self, keep_table: np.ndarray, pose_indices: Optional[Sequence[int]] = None):
        arr, n = _i32_array(pose_indices)
        tab = np.ascontiguousarray(keep_table, dtype=np.uint8)
        with self._scope():
            N.check(self._lib.ol_forest_filter(self._h, _ptr(tab), len(tab), _ptr(arr), n))
        self.version += 1

    def filter_geometric(self, keep_table: np.ndarray, terms: Sequence[tuple], pose_indices: Optional[Sequence[int]] = None):
        """`filter` whose blocks must also satisfy every geometric term (stat, op, min_points, value)
        (`ol_forest_filter_geometric`)."""
        arr, n = _i32_array(pose_indices)
        tab = np.ascontiguousarray(keep_table, dtype=np.uint8)
        term_arr = (N.GeomTerm * max(len(terms), 1))(*[N.GeomTerm(int(s), int(o), int(m), float(v)) for s, o, m, v in terms])
        with self._scope():
            N.check(self._lib.ol_forest_filter_geometric(self._h, _ptr(tab), len(tab), term_arr, len(terms), _ptr(arr), n))
        self.version += 1

    def ransac(self, table: np.ndarray, threshold: float, pose_rank: Optional[Sequence[int]] = None,
               poses_per_batch: int = 10, apply: bool = True, flags: int = 0, pose_start=None):
        """pose_start: multi-GPU only - batch-global index of the first point of every pose index held by this forest
        (include/octreelib_b200.h, ol_forest_ransac)."""
        tab = np.ascontiguousarray(table, dtype=np.float64)
        H, K = tab.shape
        pr, _ = _i32_array(pose_rank)
        ps = None if pose_start is None else np.ascontiguousarray(pose_start, dtype=np.int64)
        with self._scope():
            N.check(self._lib.ol_forest_ransac(self._h, _ptr(tab), H, K, float(threshold), _ptr(pr), int(poses_per_batch),
                                               1 if apply else 0, int(flags) | int(self.extra_ransac_flags), _ptr(ps)))
        self.version += 1

    def pose_point_counts(self, n_poses: int) -> np.ndarray:
        out = np.zeros(max(n_poses, 1), dtype=np.int64)
        with self._scope():
            N.check(self._lib.ol_forest_pose_point_counts(self._h, _ptr(out)))
        return out[:n_poses]

    def apply_mask(self):
        with self._scope():
            N.check(self._lib.ol_forest_apply_mask(self._h))
        self.version += 1

    def apply_pose_mask(self, pose_index: int, mask):
        m = np.ascontiguousarray(np.asarray(mask).astype(bool), dtype=np.uint8)
        with self._scope():
            N.check(self._lib.ol_forest_apply_pose_mask(self._h, None, int(pose_index), _ptr(m), len(m)))
        self.version += 1

    # ---- measurement ---------------------------------------------------------------------------
    def profile(self, enable: bool = True):
        with self._scope():
            N.check(self._lib.ol_forest_profile(self._h, 1 if enable else 0))

    def profile_read(self) -> dict:
        """{stage: (launch groups, total ms, elements processed)} since the last read; synchronises."""
        buf = C.create_string_buffer(1 << 16)
        n = C.c_int64(0)
        with self._scope():
            N.check(self._lib.ol_forest_profile_read(self._h, buf, len(buf), C.byref(n)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, count, ms, units = line.split()
            out[name] = (int(count), float(ms), float(units))
        return out

    # ---- queries -------------------------------------------------------------------------------
    def _host_array(self, shape, dtype) -> np.ndarray:
        """Host destination of an export: page-locked (torch's caching host allocator) when large, so
        that the device-to-host copy runs at full PCIe speed; small tables use plain numpy memory."""
        n = int(np.prod(shape))
        if n * np.dtype(dtype).itemsize < (1 << 20):
            return np.zeros(shape, dtype=dtype)
        t = self._torch.empty(n * np.dtype(dtype).itemsize, dtype=self._torch.uint8, pin_memory=True)
        return t.numpy().view(dtype).reshape(shape)

    def stats(self, light: bool = False) -> dict:
        """Counters of the forest.  light=True builds no derived table (n_blocks / max_block_size are -1 when
        the block table is stale) and only waits for the enqueued work."""
        s = N.ForestStats()
        fn = self._lib.ol_forest_stats_light if light else self._lib.ol_forest_stats_get
        with self._scope():
            N.check(fn(self._h, C.byref(s)))
        self._pending_sources.clear()  # both variants synchronise the stream
        return {name: int(getattr(s, name)) for name, _ in s._fields_}

    def pose_counts(self, n_poses: int) -> np.ndarray:
        out = np.zeros((max(n_poses, 1), 3), dtype=np.int64)
        with self._scope():
            N.check(self._lib.ol_forest_pose_counts(self._h, _ptr(out)))
        return out[:n_poses]

    def export_cells(self) -> dict:
        st = self.stats()
        Cn = st["n_cells"]
        q = np.zeros((Cn, 3), dtype=np.int64)
        corner = np.zeros((Cn, 3), dtype=np.float64)
        first_pose = np.zeros(Cn, dtype=np.int32)
        n_nodes = np.zeros(Cn, dtype=np.int64)
        leaf_begin = np.zeros(Cn + 1, dtype=np.int64)
        with self._scope():
            N.check(self._lib.ol_forest_export_cells(self._h, _ptr(q), _ptr(corner), _ptr(first_pose), _ptr(n_nodes),
                                                     _ptr(leaf_begin)))
        return dict(q=q, corner=corner, first_pose=first_pose, n_nodes=n_nodes, leaf_begin=leaf_begin)

    def export_cell_poses(self) -> dict:
        st = self.stats()
        n = st["n_cell_poses"]
        cell = np.zeros(n, dtype=np.int32)
        pose = np.zeros(n, dtype=np.int32)
        with self._scope():
            N.check(self._lib.ol_forest_export_cell_poses(self._h, _ptr(cell), _ptr(pose)))
        return dict(cell=cell, pose=pose)

    def export_leaves(self) -> dict:
        st = self.stats(light=True)  # the leaf count needs no derived table (a full stats call rebuilds the block table)
        L = st["n_leaves"]
        corner = self._host_array((L, 3), np.float64)
        edge = self._host_array(L, np.float64)
        cell = self._host_array(L, np.int32)
        depth = self._host_array(L, np.int32)
        epoch = self._host_array(L, np.int32)
        with self._scope():
            N.check(self._lib.ol_forest_export_leaves(self._h, _ptr(corner), _ptr(edge), _ptr(cell), _ptr(depth), _ptr(epoch)))
        return dict(corner=corner, edge=edge, cell=cell, depth=depth, parent_epoch=epoch)

    def export_blocks(self, pose_rank: Optional[Sequence[int]] = None) -> dict:
        st = self.stats()
        B = st["n_blocks"]
        pose = np.zeros(B, dtype=np.int32)
        leaf = np.zeros(B, dtype=np.int32)
        size = np.zeros(B, dtype=np.int32)
        pr, _ = _i32_array(pose_rank)
        with self._scope():
            N.check(self._lib.ol_forest_export_blocks(self._h, _ptr(pr), _ptr(pose), _ptr(leaf), _ptr(size)))
        return dict(pose=pose, leaf=leaf, size=size)

    def export_block_stats(self, pose_index: int = -1, pose_rank: Optional[Sequence[int]] = None) -> dict:
        """Point statistics of the non-empty (pose, leaf) blocks in `export_blocks` order, of one pose or of all (-1):
        n, mean (B,3), cov (B,6: xx xy xz yy yz zz, population), extent (B,3) (`ol_forest_export_block_stats`)."""
        B = self.stats()["n_blocks"]
        pose = self._host_array(B, np.int32)
        n = self._host_array(B, np.int64)
        mean = self._host_array((B, 3), np.float64)
        cov = self._host_array((B, 6), np.float64)
        extent = self._host_array((B, 3), np.float64)
        pr, _ = _i32_array(pose_rank)
        rows = C.c_int64(0)
        with self._scope():
            N.check(self._lib.ol_forest_export_block_stats(self._h, _ptr(pr), int(pose_index), _ptr(pose), _ptr(n), _ptr(mean),
                                                           _ptr(cov), _ptr(extent), C.byref(rows)))
        k = rows.value
        return dict(pose=pose[:k], n=n[:k], mean=mean[:k], cov=cov[:k], extent=extent[:k])

    def export_ransac(self, scored_only: bool = False) -> dict:
        """Per-block result table of the last RANSAC run (reference block order)."""
        n = C.c_int64(0)
        so = 1 if scored_only else 0
        with self._scope():
            N.check(self._lib.ol_forest_export_ransac(self._h, so, None, None, None, None, None, None, C.byref(n)))
        B = n.value
        pose = self._host_array(B, np.int32)
        leaf = self._host_array(B, np.int32)
        size = self._host_array(B, np.int32)
        plane = self._host_array((B, 4), np.float32)
        best = self._host_array(B, np.int32)
        count = self._host_array(B, np.int32)
        with self._scope():
            N.check(self._lib.ol_forest_export_ransac(self._h, so, _ptr(pose), _ptr(leaf), _ptr(size), _ptr(plane), _ptr(best),
                                                      _ptr(count), C.byref(n)))
        return dict(pose=pose, leaf=leaf, size=size, plane=plane, best=best, best_count=count)

    def export_points(self, pose_index: int = -1, order: int = 0, pose_rank: Optional[Sequence[int]] = None,
                      n_hint: Optional[int] = None, want_mask: bool = False) -> dict:
        """order 0: reference block order; order 1: cells lexicographic x depth-first leaves."""
        if n_hint is None:
            n_hint = self.stats()["n_points_alive"]
        xyz = self._host_array((n_hint, 3), np.float64)
        idx = self._host_array(n_hint, np.int64)
        cell = self._host_array(n_hint, np.int32)
        mask = self._host_array(n_hint, np.uint8) if want_mask else None
        pr, _ = _i32_array(pose_rank)
        n = C.c_int64(0)
        with self._scope():
            N.check(self._lib.ol_forest_export_points(self._h, _ptr(pr), int(pose_index), int(order), _ptr(xyz), _ptr(idx),
                                                      _ptr(cell), _ptr(mask), C.byref(n)))
        k = n.value
        out = dict(xyz=xyz[:k], idx=idx[:k], cell=cell[:k])
        if want_mask:
            out["mask"] = mask[:k]
        return out
