"""
CPU ORACLE (test infrastructure, NOT product code) -- RANSAC half, Python side.

* `ransac_evaluate`  : ctypes front-end of oracle/ransac_oracle.c (fast, pthreads).
* `ransac_numpy`     : an independent numpy restatement of the same kernel
                       (/root/reference/octreelib/ransac/cuda_ransac.py:85-155, util.py:16-84),
                       used to cross-check the C version on small inputs.
* `make_table`       : the hypothesis table exactly as the reference draws it
                       (cuda_ransac.py:39-41: `np.random.random((min(H,1024), K))` from the
                       GLOBAL numpy RNG; seed it with `np.random.seed(s)` right before).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libransac_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile oracle/ransac_oracle.c with gcc (see oracle/Makefile).  In a read-only tree (bench.py may run from
    one) a stale or missing library is compiled into a temporary directory instead of oracle/_build."""
    global _LIB_PATH
    src = os.path.join(_HERE, "ransac_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        if os.access(_HERE, os.W_OK):
            subprocess.check_call(["make", "-s", "-C", _HERE, "-B"])
        else:
            out = tempfile.mkdtemp(prefix="ol_oracle_")
            subprocess.check_call(["make", "-s", "-C", _HERE, "-B", f"BUILD={out}"])
            _LIB_PATH = os.path.join(out, "libransac_oracle.so")
    return _LIB_PATH


def _load():
    global _lib
    if _lib is None:
        build()
        lib = ctypes.CDLL(_LIB_PATH)
        c = ctypes
        lib.ol_oracle_ransac.restype = c.c_int64
        lib.ol_oracle_ransac.argtypes = [c.c_void_p, c.c_int64, c.c_void_p, c.c_void_p, c.c_int64, c.c_void_p,
                                         c.c_int, c.c_int, c.c_double, c.c_void_p, c.c_void_p, c.c_void_p,
                                         c.c_void_p, c.c_void_p, c.c_void_p, c.c_int]
        lib.ol_oracle_mask_for_plane.restype = None
        lib.ol_oracle_mask_for_plane.argtypes = [c.c_void_p, c.c_int64, c.c_int32, c.c_void_p, c.c_double,
                                                 c.c_void_p]
        _lib = lib
    return _lib


def make_table(hypotheses_number: int = 1024, initial_points_number: int = 6, seed=None) -> np.ndarray:
    if seed is not None:
        np.random.seed(seed)
    return np.random.random((min(hypotheses_number, 1024), initial_points_number))


def block_starts(block_sizes: np.ndarray) -> np.ndarray:
    """cuda_ransac.py:65-67: exclusive cumulative sum, int64."""
    bs = np.asarray(block_sizes)
    return np.cumsum(np.concatenate(([0], bs[:-1]))).astype(np.int64)


def ransac_evaluate(points, block_sizes, table, threshold, block_start=None, full=False, threads=1):
    """Run the C oracle.  Returns dict(mask, best, best_count, plane[, counts, planes], oob)."""
    lib = _load()
    pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
    bs = np.ascontiguousarray(block_sizes, dtype=np.int32)
    st = block_starts(bs) if block_start is None else np.ascontiguousarray(block_start, dtype=np.int64)
    tab = np.ascontiguousarray(table, dtype=np.float64)
    H, K = tab.shape
    assert K <= 64
    B, N = len(bs), len(pts)
    mask = np.zeros(N, dtype=np.uint8)
    best = np.zeros(B, dtype=np.int32)
    best_cnt = np.zeros(B, dtype=np.int32)
    plane = np.zeros((B, 4), dtype=np.float32)
    counts = np.zeros((B, H), dtype=np.int32) if full else None
    planes = np.zeros((B, H, 4), dtype=np.float32) if full else None
    ptr = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    oob = lib.ol_oracle_ransac(ptr(pts), N, ptr(bs), ptr(st), B, ptr(tab), H, K, float(threshold), ptr(mask),
                               ptr(best), ptr(best_cnt), ptr(plane), ptr(counts), ptr(planes), int(threads))
    out = dict(mask=mask, best=best, best_count=best_cnt, plane=plane, oob=int(oob), block_start=st)
    if full:
        out["counts"], out["planes"] = counts, planes
    return out


def mask_for_plane(points, start, n, plane, threshold) -> np.ndarray:
    lib = _load()
    pts = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
    pl = np.ascontiguousarray(plane, dtype=np.float32)
    out = np.zeros(n, dtype=np.uint8)
    lib.ol_oracle_mask_for_plane(pts.ctypes.data, int(start), int(n), pl.ctypes.data, float(threshold),
                                 out.ctypes.data)
    return out


# ---------------------------------------------------------------------------------------------
# independent numpy restatement (vectorised over hypotheses; float64 elementwise == IEEE, no FMA)
# ---------------------------------------------------------------------------------------------
def plane_from_points_numpy(pts: np.ndarray, idx: np.ndarray) -> np.ndarray:
    """util.py:28-84 for a batch: pts (N,3) f64, idx (H,K) int -> planes (H,4) float32."""
    H, K = idx.shape
    c = np.zeros((H, 3))
    for i in range(K):  # sequential accumulation order of util.py:37-40
        c = c + pts[idx[:, i]]
    c = c / K
    xx = xy = xz = yy = yz = zz = np.zeros(H)
    for i in range(K):
        r = pts[idx[:, i]] - c
        xx = xx + r[:, 0] * r[:, 0]
        xy = xy + r[:, 0] * r[:, 1]
        xz = xz + r[:, 0] * r[:, 2]
        yy = yy + r[:, 1] * r[:, 1]
        yz = yz + r[:, 1] * r[:, 2]
        zz = zz + r[:, 2] * r[:, 2]
    det_x = yy * zz - yz * yz
    det_y = xx * zz - xz * xz
    det_z = xx * yy - xy * xy
    sel_x = (det_x > det_y) & (det_x > det_z)
    sel_y = ~sel_x & (det_y > det_z)
    a_xy = xz * yz - xy * zz
    a_xz = xy * yz - xz * yy
    a_yz = xy * xz - yz * xx
    ax = np.where(sel_x, det_x, np.where(sel_y, a_xy, a_xz))
    ay = np.where(sel_x, a_xy, np.where(sel_y, det_y, a_yz))
    az = np.where(sel_x, a_xz, np.where(sel_y, a_yz, det_z))
    norm = np.sqrt(ax * ax + ay * ay + az * az)
    ok = norm != 0
    sn = np.where(ok, norm, 1.0)
    ax, ay, az = ax / sn, ay / sn, az / sn
    d = -(ax * c[:, 0] + ay * c[:, 1] + az * c[:, 2])
    planes = np.stack([ax, ay, az, d], axis=1)
    planes[~ok] = 0.0
    return planes.astype(np.float32)


def ransac_numpy(points, block_sizes, table, threshold, block_start=None):
    pts = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    bs = np.asarray(block_sizes, dtype=np.int32)
    st = block_starts(bs) if block_start is None else np.asarray(block_start, dtype=np.int64)
    H, K = table.shape
    mask = np.zeros(len(pts), dtype=np.uint8)
    best = np.full(len(bs), -1, dtype=np.int32)
    best_cnt = np.zeros(len(bs), dtype=np.int32)
    plane = np.zeros((len(bs), 4), dtype=np.float32)
    counts = np.zeros((len(bs), H), dtype=np.int32)
    for b, (n, s) in enumerate(zip(bs, st)):
        if n < K:
            continue
        idx = (table * np.float64(n) + np.float64(s)).astype(np.int32).astype(np.int64)  # cuda_ransac.py:104-107
        idx = np.clip(idx, 0, len(pts) - 1)
        pl = plane_from_points_numpy(pts, idx).astype(np.float64)  # f32 values, f64 arithmetic below
        blk = pts[s:s + n]
        dist = np.abs(((pl[:, 0:1] * blk[None, :, 0] + pl[:, 1:2] * blk[None, :, 1]) + pl[:, 2:3] * blk[None, :, 2])
                      + pl[:, 3:4])
        cnt = (dist < threshold).sum(axis=1).astype(np.int32)
        counts[b] = cnt
        t = int(np.argmax(cnt))  # first maximum == lowest index
        best[b], best_cnt[b] = t, cnt[t]
        plane[b] = pl[t].astype(np.float32)
        mask[s:s + n] = dist[t] < threshold
    return dict(mask=mask, best=best, best_count=best_cnt, plane=plane, counts=counts, block_start=st)
