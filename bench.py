#!/usr/bin/env python
"""
bench.py -- points/sec over insert + subdivide + per-leaf RANSAC (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this build
    python bench.py --impl reference --gpus N ...            # CPU reference arm (oracle port, host cores)

A "step" = one full pass of the hot path over one synthetic map: Grid() -> insert_points x P ->
subdivide([len > 100]) -> map_leaf_points_cuda_ransac(H=1024, K=6).  Workload at every N: BASELINE
config 4, the 100M-point multi-pose "infinite street" LiDAR map (SURVEY.md 8(d)), total size fixed
(strong scaling); with N > 1 the poses are sharded over the ranks, points are routed to the rank
that owns their grid cell (hash of the cell key) with one NCCL all-to-all, and every cell is then
subdivided and segmented locally.

`value`  : device-resident inputs (points already in HBM when the timed region starts).
`e2e`    : the same step through the public API with HOST (pinned) input buffers and the result
           tables (leaf table + per-block plane table) read back to the host inside the timed region.
Timing   : CUDA events on the work stream, max over ranks, barrier + synchronize on both sides, W >= 3 warm-up
           steps.  The inputs (2.4 GB) are far larger than L2 (126 MB), so no extra L2 flush is needed.
`roofline`: the dominant HBM-bound kernel (one onesweep radix digit pass over all points), timed live by the
           library's CUDA-event stage profiler in a separate profiled step; `stages` lists every stage the same way,
           `roofline_ransac` the FP64-bound RANSAC kernel.  Peak = MEASURED_PEAKS.json (HBM copy GB/s).
`clocks` : NVML samples taken by the benchmark thread inside every warm-up and timed step (see ClockSampler).
`cpu_baseline` / `--impl reference`: the CPU oracle port (oracle/) on a bounded sample of the same workload.
`--dump-outputs DIR`: after the timed steps, what the last one computed goes to DIR/<name>.npy (see dump_outputs); the
           inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (generator, total points, edge, max points per leaf, ransac threshold)
    "c4_street_100M": dict(kind="street", points=100_000_000, edge=1.0, max_points=100, threshold=0.02),
    "c3_indoor_10M": dict(kind="indoor", points=10_000_000, edge=0.5, max_points=100, threshold=0.01),
    "c2_lidar_10x120k": dict(kind="lidar10", points=1_200_000, edge=1.0, max_points=100, threshold=0.02),
}
H, K = 1024, 6
POINTS_PER_POSE_EST = 118_000


# ------------------------------------------------------------------------------------------------
# distributed plumbing
# ------------------------------------------------------------------------------------------------
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def bind_to_gpu_numa_node(local):
    """Pin this process to the CPU cores NVML reports as local to its GPU (one process per GPU: the page-locked host
    buffers of the e2e leg are then first-touched on the GPU's own NUMA node and the host thread that drives the GPU runs
    next to it; torchrun does not bind its workers).  Returns a short description for the bench line, None if NVML or the
    affinity call is unavailable."""
    try:
        import pynvml

        pynvml.nvmlInit()
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local), n_words)
        cpus = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return f"{len(allowed)} cores local to GPU {local} ({allowed[0]}-{allowed[-1]})"
    except Exception:  # noqa: BLE001 - a measurement convenience, never a failure
        return None


def init_dist(world, local, backend="nccl"):
    import torch
    import torch.distributed as dist

    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        dist.init_process_group(backend=backend, device_id=torch.device("cuda", local) if backend == "nccl" else None)
    return dist


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle-reason samples taken DURING the warm-up and the timed steps.

    Source: NVML queried from the benchmark's own thread twice per step while the step's kernels are in flight
    (`sample()`; 3-10 us per query, measured with tools/nvml_cost.py) - the same counters that
    `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints (B200_PROFILING.md).  A polling side process
    (`nvidia-smi -lms 200`) or a polling thread was measured to stall the GPU for 10-300 ms per sample once
    peer-mapped memory exists (24 ms steps became 50-60 ms at N = 2), which would put the measurement tool inside
    the measurement; the subprocess is therefore only the fallback when NVML cannot be loaded."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.nvml = None
        self.handle = None
        self.max_mhz = None
        self.samples = []  # (sm_mhz, reasons bitmask)
        self.path = f"/tmp/ol_clocks_{os.getpid()}.csv"
        self.source = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")  # NVML enumerates physical devices
            idx = self.gpu_index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                idx = int(vis.split(",")[self.gpu_index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))  # 1.5 ms: once
            self.nvml = pynvml
            self.source = "nvml, benchmark thread, two samples per step while its kernels are in flight"
            return
        except Exception:  # noqa: BLE001
            self.nvml = None
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
            self.source = "nvidia-smi -lms 200"
        except Exception:  # noqa: BLE001
            self.proc = None

    def sample(self):
        if self.nvml is None:
            return
        p = self.nvml
        t0 = time.perf_counter()
        try:
            sm = p.nvmlDeviceGetClockInfo(self.handle, p.NVML_CLOCK_SM)
            try:
                reasons = p.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
            except Exception:  # noqa: BLE001 - older bindings
                reasons = p.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
            self.samples.append((float(sm), int(reasons)))
        except Exception:  # noqa: BLE001
            pass
        self.max_sample_ms = max(getattr(self, "max_sample_ms", 0.0), 1e3 * (time.perf_counter() - t0))

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        if self.nvml is not None:
            p = self.nvml
            bits = {"hw_slowdown": getattr(p, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(p, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(p, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(p, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            if self.samples:
                seen = 0
                for _, r in self.samples:
                    seen |= r
                out.update(sm_mhz=statistics.median(s[0] for s in self.samples), sm_max_mhz=self.max_mhz,
                           reasons=sorted(n for n, b in bits.items() if seen & b), samples=len(self.samples),
                           slowest_query_ms=round(getattr(self, "max_sample_ms", 0.0), 3))
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def make_workload(name, rank, world, device, scale=1.0):
    """Returns (list of per-pose CUDA float64 tensors owned by this rank, list of their global pose
    numbers, total pose count, total point count)."""
    import torch

    from octreelib_b200 import synthetic

    w = WORKLOADS[name]
    total = int(w["points"] * scale)
    if w["kind"] == "street":
        # the street is translation invariant along x, so every pose returns the same number of
        # points c0; P = ceil(total / c0) poses, the last one truncated to hit `total` exactly
        _, cnt = synthetic.lidar_street_torch(0, 1, seed=0, device=device)
        c0 = cnt[0]
        P = (total + c0 - 1) // c0
        lo, hi = rank * P // world, (rank + 1) * P // world
        mine, numbers = [], []
        chunk = 16
        for first in range(lo, hi, chunk):
            n = min(chunk, hi - first)
            pts, cnts = synthetic.lidar_street_torch(first, n, seed=0, device=device)
            off = 0
            for j, c in enumerate(cnts):
                pose = first + j
                take = min(c, total - pose * c0)
                mine.append(pts[off:off + take].clone())
                numbers.append(pose)
                off += c
        torch.cuda.empty_cache()
        return mine, numbers, P, total
    if w["kind"] == "indoor":
        pts = synthetic.indoor_torch(total, seed=0, device=device)
        P = 1
        if world > 1:  # a single pose split into contiguous index ranges (one run per rank)
            lo, hi = rank * total // world, (rank + 1) * total // world
            return [pts[lo:hi].clone()], [0], P, total
        return [pts], [0], P, total
    if w["kind"] == "lidar10":
        clouds = [torch.from_numpy(synthetic.lidar64_scan(p, seed=0)).to(device) for p in range(10)]
        P = 10
        lo, hi = rank * P // world, (rank + 1) * P // world
        return clouds[lo:hi], list(range(lo, hi)), P, sum(len(c) for c in clouds)
    raise ValueError(name)


# ------------------------------------------------------------------------------------------------
# one step of this build
# ------------------------------------------------------------------------------------------------
def run_step(clouds, numbers, n_poses_total, w, world, profile=False, read_tables=False, sampler=None):
    """clouds: per-pose arrays (CUDA tensors for `value`, pinned numpy arrays for `e2e`)."""
    from octreelib_b200.criteria import MaxPoints
    from octreelib_b200.grid import Grid, GridConfig

    np.random.seed(0)
    sharded = world > 1 or os.environ.get("OL_BENCH_SHARDED") == "1"  # debug: the multi-GPU host path on one GPU
    if sharded:
        from octreelib_b200.parallel import ShardedGrid

        grid = ShardedGrid(GridConfig(voxel_edge_length=w["edge"]), n_poses_total)
    else:
        grid = Grid(GridConfig(voxel_edge_length=w["edge"]))
    forest = grid._host.forest
    if profile:
        forest.profile(True)
        forest.extra_ransac_flags = 8  # OL_RANSAC_STATS: tally the executed fits / distance evaluations (profiled step only)
    for number, cloud in zip(numbers, clouds):
        grid.insert_points(number, cloud)
    if sharded:
        if profile:
            import torch
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
        grid.exchange()
        if profile:
            ev[1].record()
            torch.cuda.synchronize()
            grid.last_exchange["ms"] = ev[0].elapsed_time(ev[1])
    grid.subdivide([MaxPoints(w["max_points"])])
    if sampler is not None:
        sampler.sample()
    grid.map_leaf_points_cuda_ransac(poses_per_batch=10, threshold=w["threshold"], hypotheses_number=H,
                                     initial_points_number=K)
    if sampler is not None:
        sampler.sample()  # the mask compaction kernels of this step are still in flight
    d2h = 0
    if read_tables:
        planes = forest.export_ransac(scored_only=True)
        leaves = forest.export_leaves()
        d2h = sum(a.nbytes for a in planes.values()) + sum(a.nbytes for a in leaves.values())
    stats = forest.stats(light=True)  # waits for the step; the step's scalar results (alive points, leaves, ...)
    prof = forest.profile_read() if profile else None
    return grid, stats, prof, d2h


# ------------------------------------------------------------------------------------------------
# --dump-outputs
# ------------------------------------------------------------------------------------------------
DUMP_COUNTERS = ("n_points_inserted", "n_points_alive", "n_cells", "n_leaves", "n_internal", "n_blocks", "max_depth_reached")
DUMP_ROWS = {"leaf": 1 << 18, "plane": 1 << 18, "point": 1 << 19}  # 48 + 56 + 32 B per row: 44 MB at most
DUMP_SEED = 20240917


def _sample_rows(n, k, salt):
    """sorted indices of a fixed, seeded sample of k of n rows (every row when n <= k)"""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng([DUMP_SEED, salt]).choice(n, size=k, replace=False))


def dump_outputs(grid, out_dir):
    """Write what a step hands its caller as out_dir/<name>.npy, float64 throughout except the float32 planes:
      counters           the forest's counters (DUMP_COUNTERS order)
      pose_counts        (poses, 3) leaves, points, nodes per pose, in insertion order (Grid.n_leaves / n_points / n_nodes)
      leaf_*             leaf table (corner, edge, cell, depth)
      plane, plane_*     per-block RANSAC table, reference block order (plane, pose, leaf, size, best, best_count)
      point_xyz, _idx    surviving points in reference block order, with their index in their pose's cloud
    The three tables are sampled to at most DUMP_ROWS rows each; the sample depends only on the table's length."""
    forest = grid._host.forest
    st = forest.stats()
    out = {"counters": np.array([st[k] for k in DUMP_COUNTERS], dtype=np.float64),
           "pose_counts": np.asarray(grid._host.counts(), dtype=np.float64)}
    leaves = forest.export_leaves()
    rows = _sample_rows(len(leaves["edge"]), DUMP_ROWS["leaf"], 0)
    for k in ("corner", "edge", "cell", "depth"):
        out["leaf_" + k] = leaves[k][rows].astype(np.float64)
    planes = forest.export_ransac(scored_only=True)
    rows = _sample_rows(len(planes["plane"]), DUMP_ROWS["plane"], 1)
    out["plane"] = planes["plane"][rows].astype(np.float32)
    for k in ("pose", "leaf", "size", "best", "best_count"):
        out["plane_" + k] = planes[k][rows].astype(np.float64)
    points = forest.export_points(-1, order=0)
    rows = _sample_rows(len(points["idx"]), DUMP_ROWS["point"], 2)
    out["point_xyz"] = points["xyz"][rows].astype(np.float64)
    out["point_idx"] = points["idx"][rows].astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the REAL reference (oracle/_ref, made by oracle/make_ref.sh) on a bounded sample
# ------------------------------------------------------------------------------------------------
def _sample_clouds(workload, n_sample_points):
    """(clouds {pose: (n,3) f64}, edge, ransac threshold) of the bounded CPU sample of a workload"""
    from octreelib_b200 import synthetic

    w = WORKLOADS[workload]
    if w["kind"] == "street":
        n_poses = max(1, n_sample_points // POINTS_PER_POSE_EST)
        clouds = {p: synthetic.lidar_street_scan(p, seed=0) for p in range(n_poses)}
    elif w["kind"] == "indoor":
        clouds = {0: synthetic.indoor_scene(n_sample_points, seed=0) * (1.0 / w["edge"])}  # exact power-of-two rescale
    else:
        clouds = {p: synthetic.lidar64_scan(p, seed=0) for p in range(max(1, n_sample_points // 120_000))}
    edge = 1.0 if w["kind"] == "indoor" else w["edge"]
    thr = w["threshold"] / w["edge"] if w["kind"] == "indoor" else w["threshold"]
    return clouds, edge, thr


def cpu_reference_sample(workload, n_sample_points, threads):
    """One step of the hot path on the host cores, on a bounded sample of the workload.

    kind "reference": the UNMODIFIED reference package (oracle/_ref, a verbatim copy of /root/reference/octreelib; import
    shim only) runs `Grid.insert_points` x P -> `subdivide([len > max])` -> `map_leaf_points_cuda_ransac` (grid/grid.py:
    58-109, 244-258, 124-215: batching, `get_leaf_points`, vstack, `apply_mask` all as written) on ONE core - it is
    single-threaded Python.  The reference has no CPU RANSAC: its `CudaRansac` (a numba CUDA kernel, which cannot even be
    launched with the default 1024 threads per block on sm_100, see `reference_gpu_kernel` in the bench line) is
    substituted inside that call by the C restatement of the same kernel (oracle/ransac_oracle.c) on `threads` host threads.
    kind "port": no oracle/_ref on this machine - the numpy / C oracle port (oracle/structure.py) does everything."""
    from oracle import ransac as oransac

    w = WORKLOADS[workload]
    oransac.build()
    clouds, edge, thr = _sample_clouds(workload, n_sample_points)
    n = sum(len(c) for c in clouds.values())
    out = dict(points=n, poses=len(clouds))
    ref = None
    try:
        from oracle import ref_loader

        if ref_loader.reference_root() is not None:
            ref = ref_loader.load(cudasim=True)  # the numba kernel is never launched here
    except Exception as exc:  # noqa: BLE001
        out["reference_import_error"] = f"{type(exc).__name__}: {exc}"
        ref = None
    if ref is not None:
        import octreelib.grid.grid as ref_grid_module
        from octreelib.grid import Grid as RefGrid, GridConfig as RefGridConfig

        timer = {"ransac": 0.0}

        class HostRansac:  # stands in for octreelib.ransac.cuda_ransac.CudaRansac inside the reference's own call
            def __init__(self, threshold=0.01, hypotheses_number=1024, initial_points_number=6):
                self.threshold = threshold
                self.table = np.random.random((min(hypotheses_number, 1024), initial_points_number))  # cuda_ransac.py:39-41

            def evaluate(self, point_cloud, block_sizes):
                t = time.perf_counter()
                res = oransac.ransac_evaluate(point_cloud, block_sizes, self.table, self.threshold, threads=threads)
                timer["ransac"] += time.perf_counter() - t
                return res["mask"].astype(np.bool_)

        saved = ref_grid_module.CudaRansac
        ref_grid_module.CudaRansac = HostRansac
        try:
            np.random.seed(0)
            t0 = time.perf_counter()
            g = RefGrid(RefGridConfig(voxel_edge_length=edge))
            for p, c in clouds.items():
                g.insert_points(p, c)
            g.subdivide([lambda points, m=w["max_points"]: len(points) > m])
            t1 = time.perf_counter()
            g.map_leaf_points_cuda_ransac(poses_per_batch=10, threshold=thr, hypotheses_number=H, initial_points_number=K)
            t2 = time.perf_counter()
        finally:
            ref_grid_module.CudaRansac = saved
        out.update(kind="reference", seconds=t2 - t0, structure_s=(t2 - t0) - timer["ransac"], ransac_s=timer["ransac"],
                   alive=int(sum(g.n_points(p) for p in clouds)))
        return out
    from oracle.structure import OracleGrid, max_points_criterion

    np.random.seed(0)
    table = oransac.make_table(H, K)
    t0 = time.perf_counter()
    og = OracleGrid(edge)
    for p, c in clouds.items():
        og.insert_points(p, c)
    og.subdivide([max_points_criterion(w["max_points"])])
    t1 = time.perf_counter()
    og.map_leaf_points_ransac(table, threshold=thr, poses_per_batch=10,
                              evaluate=lambda pts, bs, tab, th: oransac.ransac_evaluate(pts, bs, tab, th, threads=threads))
    t2 = time.perf_counter()
    out.update(kind="port", seconds=t2 - t0, structure_s=t1 - t0, ransac_s=t2 - t1)
    return out


def _cpu_sample_text(r, workload, threads):
    if r["kind"] == "reference":
        return (f"{r['points']} points ({r['poses']} poses) of {workload}: the unmodified reference package (oracle/_ref) on 1 core "
                f"for insert_points + subdivide + the host side of map_leaf_points_cuda_ransac ({r['structure_s']:.2f} s); its numba "
                f"CUDA kernel replaced by the C port of that kernel on {threads} host thread(s) ({r['ransac_s']:.2f} s)")
    return (f"{r['points']} points ({r['poses']} poses) of {workload}: oracle port (no oracle/_ref here), structure "
            f"{r['structure_s']:.2f} s on 1 core + RANSAC {r['ransac_s']:.2f} s on {threads} thread(s)")


def ransac_stats_read(lib, reset=True):
    import ctypes as C

    out = (C.c_uint64 * 16)()
    lib.ol_ransac_stats_read(C.byref(out), 1 if reset else 0)
    keys = ["blocks", "prefiltered_hypotheses", "trivial_intervals", "candidate_evaluations", "early_exits", "interval_violations",
            "exact_fits", "exact_distance_evals", "fp32_distance_evals"]
    return {k: int(out[i]) for i, k in enumerate(keys)}


FIT_FLOPS_F64 = 152   # one exact plane fit at K = 6 (util.py:28-84: centroid 21, covariance 90, cofactors 15, normalise 9, d 5, indices 12)
DIST_FLOPS = 6        # one point-plane distance (util.py:16-24: 3 multiplications + 3 additions)
FIT_FLOPS_F32 = 120   # one float32 pre-filter fit incl. its error bounds


def ransac_rooflines(stats, kernel_ms, fp64_tflops, fp32_tflops):
    """Executed arithmetic of a RANSAC launch against the measured pipe peaks (FMA microbenchmark, 2 flops per FMA)."""
    f64 = stats["exact_fits"] * FIT_FLOPS_F64 + stats["exact_distance_evals"] * DIST_FLOPS
    f32 = stats["prefiltered_hypotheses"] * FIT_FLOPS_F32 + stats["fp32_distance_evals"] * DIST_FLOPS
    t = kernel_ms * 1e-3
    out = {"fp64_flops_executed": f64, "fp32_flops_executed": f32, "achieved_fp64_tflops": f64 / t / 1e12 if t else None,
           "achieved_fp32_tflops": f32 / t / 1e12 if t else None, "peak_fp64_tflops": fp64_tflops, "peak_fp32_tflops": fp32_tflops}
    if t and fp64_tflops and fp32_tflops:
        # both pipes work for the launch: the time each would need at its peak, added up, over the time taken
        out["frac"] = (f64 / (fp64_tflops * 1e12) + f32 / (fp32_tflops * 1e12)) / t
        out["frac_fp64_only"] = f64 / t / (fp64_tflops * 1e12)
    return out


def full_path_ransac(lib, device, fp64_tflops, fp32_tflops, n_points=2_000_000):
    """RANSAC where the early exit does NOT fire (VERDICT r1 #5c): uniformly random points (no planes), threshold 5 mm -
    no hypothesis keeps every point of its leaf, so all 1024 hypotheses of every block go through the float32 pre-filter
    and the surviving candidates through the exact float64 evaluation."""
    import torch

    from octreelib_b200.criteria import MaxPoints
    from octreelib_b200.grid import Grid, GridConfig

    g = torch.Generator(device=device)
    g.manual_seed(7)
    pts = torch.rand((n_points, 3), generator=g, device=device, dtype=torch.float32).to(torch.float64) * torch.tensor(
        [40.0, 40.0, 3.0], device=device, dtype=torch.float64)
    out = None
    for rep in range(2):  # the first repetition warms the allocator
        grid = Grid(GridConfig(voxel_edge_length=1.0))
        grid.insert_points(0, pts)
        grid.subdivide([MaxPoints(100)])
        f = grid._host.forest
        f.profile(True)
        f.extra_ransac_flags = 8
        ransac_stats_read(lib)
        np.random.seed(0)
        grid.map_leaf_points_cuda_ransac(poses_per_batch=10, threshold=0.005, hypotheses_number=H, initial_points_number=K)
        st = ransac_stats_read(lib)
        prof = f.profile_read()
        alive = f.stats(light=True)["n_points_alive"]
        ms = prof["ransac_kernel"][1]
        out = {"workload": f"clutter: {n_points} uniformly random points in 40 x 40 x 3 m, edge 1.0, <= 100 points / leaf, threshold 0.005",
               "blocks_fitted": st["blocks"], "early_exits": st["early_exits"], "kernel_ms": ms,
               "hypotheses_per_block": st["prefiltered_hypotheses"] / max(st["blocks"], 1) + 32,
               "exact_candidate_evaluations_per_block": st["candidate_evaluations"] / max(st["blocks"], 1),
               "points_kept": alive, "points_per_s": n_points / (ms * 1e-3) if ms else None,
               "hypothesis_evaluations_per_s": st["blocks"] * H / (ms * 1e-3) if ms else None}
        out.update(ransac_rooflines(st, ms, fp64_tflops, fp32_tflops))
        del grid, f
    return out


def _claim_stdout():
    """The driver reads ONE JSON line from stdout, but libraries write there too (NCCL prints its version banner to
    stdout during communicator creation).  Point file descriptor 1 at stderr for the whole run and keep a private
    duplicate of the real stdout for the result line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    sys.dont_write_bytecode = True  # the benchmark may run from a read-only tree: it writes nothing there
    result_out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4_street_100M", choices=list(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the workload's points (debug only)")
    ap.add_argument("--cpu-sample", type=int, default=250_000, help="points of the CPU baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-path", action="store_true", help="skip the clutter workload (RANSAC without early exits)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    rank, world, local = dist_env()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    w = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    base = {"metric": "points/sec (insert+subdivide+per-leaf RANSAC)", "unit": "points/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "data": "synthetic",
            "config": {"workload": args.workload, "points": int(w["points"] * args.scale), "voxel_edge_length": w["edge"],
                       "max_points_per_leaf": w["max_points"], "ransac": {"hypotheses": H, "initial_points": K,
                                                                         "threshold": w["threshold"]},
                       "l2": "inputs (24 B/point) exceed the 126 MB L2 by >10x; no extra flush",
                       "parallelism": f"cell-hash x{args.gpus}" if args.gpus > 1 else "single GPU"}}

    # ---------------------------------------------------------------- reference arm (CPU) --------
    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = cores
        times, pts = [], 0
        for i in range(args.warmup + args.steps):
            r = cpu_reference_sample(args.workload, args.cpu_sample, threads)
            if i >= args.warmup:
                times.append(r["seconds"])
                pts = r["points"]
        mean = sum(times) / len(times)
        val = pts / mean
        out = dict(base, impl="reference", value=val, ms_per_step=mean * 1e3, dtype="f64",
                   cpu_baseline={"value": val, "unit": "points/s", "cores": threads, "kind": r["kind"],
                                 "sample": _cpu_sample_text(r, args.workload, threads)},
                   e2e={"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                   gpu_launches=0)
        print(json.dumps(out), file=result_out, flush=True)
        return 0

    # ---------------------------------------------------------------- this build -----------------
    import torch

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    cpu_binding = bind_to_gpu_numa_node(local) if world > 1 else None
    dist = init_dist(world, local)
    from octreelib_b200 import _native

    lib = _native.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clouds, numbers, P, total = make_workload(args.workload, rank, world, device, args.scale)
    local_points = sum(int(c.shape[0]) for c in clouds)

    def timed(fn, steps):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        res = None
        for _ in range(steps):
            # drop the previous step's grid BEFORE building the next one, exactly like the warm-up loop does: with two
            # grids alive the caching allocator needs a second set of multi-GB blocks that the warm-up never created,
            # and the cudaMalloc calls for it (100-300 ms) would land inside the timed region
            res = None
            res = fn()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, res

    # clock samples are taken inside the warm-up and the timed steps (same load); see ClockSampler
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    smp = sampler if rank == 0 else None
    # warm-up (also warms torch's caching allocator so the timed steps do not call cudaMalloc)
    for _ in range(args.warmup):
        run_step(clouds, numbers, P, w, world, sampler=smp)
    launches0 = lib.ol_launch_count()
    ms, res = timed(lambda: run_step(clouds, numbers, P, w, world, sampler=smp), args.steps)
    launches_total = lib.ol_launch_count() - launches0  # this rank's kernels inside the timed region
    launches = launches_total // max(args.steps, 1)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms / args.steps
    value = total / (ms_per_step * 1e-3)
    stats = res[1]
    if args.dump_outputs:
        dump_outputs(res[0], args.dump_outputs)
    del res  # the last timed grid must not stay alive next to the profiled / e2e grids (memory at the 1e9-point scale)

    # profiled step (separate from the timed ones): per-stage times for the roofline object, executed-arithmetic tallies of
    # the RANSAC kernel (OL_RANSAC_STATS instantiation)
    import ctypes as C
    fp64_peak, fp32_peak = C.c_double(0.0), C.c_double(0.0)
    lib.ol_measure_fma_peak(C.c_void_p(torch.cuda.current_stream(device).cuda_stream), C.byref(fp64_peak), C.byref(fp32_peak))
    ransac_stats_read(lib)
    pgrid, pstats, prof, _ = run_step(clouds, numbers, P, w, world, profile=True)
    exchange_info = getattr(pgrid, "last_exchange", None)
    del pgrid
    # per-rank view of the profiled step (multi-GPU): the step time is set by the slowest rank, the others wait inside the
    # exchange's flag rounds - kernel time, the share of it spent in the two exchange stages, and the shard sizes
    ranks_info = None
    if world > 1 and dist is not None:
        mine = dict(rank=rank, kernel_ms=round(sum(v[1] for v in (prof or {}).values()), 3),
                    exchange_ms=round(sum(v[1] for k, v in (prof or {}).items() if k.startswith("exchange")), 3),
                    points=int(pstats["n_points_inserted"]), leaves=int(pstats["n_leaves"]), cells=int(pstats["n_cells"]))
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        ranks_info = gathered
    rstats = ransac_stats_read(lib)
    assert pstats["sample_oob_seen"] == 0 and stats["sample_oob_seen"] == 0, "a RANSAC sample index left its block"
    full_path = full_path_ransac(lib, device, fp64_peak.value, fp32_peak.value) if (rank == 0 and not args.no_full_path) else None

    # e2e: pinned host inputs, result tables read back
    e2e = None
    if not args.no_e2e:
        host_clouds = []
        for c in clouds:
            h = torch.empty(c.shape, dtype=torch.float64, pin_memory=True)
            h.copy_(c)
            host_clouds.append(h.numpy())
        torch.cuda.synchronize()
        h2d = sum(a.nbytes for a in host_clouds)
        run_step(host_clouds, numbers, P, w, world, read_tables=True)
        e_ms, e_res = timed(lambda: run_step(host_clouds, numbers, P, w, world, read_tables=True), args.steps)
        e_ms /= args.steps
        e2e = {"value": total / (e_ms * 1e-3), "unit": "points/s", "ms_per_step": e_ms, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": e_res[3]}
        del host_clouds, e_res

    if rank != 0:
        if world > 1:
            dist.barrier()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    # algorithmic bytes per processed element of every HBM-bound stage (DESIGN.md section 4)
    # (Morton codes are 32-bit words for trees of at most 10 levels, which covers every bench workload; the grid-wide sort
    # moves 32-bit keys when the packed cell key fits them - `key_bits` <= 32, every BASELINE configuration)
    kb = 4 if stats["key_bits"] <= 32 else 8
    # (when the Morton code rides in the low bits of the 32-bit sort key - no "gather_morton" stage - keygen writes no
    # Morton array and the cell segmentation peels the code off while it reads the sorted keys)
    embedded = bool(prof) and "gather_morton" not in prof
    BYTES = {"bbox": 24, "insert_batch": 48, "keygen": 24 + kb + 4 + (0 if embedded else 4), "sort_main_hist": kb,
             "sort_main_pass": 2 * (kb + 4),
             "radix_hist_u64": 8, "radix_scatter_u64": 24, "radix_hist_u32": 4, "radix_scatter_u32": 16, "scan": 8,
             "gather_morton": 12, "cells": kb + 4 + (4 if embedded else 0), "part_hist": 8, "part_move": 24, "gather_points": 52}
    KERNELS = {"sort_main_pass": f"os_pass_kernel<u{8 * kb}> (one onesweep radix digit pass over all points, K2)",
               "part_move": "part_move_kernel<u32> (fused rank + stable 8-way partition of one octree level, K4)"}
    stage_ms = {k: v[1] for k, v in (prof or {}).items()}
    stages = {}
    for k, (cnt, tot_ms, units) in (prof or {}).items():
        if k in BYTES and tot_ms > 0 and units > 0:
            gbs = BYTES[k] * units / (tot_ms * 1e-3) / 1e9
            stages[k] = {"launches": cnt, "ms": tot_ms, "elements": units, "bytes_per_element": BYTES[k], "GB/s": gbs,
                         "frac_of_hbm_peak": gbs / hbm_peak}
    hbm_total_bytes = sum(v["bytes_per_element"] * v["elements"] for v in stages.values())
    hbm_total_ms = sum(v["ms"] for v in stages.values())
    # ncu DRAM traffic per launch of the CURRENT build (profiles/r02_ncu_traffic.json, written by tools/ncu_traffic.py from
    # an `ncu --set full` capture of this workload); null when no capture of this build exists
    traffic_table = {}
    try:
        traffic_table = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
    except Exception:  # noqa: BLE001
        pass
    roofline = None
    dominant = max((k for k in KERNELS if k in stages), key=lambda k: stages[k]["ms"], default=None)
    if dominant:
        # the dominant HBM-bound kernel by time inside the step
        st = stages[dominant]
        per_launch_units = st["elements"] / st["launches"]
        tr = traffic_table.get(dominant)
        traffic = tr["dram_bytes_per_launch"] * per_launch_units / tr["elements_per_launch"] if tr else None
        roofline = {"kernel": KERNELS[dominant], "bound": "hbm", "achieved": st["GB/s"], "peak": hbm_peak, "unit": "GB/s",
                    "frac": st["frac_of_hbm_peak"], "traffic": traffic,
                    "traffic_source": (tr or {}).get("source"),
                    "algorithmic_bytes_per_launch": st["bytes_per_element"] * per_launch_units,
                    "avg_launch_ms": st["ms"] / st["launches"], "peak_source": peak_src, "launches": st["launches"],
                    "all_hbm_stages": {"bytes": hbm_total_bytes, "ms": hbm_total_ms,
                                       "GB/s": hbm_total_bytes / (hbm_total_ms * 1e-3) / 1e9 if hbm_total_ms else None,
                                       "frac": hbm_total_bytes / (hbm_total_ms * 1e-3) / 1e9 / hbm_peak if hbm_total_ms else None},
                    "note": f"achieved = {st['bytes_per_element']} B x elements per launch / average CUDA-event duration of the "
                            "launches of one step; `all_hbm_stages` aggregates every HBM-bound stage of the step (`stages`); "
                            "the FP64-bound RANSAC kernel is under `roofline_ransac`"}
    out = dict(base, value=value, ms_per_step=ms_per_step, dtype="f64", clocks=clocks, gpu_launches=int(launches_total), gpu_launches_per_step=int(launches),
               stage_ms=stage_ms, stages=stages,
               result={k: stats[k] for k in ("n_points_inserted", "n_points_alive", "n_cells", "n_leaves",
                                             "max_depth_reached", "key_bits", "device_bytes_peak", "sample_oob_seen")},
               n_poses=P)
    if roofline:
        out["roofline"] = roofline
    if prof and "ransac_kernel" in prof:
        r_ms, r_blocks = prof["ransac_kernel"][1], prof["ransac_kernel"][2]
        rr = {"kernel": "ransac_small_kernel (K6; ransac_kernel for blocks > 128 points)", "bound": "fp64 pipe", "ms": r_ms,
              "blocks_fitted": r_blocks, "executed": rstats,
              "reference_equivalent_hypotheses_per_s": r_blocks * H / (r_ms * 1e-3) if r_ms else None,
              "peak_source": "ol_measure_fma_peak: dense FMA microbenchmark on this GPU at the clocks of this run (2 flops per FMA)",
              "note": "executed flops = exact fits x 152 + exact point distances x 6 (float64), pre-filter fits x 120 + distances x 6 "
                      "(float32), tallied by the OL_RANSAC_STATS instantiation in the profiled step; the reference's arithmetic "
                      "forbids FMA contraction (-fmad=false), so a multiply-add pair can reach at most half of the FMA peak. On "
                      "this workload every block exits after its first group of 8 exact hypotheses (planar leaves); "
                      "`roofline_ransac_full_path` is the same kernel on a workload without early exits"}
        rr.update(ransac_rooflines(rstats, r_ms, fp64_peak.value, fp32_peak.value))
        out["roofline_ransac"] = rr
    if full_path:
        out["roofline_ransac_full_path"] = full_path
    ref_gpu = os.path.join(ROOT, "profiles", "r02_reference_numba_on_b200_v2.json")
    if os.path.exists(ref_gpu):
        try:
            rg = json.load(open(ref_gpu))
            runs = {r["H"]: r for r in rg.get("runs", [])}
            out["reference_gpu_kernel"] = {
                "source": "profiles/r02_reference_numba_on_b200_v2.json (tools/ref_on_gpu.py on a B200 of this pool: the unmodified "
                          "reference kernel through numba " + str(rg.get("numba_version")) + ", BASELINE config 1 blocks)",
                "H1024": runs.get(1024, {}).get("reference_error"),
                "H512_evaluate_wall_ms": {"reference": runs.get(512, {}).get("reference_evaluate", {}).get("wall_ms_best"),
                                          "ours": runs.get(512, {}).get("ours_evaluate", {}).get("wall_ms_best")},
                "H512_parity": runs.get(512, {}).get("parity_vs_reference_kernel_on_b200")}
        except Exception:  # noqa: BLE001
            pass
    if cpu_binding:
        out["cpu_binding"] = cpu_binding
    if ranks_info:
        out["ranks"] = ranks_info
    if exchange_info:
        out["exchange"] = dict(exchange_info, note="rank 0; ms = CUDA events around ShardedGrid.exchange() in the profiled step "
                                                   "(fused exchange: slab boundaries from a sample histogram, counting pass, flag "
                                                   "rounds over peer-mapped control blocks, scatter into the owners' receive buffers, "
                                                   "key / sort / cell kernels enqueued behind it; includes the wait for the slowest "
                                                   "rank); bytes = point rows this rank sent to other ranks x 24")
    if e2e:
        out["e2e"] = e2e
    if not args.no_cpu_baseline and world == 1:
        r = cpu_reference_sample(args.workload, args.cpu_sample, 1)
        out["cpu_baseline"] = {"value": r["points"] / r["seconds"], "unit": "points/s", "cores": 1, "kind": r["kind"],
                               "sample": _cpu_sample_text(r, args.workload, 1)}
    print(json.dumps(out), file=result_out, flush=True)
    if world > 1:
        dist.barrier()
    return 0


if __name__ == "__main__":
    sys.exit(main())
