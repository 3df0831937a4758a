"""Throughput of `Grid.locate_points` on the 100 M-point street workload (bench.py's c4_street_100M), one GPU.

The map is built like tools/leaf_map_bench.py does it: every pose inserted as a CUDA tensor, `subdivide([MaxPoints(100)])`,
the derived tables made current before anything is timed.  Then:

  (a) every map point, as one CUDA tensor, located without a pose number and with one (the first pose's rows);
  (b) one fresh street scan (~120 k points, a pose in the middle of the street with other noise) located over and over,
      as the inner loop of a scan-to-map registration would: as a CUDA tensor and as a numpy array (host copies in the
      call).

Device times are CUDA events around `--reps` calls after one warm-up call; the numpy path is timed with host clocks
around calls that end in a synchronisation.  The roofline denominator is 32 B per query (24 B coordinates read, 8 B
result written); the cell keys, leaf paths and ranks are looked up through L2 and not counted.  (a) streams 3.2 GB per
call, far more than the 126 MB L2; the scan of (b) is 3.8 MB and stays in L2 across repetitions, so its GB/s is not an
HBM figure.  Writes one JSON file with the card name and power limit read in the same run.
Usage: python tools/locate_bench.py [--scale S] [--reps R] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from octreelib_b200 import synthetic  # noqa: E402
from octreelib_b200.criteria import MaxPoints  # noqa: E402
from octreelib_b200.grid import Grid, GridConfig  # noqa: E402

BYTES_PER_QUERY = 24 + 8


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60)
    name, limit = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
    return name, limit


def device_ms(fn, reps):
    fn()  # warm-up
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / reps


def host_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0) / reps


def row(n, ms, **extra):
    return dict(queries=n, ms=ms, queries_per_s=n / (ms * 1e-3), gb_per_s=n * BYTES_PER_QUERY / (ms * 1e-3) / 1e9, **extra)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_locate_v1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("locate_bench.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    name, limit = card()
    clouds, numbers, P, total = bench.make_workload("c4_street_100M", 0, 1, dev, args.scale)
    grid = Grid(GridConfig(voxel_edge_length=1.0))
    for n, c in zip(numbers, clouds):
        grid.insert_points(n, c)
    grid.subdivide([MaxPoints(100)])
    st = grid._host.forest.stats()
    res = dict(card=name, power_limit=limit, workload="c4_street_100M", scale=args.scale, points=total, poses=P,
               cells=st["n_cells"], leaves=st["n_leaves"], depth=st["max_depth_reached"], reps=args.reps,
               bytes_per_query=BYTES_PER_QUERY)
    pose = numbers[0]
    grid.locate_points(clouds[0][:1], pose)  # the pose-row table of `pose` uploaded before the timed calls
    everything = torch.cat(clouds)
    del clouds
    torch.cuda.empty_cache()
    located = grid.locate_points(everything)
    res["map_all"] = row(len(everything), device_ms(lambda: grid.locate_points(everything), args.reps),
                         located=int((located >= 0).sum()))
    res["map_all_pose"] = row(len(everything), device_ms(lambda: grid.locate_points(everything, pose), args.reps))
    del everything, located
    scan, _ = synthetic.lidar_street_torch(P // 2, 1, seed=1, device=dev)
    scan_np = scan.cpu().numpy()
    got = grid.locate_points(scan)
    assert (got.cpu().numpy() == grid.locate_points(scan_np)).all()
    res["scan_cuda"] = row(len(scan), device_ms(lambda: grid.locate_points(scan), args.reps), located=int((got >= 0).sum()))
    res["scan_numpy"] = row(len(scan), host_ms(lambda: grid.locate_points(scan_np), args.reps))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
