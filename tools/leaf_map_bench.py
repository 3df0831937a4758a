"""Cost of the declarative leaf maps (Centroid, Shrink, FirstPoints) on the 100 M-point street workload (bench.py's
c4_street_100M), one GPU:

  * the device time of `map_leaf_points(obj)` on the full map after `subdivide([MaxPoints(100)])`, per object, with the
    per-stage timers (`leaf_map`, `leaf_map_check`, and the rebuild stages) from a separate profiled repetition;
  * the host path (the same map as a plain function, one Python call per block) against the device path on the same
    bounded sample of poses.

Times are host clocks around calls that end in a device synchronisation.  Writes one JSON file with the card name and
power limit read in the same run.  Usage: python tools/leaf_map_bench.py [--scale S] [--reps R] [--sample-points N] [--out PATH]"""
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
from octreelib_b200.criteria import MaxPoints  # noqa: E402
from octreelib_b200.grid import Grid, GridConfig  # noqa: E402
from octreelib_b200.leaf_maps import Centroid, FirstPoints, Shrink  # noqa: E402

OBJECTS = {"centroid": Centroid(), "shrink_0.5": Shrink(0.5), "first_points_1": FirstPoints(1)}
PLAIN = {"centroid": lambda c: c.mean(axis=0, keepdims=True),
         "shrink_0.5": lambda c: c.mean(axis=0) + 0.5 * (c - c.mean(axis=0)),
         "first_points_1": lambda c: c[:1]}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60)
    name, limit = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
    return name, limit


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def subdivided(clouds, numbers):
    grid = Grid(GridConfig(voxel_edge_length=1.0))
    for n, c in zip(numbers, clouds):
        grid.insert_points(n, c)
    grid.subdivide([MaxPoints(100)])
    grid._host.forest.stats()  # build, leaf order and block table done before the timed call
    return grid


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sample-points", type=int, default=300_000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_leaf_maps_v1.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("leaf_map_bench.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    name, limit = card()
    clouds, numbers, P, total = bench.make_workload("c4_street_100M", 0, 1, dev, args.scale)
    res = dict(card=name, power_limit=limit, workload="c4_street_100M", scale=args.scale, points=total, poses=P, reps=args.reps)
    for tag, obj in OBJECTS.items():
        times, prof, st = [], None, None
        for rep in range(args.reps + 2):  # rep 0: warm-up, last rep: with the per-stage timers
            grid = subdivided(clouds, numbers)
            if rep == 0:
                st = grid._host.forest.stats()
            profiled = rep == args.reps + 1
            if profiled:
                grid._host.forest.profile(True)
            ms = timed(lambda: grid.map_leaf_points(obj))
            if profiled:
                prof = grid._host.forest.profile_read()
            elif rep > 0:
                times.append(ms)
            after = grid._host.forest.stats(light=True)["n_points_alive"]
            del grid
        A, NB = st["n_points_alive"], st["n_blocks"]
        res[tag] = dict(ms=times, ms_median=float(np.median(times)), points_before=A, blocks=NB, points_after=after,
                        stages={k: dict(launches=v[0], ms=v[1]) for k, v in prof.items()})
    # host path vs device path on the first poses (about --sample-points points)
    k, acc = 0, 0
    while k < len(clouds) and acc < args.sample_points:
        acc += len(clouds[k])
        k += 1
    sample = [c.cpu().numpy() for c in clouds[:k]]
    res["sample"] = dict(points=acc, poses=k)
    for tag, obj in OBJECTS.items():
        g_dev, g_host = subdivided(sample, numbers[:k]), subdivided(sample, numbers[:k])
        dev_ms = timed(lambda: g_dev.map_leaf_points(obj))
        host_ms = timed(lambda: g_host.map_leaf_points(PLAIN[tag]))
        same = all((g_dev.get_points(n) == g_host.get_points(n)).all() for n in numbers[:k])
        res["sample"][tag] = dict(device_ms=dev_ms, host_ms=host_ms, blocks=g_dev._host.forest.stats()["n_blocks"], same_result=bool(same))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, dict)}))
    for tag in list(OBJECTS) + ["sample"]:
        print(tag, json.dumps(res[tag]))


if __name__ == "__main__":
    main()
