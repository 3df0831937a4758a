"""Cost of the geometric criteria on the 100 M-point street workload (bench.py's c4_street_100M), one GPU:

  * device time of subdivide([MaxPoints(100)]) against subdivide([MaxPoints(100), MaxThickness(0.05, min_edge=0.25)]),
    with the per-stage timers and the new kernels' share of the HBM bandwidth measured in the same run (device-to-device
    copy), from their algorithmic bytes;
  * filter([Planar(0.02)]) and leaf_statistics();
  * the host compatibility path (the same criterion as an opaque callable) on a ~1 M-point sample, for contrast.

Writes one JSON file (default profiles/r03_geometric_criteria_v1.json) with the card name and power limit read in the
same run.  Usage: python tools/geometric_criteria_bench.py [--scale S] [--reps R] [--out PATH]"""
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
from octreelib_b200.criteria import MaxPoints, MaxThickness, Planar, halvings  # noqa: E402
from octreelib_b200.grid import Grid, GridConfig  # noqa: E402

GEOM_STAGES = ("geom_moments", "geom_block_moments")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60)
    name, limit = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
    return name, limit


def copy_bandwidth(dev):
    """bytes moved per second by a 4 GB device-to-device copy (read + write), best of 5"""
    a = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * a.numel() / (e0.elapsed_time(e1) * 1e-3))
    del a, b
    torch.cuda.empty_cache()
    return best


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), out


def fresh_grid(clouds, numbers):
    grid = Grid(GridConfig(voxel_edge_length=1.0))
    for n, c in zip(numbers, clouds):
        grid.insert_points(n, c)
    grid._host.forest.stats(light=True)  # build + uploads done before the timed call
    return grid


def positions_per_level(grid, levels):
    """points held by leaves of depth >= l: the positions the level loop visits at level l"""
    f = grid._host.forest
    depth = f.export_leaves()["depth"]
    blocks = f.export_blocks()
    d = depth[blocks["leaf"]].astype(np.int64)
    sizes = blocks["size"].astype(np.int64)
    return {l: int(sizes[d >= l].sum()) for l in levels}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_geometric_criteria_v1.json"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    name, limit = card()
    bw = copy_bandwidth(dev)
    clouds, numbers, P, total = bench.make_workload("c4_street_100M", 0, 1, dev, args.scale)
    count_only = [MaxPoints(100)]
    geometric = [MaxPoints(100), MaxThickness(0.05, min_edge=0.25)]
    geom_levels = list(range(halvings(1.0, 0.25)))  # the levels on which the thickness term is active
    res = dict(card=name, power_limit=limit, copy_bandwidth_GBps=bw / 1e9, workload="c4_street_100M", points=total, poses=P,
               reps=args.reps, criteria=dict(count_only=repr(count_only), geometric=repr(geometric)))

    def run(criteria, tag):
        times, prof, stats = [], None, None
        for rep in range(args.reps + 2):  # rep 0: warm-up, last rep: with the per-stage timers
            grid = fresh_grid(clouds, numbers)
            profiled = rep == args.reps + 1
            if profiled:
                grid._host.forest.profile(True)
            ms, _ = timed(lambda: grid.subdivide(criteria))
            if profiled:
                prof = grid._host.forest.profile_read()
                stats = grid._host.forest.stats()
            elif rep > 0:
                times.append(ms)
            if rep < args.reps + 1:
                del grid
        res[tag] = dict(subdivide_ms=times, subdivide_ms_median=float(np.median(times)),
                        stages={k: dict(launches=v[0], ms=v[1]) for k, v in prof.items()},
                        leaves=stats["n_leaves"], blocks=stats["n_blocks"], depth=stats["max_depth_reached"])
        return grid

    run(count_only, "subdivide_count_only")
    grid = run(geometric, "subdivide_geometric")
    st = grid._host.forest.stats()
    pos = positions_per_level(grid, geom_levels)
    # algorithmic bytes of geom_moments: 4 B perm + 24 B coordinates per position of a level with terms, 24 B of
    # statistics per leaf of the table at that level (the leaf table grows by 7 per split; upper bound: the final L)
    gbytes = sum(28 * pos[l] for l in geom_levels) + 24 * st["n_leaves"] * len(geom_levels)
    gms = res["subdivide_geometric"]["stages"].get("geom_moments", dict(ms=float("nan")))["ms"]
    res["subdivide_geometric"]["geom_moments_bytes"] = gbytes
    res["subdivide_geometric"]["geom_moments_share_of_copy_bw"] = gbytes / (gms * 1e-3) / bw
    res["subdivide_geometric"]["positions_per_level"] = pos

    # filter and leaf statistics on the geometrically subdivided grid (each on a fresh copy of it, warm-up first)
    for tag, op in (("leaf_statistics", lambda g: g.leaf_statistics()), ("filter_planar", lambda g: g.filter([Planar(0.02)]))):
        times, prof = [], None
        for rep in range(args.reps + 2):
            g = fresh_grid(clouds, numbers)
            g.subdivide(geometric)
            g._host.forest.stats()  # block table built before the timed call
            profiled = rep == args.reps + 1
            if profiled:
                g._host.forest.profile(True)
            ms, _ = timed(lambda: op(g))
            if profiled:
                prof = g._host.forest.profile_read()
            elif rep > 0:
                times.append(ms)
            del g
        A, NB = st["n_points_alive"], st["n_blocks"]
        out_bytes = NB * (8 + 24 + 48 + 24) if tag == "leaf_statistics" else NB
        bbytes = 28 * A + out_bytes
        bms = prof.get("geom_block_moments", (0, float("nan")))[1]
        res[tag] = dict(ms=times, ms_median=float(np.median(times)), stages={k: dict(launches=v[0], ms=v[1]) for k, v in prof.items()},
                        geom_block_moments_bytes=bbytes, geom_block_moments_share_of_copy_bw=bbytes / (bms * 1e-3) / bw)

    # host compatibility path on a ~1 M-point sample: the same criterion as an opaque callable (unguarded: the host path
    # cannot see the node size)
    k, acc = 0, 0
    while k < len(clouds) and acc < 1_000_000:
        acc += len(clouds[k])
        k += 1
    sample = [c.cpu().numpy() for c in clouds[:k]]
    thick = MaxThickness(0.05)
    dev_grid = fresh_grid(sample, numbers[:k])
    dev_ms, _ = timed(lambda: dev_grid.subdivide([MaxPoints(100), thick]))
    host_grid = fresh_grid(sample, numbers[:k])
    try:
        host_ms, _ = timed(lambda: host_grid.subdivide([MaxPoints(100), lambda p: thick(p)]))
        host_note = "ok"
    except RecursionError as exc:
        host_ms, host_note = float("nan"), f"RecursionError: {exc}"
    res["host_path_sample"] = dict(points=acc, poses=k, criteria="[MaxPoints(100), MaxThickness(0.05)]", device_ms=dev_ms,
                                   host_ms=host_ms, host_note=host_note)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, dict)}))
    for tag in ("subdivide_count_only", "subdivide_geometric", "leaf_statistics", "filter_planar", "host_path_sample"):
        print(tag, json.dumps({k: v for k, v in res[tag].items() if k != "stages"}))


if __name__ == "__main__":
    main()
