"""Throughput of configuration-space occupancy (BatchedScene.cspace_occupancy, kernel k_cspace) against the composed form
a user would otherwise write: lattice poses in torch, chunk by chunk, then ag_collision_check on env ids of each grid,
then packing in torch (tests/cspace_reference.py composed_occupancy).  Both forms must give identical words (asserted).
Prints one JSON line.

    python tools/cspace_bench.py [--min-window 0.5] [--quick]

Workloads (default lattices: the whole torus from 0, axis rows included): scene_0's 9x9 map with a 4096^2 lattice
(FAST: the map form); bench.py's config-4 grid (1024^2, Bernoulli(0.002), numpy seed 4) with a 1024^2 lattice, FAST and
EXACT; bench.py's config-5 grids (256^2, Bernoulli(0.008), base cells kept free, torch seed 5), 1024 of them with a
256^2 lattice each, FAST.  The composed form checks 2^24 poses per ag_collision_check launch (268 MB of pose arrays).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import abstract_gym_b200 as ag                        # noqa: E402
from cspace_reference import composed_occupancy      # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def timed(fn, min_window):
    fn()                                                     # warm-up (and the map's first build)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 1
    while True:
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        elapsed = a.elapsed_time(b) / 1e3
        if elapsed >= min_window:
            return elapsed / reps, reps
        reps = max(reps + 1, int(reps * 1.5 * min_window / max(elapsed, 1e-6)))


def workload(name, dev, quick):
    if name == "scene0":
        grid, b = ag.OccupancyGrid(size=9, random_obstacle=False), 4096
    elif name.startswith("c4"):
        grid = ag.OccupancyGrid(size=9, random_obstacle=False)
        grid.load_from_matrix((np.random.default_rng(4).random((1024, 1024)) < 0.002).astype(np.uint8))
        b = 1024
    else:
        grid = ag.BatchedOccupancyGrid.random(64 if quick else 1024, 256, 0.008, 256, device=dev,
                                              generator=torch.Generator(device=dev).manual_seed(5), clear_base_cells=2)
        b = 256
    z = torch.zeros(1, dtype=torch.float64, device=dev)
    sc = ag.BatchedScene(ag.BatchedTwoJointRobot(z, z.clone()), grid)
    return sc, (b // 8 if quick else b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds of timed launches per form and workload")
    ap.add_argument("--quick", action="store_true", help="small lattices and 64 config-5 grids (a smoke run)")
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    out = dict(metric="configuration-space occupancy: lattice poses/s, k_cspace vs torch poses + ag_collision_check + torch "
                      "packing", gpu=gpu_info(), workloads={})
    for name, engine in (("scene0", "fast"), ("c4", "fast"), ("c4_exact", "exact"), ("c5", "fast")):
        sc, b = workload(name, dev, args.quick)
        e = ag.ENGINES[engine]
        n = int(sc.grid.n_grids)
        st = (2.0 * np.pi / b, 2.0 * np.pi / b)
        words, fc = sc.cspace_occupancy(b, packed=True, free_count=True, engine=engine)
        cw = composed_occupancy(sc, (0.0, 0.0), st, b, b, e)
        assert torch.equal(words, cw), "%s: %d words differ" % (name, int((words != cw).sum()))
        poses = n * b * b
        res = dict(grids=n, lattice=[b, b], engine=engine, poses=poses, free_fraction=float(fc.sum().item()) / poses)
        for form, fn in (("kernel", lambda: sc.cspace_occupancy(b, packed=True, engine=engine)),
                         ("composed", lambda: composed_occupancy(sc, (0.0, 0.0), st, b, b, e))):
            t, reps = timed(fn, args.min_window)
            res[form] = dict(seconds_per_call=t, reps=reps, poses_per_s=poses / t)
        res["speedup"] = res["composed"]["seconds_per_call"] / res["kernel"]["seconds_per_call"]
        out["workloads"][name] = res
        del sc, words, fc, cw
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
