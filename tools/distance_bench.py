"""Throughput of the free-space distance field (ag_cspace_distance: k_dist_init, k_dist_relax, k_dist_finish) next to the
occupancy call that makes its input (ag_cspace_occupancy), against the composed form a user would otherwise write: a
level-synchronous BFS in torch, one torch.roll step of the frontier per level (tests/distance_reference.py
composed_distance).  Both give identical distances (asserted); where the composed form cannot finish in reasonable time
(the serpentine: one level per pose of a 500,000-pose corridor) the distances are held to the scipy BFS instead.  Also
times the lattice descent (ag_cspace_descend) on scene_0.  Prints one JSON line.

    python tools/distance_bench.py [--min-window 0.5] [--quick]

Workloads (default lattices: the whole torus from 0, both axes wrapping; FAST occupancy; goals: the lattice poses nearest
the scene's own target, both inverse-kinematics solutions of target_c): scene_0's 9x9 map with a 4096^2 lattice; bench.py's
config-4 grid (1024^2, Bernoulli(0.002), numpy seed 4) with a 1024^2 lattice; bench.py's config-5 grids (256^2,
Bernoulli(0.008), base cells kept free, torch seed 5), 1024 of them with a 256^2 lattice each; a synthetic 4096^2 image
with free fraction 0.6 (just above the site-percolation threshold: long, fractal distances) and one goal, the smallest
pose of its largest component; a 1-pose-wide serpentine at 1024^2 without wrap, goal at one end: every distance is a walk
along the corridor, the worst case for tile relaxation (one pass per tile the corridor crosses).
relax_launches counts the relaxation kernels a call launches (its launches minus init and finish).  The host launches
them in groups of 16 and reads the change counter after each group, so host syncs = relax_launches / 16, and the last
group holds the first pass that changed nothing plus up to 15 more that return at once: the passes that did work number
between relax_launches - 16 and relax_launches - 1.  The composed form is timed once (the call whose distances are checked).
Descent: 2^20 starts drawn uniformly on scene_0's 4096^2 field (torch seed 3), max_len 4096, one thread per start.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import abstract_gym_b200 as ag                                   # noqa: E402
from abstract_gym_b200 import ops                                # noqa: E402
from components_reference import pack_words, special_images, unpack_free   # noqa: E402
from cspace_bench import gpu_info, timed                         # noqa: E402
from distance_reference import composed_distance, distance_numpy   # noqa: E402

SYNC_PASSES = 16


def workload(name, dev, quick):
    """(scene or None, b1, b2, wrap, int32 words [n_grids, b1, W], int32 goal words)"""
    if name == "perc":
        b = 512 if quick else 4096
        free = torch.rand(1, b, b, device=dev, generator=torch.Generator(device=dev).manual_seed(7)) < 0.6
        words = pack_words(~free)
        labels = torch.empty(1, b, b, dtype=torch.int32, device=dev)
        ops.cspace_components(words, b, b, 3, labels, None)
        sizes = torch.bincount(labels[labels >= 0].long(), minlength=b * b)
        goals = torch.zeros(1, b * b, dtype=torch.bool, device=dev)
        goals[0, int(sizes.argmax())] = True                          # a label is its component's smallest pose
        return None, b, b, 3, words, pack_words(goals.view(1, b, b))
    if name == "serpentine":
        b = 128 if quick else 1024
        free = torch.as_tensor(special_images(b, b)["comb"], device=dev)[None]
        goals = torch.zeros_like(free)
        goals[0, 0, 0] = True
        return None, b, b, 0, pack_words(~free), pack_words(goals)
    if name == "scene0":
        grid, b = ag.OccupancyGrid(size=9, random_obstacle=False), 4096
    elif name == "c4":
        grid = ag.OccupancyGrid(size=9, random_obstacle=False)
        grid.load_from_matrix((np.random.default_rng(4).random((1024, 1024)) < 0.002).astype(np.uint8))
        b = 1024
    else:
        grid = ag.BatchedOccupancyGrid.random(64 if quick else 1024, 256, 0.008, 256, device=dev,
                                              generator=torch.Generator(device=dev).manual_seed(5), clear_base_cells=2)
        b = 256
    z = torch.zeros(1, dtype=torch.float64, device=dev)
    sc = ag.BatchedScene(ag.BatchedTwoJointRobot(z, z.clone()), grid)
    b = b // 8 if quick else b
    words = sc.cspace_occupancy(b, packed=True)
    st = 2 * np.pi / b
    goals = pack_words(sc._goal_image(None, words.shape[0], b, b, (0.0, 0.0), (st, st), 3))
    return sc, b, b, 3, words, goals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds of timed launches per form and workload")
    ap.add_argument("--quick", action="store_true", help="small lattices and 64 config-5 grids (a smoke run)")
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    out = dict(metric="free-space distance: lattice poses/s, ag_cspace_distance vs a level-synchronous torch BFS; "
                      "ag_cspace_occupancy on the same lattice; ag_cspace_descend paths/s", gpu=gpu_info(), workloads={})
    composed_distance(torch.ones(1, 8, 8, dtype=torch.bool, device=dev), torch.ones(1, 8, 8, dtype=torch.bool, device=dev), 3)
    for name in ("scene0", "c4", "c5", "perc", "serpentine"):
        sc, b1, b2, wrap, words, goals = workload(name, dev, args.quick)
        n = words.shape[0]
        dist = torch.empty(n, b1, b2, dtype=torch.int32, device=dev)
        md = torch.empty(n, dtype=torch.int32, device=dev)
        run = lambda: ops.cspace_distance(words, goals, b1, b2, wrap, dist, md)
        run()
        torch.cuda.synchronize()
        before = ag.launch_count()
        run()
        launches = ag.launch_count() - before - 2
        poses = n * b1 * b2
        free = unpack_free(words, b2)
        res = dict(grids=n, lattice=[b1, b2], wrap=wrap, poses=poses, free_fraction=float(free.sum()) / poses,
                   reachable_fraction=float((dist >= 0).sum()) / poses, max_dist=int(md.max()),
                   relax_launches=launches, host_syncs=launches // SYNC_PASSES)
        t, reps = timed(run, args.min_window)
        res["distance"] = dict(seconds_per_call=t, reps=reps, poses_per_s=poses / t)
        if sc is not None:
            t, reps = timed(lambda: sc.cspace_occupancy(b1, packed=True), args.min_window)
            res["occupancy"] = dict(seconds_per_call=t, reps=reps, poses_per_s=poses / t)
            res["distance_share_of_occupancy"] = res["distance"]["seconds_per_call"] / t
        gimg = unpack_free(goals, b2) == 0
        if name == "serpentine":
            want = torch.as_tensor(distance_numpy(free.cpu().numpy(), gimg.cpu().numpy(), wrap), device=dev)
            res["reference"] = "scipy"
        else:
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            want, levels = composed_distance(free, gimg, wrap)
            e.record()
            e.synchronize()
            tc = a.elapsed_time(e) / 1e3
            res["composed"] = dict(seconds_per_call=tc, levels=levels, poses_per_s=poses / tc)
            res["speedup"] = tc / res["distance"]["seconds_per_call"]
            res["reference"] = "composed"
        assert torch.equal(dist, want), "%s: %d distances differ" % (name, int((dist != want).sum()))
        if name == "scene0":
            m, max_len = (1 << 14 if args.quick else 1 << 20), 4096
            start = torch.randint(0, b1 * b2, (m,), dtype=torch.int32, device=dev,
                                  generator=torch.Generator(device=dev).manual_seed(3))
            grid = torch.zeros(m, dtype=torch.int64, device=dev)
            path = torch.empty(m, max_len, dtype=torch.int32, device=dev)
            length = torch.empty(m, dtype=torch.int32, device=dev)
            t, reps = timed(lambda: ops.cspace_descend(dist, b1, b2, wrap, start, grid, max_len, path, length),
                            args.min_window)
            res["descend"] = dict(starts=m, max_len=max_len, seconds_per_call=t, reps=reps, paths_per_s=m / t,
                                  mean_length=float(length.double().mean()), max_length=int(length.max()))
            del path
        out["workloads"][name] = res
        del sc, words, goals, dist, free, gimg, want
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
