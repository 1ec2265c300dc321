"""Throughput of free-space component labelling (ag_cspace_components: k_ccl_local, k_ccl_border, k_ccl_compress) next
to the occupancy call that makes its input (ag_cspace_occupancy) and against the composed form a user would otherwise
write: min-label propagation over the 4 neighbours in torch, then pointer jumping L = L[L] until fixpoint, repeated
until nothing changes (tests/components_reference.py composed_components).  Both give identical labels (asserted).
Prints one JSON line.

    python tools/components_bench.py [--min-window 0.5] [--quick]

Workloads (default lattices: the whole torus from 0, both axes wrapping; FAST occupancy): scene_0's 9x9 map with a
4096^2 lattice; bench.py's config-4 grid (1024^2, Bernoulli(0.002), numpy seed 4) with a 1024^2 lattice; bench.py's
config-5 grids (256^2, Bernoulli(0.008), base cells kept free, torch seed 5), 1024 of them with a 256^2 lattice each; a
synthetic 4096^2 image with free fraction 0.6, just above the 4-neighbour site-percolation threshold (0.593), where
components are huge and fractal.  Labelling is timed with the per-grid counts on, back to back on the same buffers: the
labels of the 4096^2 and 1024^2 lattices (64 MB, 4 MB) can stay in the 126 MB L2 between calls, those of config 5
(268 MB) cannot.  The composed form is timed once (the call whose labels are checked), after a warm-up on a tiny image.
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
from components_reference import composed_components, pack_words, unpack_free   # noqa: E402
from cspace_bench import gpu_info, timed                         # noqa: E402


def workload(name, dev, quick):
    """(scene or None, lattice size, int32 words [n_grids, b, W])"""
    if name == "perc":
        b = 512 if quick else 4096
        free = torch.rand(1, b, b, device=dev, generator=torch.Generator(device=dev).manual_seed(7)) < 0.6
        return None, b, pack_words(~free)
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
    return sc, b, sc.cspace_occupancy(b, packed=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds of timed launches per form and workload")
    ap.add_argument("--quick", action="store_true", help="small lattices and 64 config-5 grids (a smoke run)")
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    out = dict(metric="free-space components: lattice poses/s labelled, ag_cspace_components vs torch min-label "
                      "propagation + pointer jumping; ag_cspace_occupancy on the same lattice", gpu=gpu_info(), workloads={})
    composed_components(torch.ones(1, 8, 8, dtype=torch.bool, device=dev), 3)          # load the torch kernels
    for name in ("scene0", "c4", "c5", "perc"):
        sc, b, words = workload(name, dev, args.quick)
        n = words.shape[0]
        labels = torch.empty(n, b, b, dtype=torch.int32, device=dev)
        nc = torch.empty(n, dtype=torch.int64, device=dev)
        label = lambda: ops.cspace_components(words, b, b, 3, labels, nc)
        label()
        free = unpack_free(words, b)
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        want, iters = composed_components(free, 3)
        e.record()
        e.synchronize()
        assert torch.equal(labels, want), "%s: %d labels differ" % (name, int((labels != want).sum()))
        poses = n * b * b
        per = labels.view(n, -1).to(torch.int64)
        sizes = torch.bincount((per + torch.arange(n, device=dev).view(-1, 1) * b * b)[per >= 0], minlength=poses)
        n_free = (per >= 0).sum(dim=1)
        share = sizes.view(n, -1).max(dim=1).values.double() / n_free.clamp(min=1).double()
        res = dict(grids=n, lattice=[b, b], poses=poses, free_fraction=float(n_free.sum()) / poses,
                   components=int(nc.sum()), components_per_grid_max=int(nc.max()),
                   largest_share_mean=float(share.mean()), largest_share_min=float(share.min()))
        t, reps = timed(label, args.min_window)
        res["label"] = dict(seconds_per_call=t, reps=reps, poses_per_s=poses / t)
        if sc is not None:
            t, reps = timed(lambda: sc.cspace_occupancy(b, packed=True), args.min_window)
            res["occupancy"] = dict(seconds_per_call=t, reps=reps, poses_per_s=poses / t)
            res["label_share_of_occupancy"] = res["label"]["seconds_per_call"] / t
        res["composed"] = dict(seconds_per_call=a.elapsed_time(e) / 1e3, iterations=iters,
                               poses_per_s=poses / (a.elapsed_time(e) / 1e3))
        res["speedup"] = res["composed"]["seconds_per_call"] / res["label"]["seconds_per_call"]
        out["workloads"][name] = res
        del sc, words, labels, free, want, per, sizes
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
