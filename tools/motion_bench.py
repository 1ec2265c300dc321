"""Throughput of batched motion checking (BatchedScene.check_motion, kernel k_check_motion) against the composed form a
user would otherwise write: per step a torch add on the joints, then ag_collision_check over all motions.  Both forms
must give identical first_collision and last_free (asserted).  Prints one JSON line.

    python tools/motion_bench.py [--min-window 0.5] [--quick]

Workloads (the issue's): scene_0's 9x9 map with 2^20 motions x 100 steps (starts collision-free, goals uniform in
[0, 2 pi)), the same with steps uniform in 1..1000, one 1024^2 Bernoulli(0.002) map with 2^16 x 100, and a distinct
256^2 Bernoulli(0.008) map per 256 motions (bench.py's c5 grids) with 2^20 x 100.  A pose check is one collision test
of one pose: sum over motions of first_collision if the motion collides, else steps.  Lane utilisation: pose checks
over 32 x the longest walk of every 32 consecutive motions (the lanes of one warp of the kernel).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import abstract_gym_b200 as ag                        # noqa: E402
from abstract_gym_b200 import _lib                    # noqa: E402
from abstract_gym_b200._device import ptr, stream_ptr  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def composed(sc, j1, j2, goal, steps):
    """per step: q += inc (torch), ag_collision_check of all motions, bookkeeping (torch)"""
    lib, g, p, dev = sc._lib, sc.grid.c_struct(), sc.params(), sc.device
    m = j1.numel()
    alpha = 1.0 / steps.to(torch.float64)
    inc1, inc2 = alpha * (goal[:, 0] - j1), alpha * (goal[:, 1] - j2)
    q1, q2 = j1.clone(), j2.clone()
    fc = torch.where(steps >= 1, -1, -2).to(torch.int32)
    hit = torch.empty(m, dtype=torch.uint8, device=dev)
    for k in range(1, int(steps.max().item()) + 1):
        n1, n2 = q1 + inc1, q2 + inc2
        _lib.check(lib.ag_collision_check(p, g, ptr(n1), ptr(n2), ptr(hit), None, m, sc.env_id0, sc.engine, stream_ptr(dev)),
                   "ag_collision_check")
        live = (fc == -1) & (steps >= k)
        h = hit != 0
        fc = torch.where(live & h, k, fc).to(torch.int32)
        move = live & ~h
        q1, q2 = torch.where(move, n1, q1), torch.where(move, n2, q2)
    return fc, torch.stack([q1, q2], dim=1)


def timed(fn, min_window):
    fn()                                                     # warm-up (and the map's first build)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, elapsed = 1, 0.0
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


def workload(name, m, dev, gen):
    rng = np.random.default_rng(3)
    steps = torch.full((m,), 100, dtype=torch.int32, device=dev)
    if name.startswith("scene0"):
        grid = ag.OccupancyGrid(size=9, random_obstacle=False)
        if name == "scene0_ragged":
            steps = torch.randint(1, 1001, (m,), dtype=torch.int32, device=dev, generator=gen)
    elif name == "c4":
        grid = ag.OccupancyGrid(size=9, random_obstacle=False)
        grid.load_from_matrix((rng.random((1024, 1024)) < 0.002).astype(np.uint8))
    else:
        grid = ag.BatchedOccupancyGrid.random(max(1, m // 256), 256, 0.008, 256, device=dev,
                                              generator=torch.Generator(device=dev).manual_seed(5), clear_base_cells=2)
    robot = ag.BatchedTwoJointRobot.random(m, device=dev, generator=gen)
    sc = ag.BatchedScene(robot, grid, engine="fast")
    sc.random_valid_pose()                                   # collision-free starts
    goal = torch.rand(m, 2, dtype=torch.float64, device=dev, generator=gen) * (2 * np.pi)
    return sc, goal, steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds of timed launches per form and workload")
    ap.add_argument("--quick", action="store_true", help="1/64 of the motions (a smoke run)")
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    gen = torch.Generator(device=dev).manual_seed(11)
    div = 64 if args.quick else 1
    out = dict(metric="motion checking: motions/s and pose-checks/s, k_check_motion vs per-step torch add + ag_collision_check",
               gpu=gpu_info(), workloads={})
    for name, m in (("scene0", 1 << 20), ("scene0_ragged", 1 << 20), ("c4", 1 << 16), ("c5", 1 << 20)):
        m //= div
        sc, goal, steps = workload(name, m, dev, gen)
        j1, j2 = sc.robot.joint_1, sc.robot.joint_2
        res = {}
        fc, extra = sc.check_motion(goal, steps=steps, last_free=True)
        cfc, clf = composed(sc, j1, j2, goal, steps)
        assert torch.equal(fc, cfc), "%s: first_collision differs in %d motions" % (name, int((fc != cfc).sum()))
        assert torch.equal(extra["last_free"], clf), "%s: last_free differs" % name
        checks = torch.where(fc > 0, fc, torch.where(fc == -1, steps, torch.zeros_like(steps))).to(torch.int64)
        pose_checks = int(checks.sum().item())
        per_warp = checks[: m - m % 32].reshape(-1, 32)
        util = float(per_warp.sum().item()) / max(1.0, float(32 * per_warp.max(dim=1).values.sum().item()))
        for form, fn in (("kernel", lambda: sc.check_motion(goal, steps=steps)),
                         ("composed", lambda: composed(sc, j1, j2, goal, steps))):
            t, reps = timed(fn, args.min_window)
            res[form] = dict(seconds_per_call=t, reps=reps, motions_per_s=m / t, pose_checks_per_s=pose_checks / t)
        res.update(motions=m, pose_checks=pose_checks, collided=int((fc > 0).sum().item()), lane_utilisation=util,
                   speedup=res["composed"]["seconds_per_call"] / res["kernel"]["seconds_per_call"])
        out["workloads"][name] = res
        del sc, goal, steps, fc, extra, cfc, clf
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
