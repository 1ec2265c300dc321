"""Time of one batched env step: BatchedScene.step (ag_step) and a captured VectorEnv.step (ag_step_obs), the two entry
points of the single-step kernel k_step.  Prints one JSON line: the card and its power limit, and per row the seconds
per call, env-steps/s and a digest of the outputs of a seeded run.

    python tools/step_bench.py [--envs 1048576] [--min-window 0.5]

Rows (2^20 envs by default; actions (u - 0.5) * 0.1 per joint, torch seed 1):
  scene0_fast_f64, scene0_fast_f32, scene0_exact_f64  BatchedScene.step on scene_0's 9x9 map
  c5_fast_f64                                         BatchedScene.step on bench.py's config-5 grid set: 1024 maps of
                                                      256x256, Bernoulli(0.008), base cells kept free, 1024 envs per map
  vec_fast, vec_fast_crop9                            VectorEnv.step replayed from its CUDA graph, scene_0, FAST, auto-reset,
                                                      without and with a 9x9 occupancy crop
Each row first runs 8 steps with distinct seeded actions and hashes what they leave (joints, sticky reward and flags,
statistics; for VectorEnv also the observations, step outputs, counters and crop): two builds of the library compute the
same thing when their digests agree.  The timed steps then repeat one action, after a warm-up step.  The per-step state
(about 40 MB at 2^20 envs) stays in the 126 MB L2 across calls, as it does for a training loop that steps every call.
Run it against another build of the library with AG_LIB_PATH=<that .so>.
"""
import argparse
import hashlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import abstract_gym_b200 as ag                                   # noqa: E402
from cspace_bench import gpu_info, timed                         # noqa: E402

CHECK_STEPS = 8


def digest(tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def actions(n, steps, dev):
    gen = torch.Generator(device=dev).manual_seed(1)
    return [(torch.rand(n, 2, dtype=torch.float64, device=dev, generator=gen) - 0.5) * 0.1 for _ in range(steps)]


def scene_row(n, dev, grid, engine, dtype):
    robot = ag.BatchedTwoJointRobot.random(n, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    sc = ag.BatchedScene(robot, grid, engine=engine, seed=3)
    acts = [a.to(dtype) for a in actions(n, CHECK_STEPS, dev)]
    for a in acts:
        sc.step(a)
    d = digest([sc.robot.joint_1, sc.robot.joint_2, sc.step_reward, sc.flags, sc.stats])
    return (lambda: sc.step(acts[-1])), d


def vector_row(n, dev, crop):
    env = ag.VectorEnv(n, device=dev, seed=4, engine="fast", crop_size=crop)
    env.reset()
    env.capture()
    acts = actions(n, CHECK_STEPS, dev)
    for a in acts:
        obs, reward, term, _, info = env.step(a)
    sc = env.scene
    d = digest([obs, reward, term, info["collision"], info["final_obs"], sc.robot.joint_1, sc.robot.joint_2,
                sc.step_reward, sc.flags, sc.reset_ctr, sc.ep_len, sc.stats] + ([info["crop"]] if crop else []))
    return (lambda: env.step(acts[-1])), d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds of timed steps per row")
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    n = args.envs
    scene0 = ag.OccupancyGrid(size=9, random_obstacle=False)
    c5 = ag.BatchedOccupancyGrid.random(1024, 256, 0.008, 1024, device=dev,
                                        generator=torch.Generator(device=dev).manual_seed(5), clear_base_cells=2)
    rows = {
        "scene0_fast_f64": lambda: scene_row(n, dev, scene0, "fast", torch.float64),
        "scene0_fast_f32": lambda: scene_row(n, dev, scene0, "fast", torch.float32),
        "scene0_exact_f64": lambda: scene_row(n, dev, scene0, "exact", torch.float64),
        "c5_fast_f64": lambda: scene_row(n, dev, c5, "fast", torch.float64),
        "vec_fast": lambda: vector_row(n, dev, 0),
        "vec_fast_crop9": lambda: vector_row(n, dev, 9),
    }
    out = dict(metric="one batched env step: seconds per call and env-steps/s", gpu=gpu_info(), envs=n,
               lib=os.environ.get("AG_LIB_PATH") or "in-tree", rows={})
    for name, make in rows.items():
        fn, d = make()
        t, reps = timed(fn, args.min_window)
        out["rows"][name] = dict(seconds_per_call=t, env_steps_per_s=n / t, reps=reps, digest=d)
        del fn
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
