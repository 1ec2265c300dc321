"""The reference composition of a batched motion check, on the CPU oracle: move_to_joint_pose's poses
(robot/two_joint_robot.py:49-62) built with numpy and Scene.collision_check (scenario/scene_0.py:60-76) at each of
them.  tests/test_motion_cpu.py checks this composition itself; tests/test_motion_gpu.py checks the kernel against it."""
import numpy as np


def motion_poses(start, goal, n):
    """[k,2] starts and goals, n >= 1 increments -> poses 1..n as [k,n,2]: alpha = 1.0/n, inc = alpha*(goal - start),
    pose_k = pose_{k-1} + inc.  np.cumsum is np.add.accumulate, a sequential sum along each row."""
    start, goal = np.asarray(start, np.float64), np.asarray(goal, np.float64)
    alpha = 1.0 / n
    inc = alpha * (goal - start)
    seq = np.concatenate([start[:, None, :], np.broadcast_to(inc[:, None, :], (len(start), n, 2))], axis=1)
    return np.cumsum(seq, axis=1)[:, 1:, :]


def reference_motion(orc, start, goal, steps, grids, grid_of=None):
    """(first_collision [m] int32, first_hit [m] int32, last_free [m,2] float64) of every motion.
    grids: list of (squares, cell_index) from the oracle; grid_of: [m] index into it (default: all grid 0)."""
    start, goal = np.asarray(start, np.float64).reshape(-1, 2), np.asarray(goal, np.float64).reshape(-1, 2)
    steps = np.asarray(steps, np.int64).reshape(-1)
    m = len(start)
    grid_of = np.zeros(m, np.int64) if grid_of is None else np.asarray(grid_of, np.int64)
    fc = np.full(m, -2, np.int32)
    fh = np.full(m, -1, np.int32)
    lf = start.copy()
    for gi, (sq, ci) in enumerate(grids):
        for n in np.unique(steps[(steps >= 1) & (grid_of == gi)]):
            idx = np.nonzero((steps == n) & (grid_of == gi))[0]
            poses = motion_poses(start[idx], goal[idx], int(n))
            k = len(idx)
            hit, fhit, _ = orc.collision_batch(poses[..., 0].ravel(), poses[..., 1].ravel(), sq, cell_index=ci)
            hit = hit.reshape(k, n) != 0
            fhit = fhit.reshape(k, n)
            coll = hit.any(axis=1)
            first = np.argmax(hit, axis=1)
            rows = np.arange(k)
            fc[idx] = np.where(coll, first + 1, -1)
            fh[idx] = np.where(coll, fhit[rows, first], -1)
            before = np.where((first > 0)[:, None], poses[rows, np.maximum(first - 1, 0)], start[idx])
            lf[idx] = np.where(coll[:, None], before, poses[:, -1])
    return fc, fh, lf
