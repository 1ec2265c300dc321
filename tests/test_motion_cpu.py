"""Motion checking without a device: ag_check_motion's argument validation, and the reference composition that
tests/test_motion_gpu.py holds the kernel to (move_to_joint_pose's poses + the oracle's collision check)."""

import numpy as np
import pytest

from motion_reference import motion_poses, reference_motion


@pytest.fixture(scope="module")
def lib():
    from abstract_gym_b200 import _lib
    return _lib.load()


def _grid():
    from abstract_gym_b200 import _lib
    g = _lib.Grid()
    g.bits = g.min_x = g.min_y = 256
    g.S, g.words_per_row, g.n_grids, g.grid_stride_words, g.envs_per_grid = 9, 1, 1, 12, 1
    g.side, g.env_size = 0.2, 1.6
    return g


def test_check_motion_argument_errors(lib):
    """every bad argument gets its status before anything touches the device, in ag_collision_check's order"""
    from abstract_gym_b200 import _lib
    p, g = _lib.default_params(), _grid()
    d, al = 4096, 4104                      # fake device addresses: 16-byte aligned and not
    call = lambda m, goal=d, lf=None, engine=_lib.ENGINE_FAST, j1=d, steps=d, fc=d, g=g, p=p: lib.ag_check_motion(
        p, g, j1, d, goal, steps, fc, None, lf, m, 0, engine, None)
    assert call(-1) == -2                                           # m < 0
    assert call(-1, engine=9) == -2                                 # ... before anything else
    assert lib.ag_check_motion(None, g, d, d, d, d, d, None, None, 4, 0, 1, None) == -1
    assert lib.ag_check_motion(p, None, d, d, d, d, d, None, None, 4, 0, 1, None) == -1
    assert call(0) == 0 and call(0, engine=9) == 0                  # m = 0 launches nothing
    assert call(4, j1=None) == -1 and call(4, steps=None) == -1 and call(4, fc=None) == -1 and call(4, goal=None) == -1
    assert call(4, goal=al) == -4 and call(4, lf=al) == -4           # [m][2] arrays are 16-byte aligned
    assert call(4, engine=9) == -3 and call(4, engine=-1) == -3
    bad = _grid()
    bad.words_per_row = 2
    assert call(4, g=bad) == -2                                     # inconsistent grid
    long_links = _lib.default_params()
    long_links.link_1 = 1.5
    assert call(4, p=long_links) == -3                              # outside the FAST engine's error budget


def test_check_motion_without_device_is_a_cuda_error(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present: valid arguments would launch on the fake addresses")
    from abstract_gym_b200 import _lib
    for engine in (_lib.ENGINE_EXACT, _lib.ENGINE_FAST, _lib.ENGINE_BRUTE):
        st = lib.ag_check_motion(_lib.default_params(), _grid(), 4096, 4096, 4096, 4096, 4096, 4096, 4096, 4, 0, engine, None)
        assert st in (100, 35), st                                  # cudaErrorNoDevice / cudaErrorInsufficientDriver


def test_reference_poses_are_move_to_joint_pose(oracle):
    """the composition's last pose is the reference's move_to_joint_pose, bit for bit, and its poses are the
    sequential sum (not start + k * inc)"""
    rng = np.random.default_rng(5)
    for n in (1, 2, 7, 100, 1000):
        start = rng.uniform(-7.0, 7.0, (64, 2))
        goal = rng.uniform(-7.0, 7.0, (64, 2))
        goal[:4] = start[:4]                                       # start == goal
        poses = motion_poses(start, goal, n)
        assert poses.shape == (64, n, 2)
        for i in range(64):
            a, b = oracle.move_to_joint_pose(start[i, 0], start[i, 1], goal[i, 0], goal[i, 1], n)
            assert poses[i, -1, 0] == a and poses[i, -1, 1] == b
        inc = (1.0 / n) * (goal - start)
        step = start + inc
        for k in range(1, min(n, 5)):
            step = step + inc
            assert np.array_equal(poses[:, k], step)
        if n >= 7:
            assert not np.array_equal(poses[:, 6], start + 7 * inc)     # rounding differs from the closed form


def test_reference_motion_semantics(oracle):
    """first collision, first hit and last free pose of the composition on scene_0's map, cross-checked pose by pose"""
    sq, ci = oracle.manual_grid()
    rng = np.random.default_rng(6)
    m = 400
    start = rng.uniform(0.0, 2 * np.pi, (m, 2))
    goal = rng.uniform(0.0, 2 * np.pi, (m, 2))
    steps = rng.choice([-3, 0, 1, 7, 30], m).astype(np.int32)
    fc, fh, lf = reference_motion(oracle, start, goal, steps, [(sq, ci)])
    assert np.array_equal(fc[steps < 1], np.full((steps < 1).sum(), -2))
    assert np.array_equal(lf[steps < 1], start[steps < 1])
    assert (fc > 0).sum() > 20 and (fc == -1).sum() > 20
    for i in np.nonzero(steps >= 1)[0][:60]:
        n = int(steps[i])
        poses = motion_poses(start[i:i + 1], goal[i:i + 1], n)[0]
        hit, fhit, _ = oracle.collision_batch(poses[:, 0].copy(), poses[:, 1].copy(), sq, cell_index=ci)
        k = next((k for k in range(n) if hit[k]), None)
        if k is None:
            assert fc[i] == -1 and fh[i] == -1 and np.array_equal(lf[i], poses[-1])
        else:
            assert fc[i] == k + 1 and fh[i] == fhit[k]
            assert np.array_equal(lf[i], start[i] if k == 0 else poses[k - 1])
