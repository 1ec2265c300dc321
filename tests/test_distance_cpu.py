"""Free-space distance without a device: the argument validation of ag_cspace_distance and ag_cspace_descend, and the
references of tests/distance_reference.py that tests/test_distance_gpu.py holds the kernels to."""
import collections

import numpy as np
import pytest

from components_reference import special_images
from distance_reference import descend_numpy, distance_numpy, neighbours


@pytest.fixture(scope="module")
def lib():
    from abstract_gym_b200 import _lib
    return _lib.load()


def test_cspace_distance_argument_errors(lib):
    """every bad argument gets its status before anything touches the device, in the documented order"""
    d = 4096                                 # fake device address
    call = lambda n=1, b1=8, b2=8, wrap=3, bits=d, goals=d, dist=d, md=None: \
        lib.ag_cspace_distance(bits, goals, n, b1, b2, wrap, dist, md, None)
    assert call(n=-1) == -2 and call(b1=0) == -2 and call(b2=0) == -2 and call(b1=-5) == -2
    assert call(n=-1, wrap=9, bits=None, dist=d + 1) == -2                       # shape before everything else
    assert call(b1=46341, b2=46341) == -2 and call(b1=1 << 16, b2=1 << 15) == -2  # b1 * b2 > INT32_MAX - 1
    assert call(b1=1, b2=(1 << 31) - 1, wrap=9) == -2                            # exactly INT32_MAX poses
    assert call(b1=2, b2=(1 << 30) - 1, wrap=9) == -3                            # INT32_MAX - 1 poses: the mode is next
    assert call(n=1 << 40, b1=1 << 15, b2=1 << 15, wrap=9) == -2                 # n_grids * b1 * b2 beyond int64
    assert call(n=1 << 32, b1=1 << 15, b2=1 << 15, wrap=9) == -3                 # 2^62 poses fit: the mode is next
    assert call(wrap=4) == -3 and call(wrap=-1) == -3 and call(wrap=9, bits=None) == -3
    assert call(n=0, bits=None, goals=None, dist=None, md=d + 1) == 0             # nothing to do, nothing touched
    assert call(bits=None) == -1 and call(goals=None) == -1 and call(dist=None) == -1
    assert call(dist=None, bits=d + 2) == -1
    assert call(bits=d + 2) == -4 and call(goals=d + 1) == -4 and call(dist=d + 3) == -4 and call(md=d + 2) == -4


def test_cspace_descend_argument_errors(lib):
    d = 4096
    call = lambda n=1, b1=8, b2=8, wrap=3, m=5, max_len=4, dist=d, start=d, grid=d, path=d, length=d: \
        lib.ag_cspace_descend(dist, n, b1, b2, wrap, start, grid, m, max_len, path, length, None)
    assert call(n=-1) == -2 and call(b1=0) == -2 and call(b2=0) == -2
    assert call(b1=46341, b2=46341, wrap=9) == -2 and call(n=1 << 40, b1=1 << 15, b2=1 << 15, wrap=9) == -2
    assert call(m=-1, wrap=9, dist=None) == -2 and call(max_len=0, wrap=9) == -2 and call(max_len=-3) == -2
    assert call(m=1 << 40, max_len=1 << 24, wrap=9) == -2                        # m * max_len beyond int64
    assert call(m=1 << 40, max_len=1 << 22, wrap=9) == -3
    assert call(wrap=4) == -3 and call(wrap=-2, start=None) == -3
    assert call(m=0, dist=None, start=None, grid=None, path=None, length=None) == 0
    assert call(n=0, m=0) == 0
    for name in ("dist", "start", "grid", "path", "length"):
        assert call(**{name: None}) == -1
    assert call(start=None, grid=d + 4) == -1
    assert call(dist=d + 2) == -4 and call(start=d + 1) == -4 and call(grid=d + 4) == -4
    assert call(path=d + 2) == -4 and call(length=d + 3) == -4


def test_without_device_is_a_cuda_error(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present: valid arguments would launch on the fake addresses")
    for wrap in range(4):
        for md in (None, 8192):
            st = lib.ag_cspace_distance(4096, 4096, 3, 40, 70, wrap, 16384, md, None)
            assert st in (100, 35), st                                          # cudaErrorNoDevice / cudaErrorInsufficientDriver
        st = lib.ag_cspace_descend(4096, 3, 40, 70, wrap, 8192, 16384, 9, 5, 32768, 65536, None)
        assert st in (100, 35), st


def bfs(free, goals, wrap):
    """plain multi-source BFS from the free goals"""
    b1, b2 = free.shape
    dist = np.where(free, -2, -1)
    q = collections.deque()
    for i, j in zip(*np.nonzero(goals & free)):
        dist[i, j] = 0
        q.append((i, j))
    while q:
        x, y = q.popleft()
        for u, v in ((x + 1, y), (x - 1, y), (x, y + 1), (x, y - 1)):
            if wrap & 1:
                u %= b1
            if wrap & 2:
                v %= b2
            if 0 <= u < b1 and 0 <= v < b2 and dist[u, v] == -2:
                dist[u, v] = dist[x, y] + 1
                q.append((u, v))
    return dist


def test_scipy_reference_equals_bfs_random():
    rng = np.random.default_rng(21)
    for _ in range(200):
        b1, b2 = (int(v) for v in rng.integers(1, 41, 2))
        free = rng.random((b1, b2)) < rng.uniform(0.3, 0.95)
        goals = rng.random((b1, b2)) < rng.choice([0.0, 0.002, 0.02, 0.2])
        for wrap in range(4):
            assert np.array_equal(distance_numpy(free, goals, wrap), bfs(free, goals, wrap)), (b1, b2, wrap)


@pytest.mark.parametrize("wrap", range(4))
def test_scipy_reference_equals_bfs_special(wrap):
    for name, free in special_images(14, 18).items():
        for goals in (np.zeros_like(free), np.eye(14, 18, dtype=bool), np.ones_like(free)):
            assert np.array_equal(distance_numpy(free, goals, wrap), bfs(free, goals, wrap)), (name, wrap)
    sp = special_images(14, 18)["spiral"]
    g = np.zeros_like(sp)
    g[0, 0] = True
    if wrap == 0:                                                               # one corridor: 0, 1, 2, ...
        assert sorted(distance_numpy(sp, g, wrap)[sp].tolist()) == list(range(int(sp.sum())))


def test_scipy_reference_keeps_grids_apart():
    rng = np.random.default_rng(5)
    free = rng.random((4, 9, 7)) < 0.7
    free[:, 0, :] = free[:, -1, :] = True
    goals = np.zeros_like(free)
    goals[0, 4, 3] = True
    goals[2] = rng.random((9, 7)) < 0.1
    for wrap in range(4):
        got = distance_numpy(free, goals, wrap)
        for g in range(4):
            assert np.array_equal(got[g], bfs(free[g], goals[g], wrap))


def test_descent_reference_invariants():
    rng = np.random.default_rng(8)
    for trial in range(60):
        b1, b2 = (int(v) for v in rng.integers(1, 30, 2))
        wrap = trial % 4
        free = rng.random((2, b1, b2)) < 0.75
        goals = rng.random((2, b1, b2)) < 0.01
        dist = distance_numpy(free, goals, wrap)
        m = 40
        start = rng.integers(-3, b1 * b2 + 3, m)
        grid = rng.integers(-1, 3, m)
        max_len = int(rng.integers(1, 40))
        path, length = descend_numpy(dist, start, grid, max_len, wrap)
        for q in range(m):
            g, s = int(grid[q]), int(start[q])
            valid = 0 <= g < 2 and 0 <= s < b1 * b2 and dist[g].flat[s] >= 0
            assert length[q] == (min(int(dist[g].flat[s]) + 1, max_len) if valid else 0)
            assert (path[q, length[q]:] == -1).all()
            for k in range(1, length[q]):
                i, j = divmod(int(path[q, k - 1]), b2)
                u, v = divmod(int(path[q, k]), b2)
                assert (u, v) in neighbours(i, j, b1, b2, wrap)                 # adjacent
                assert dist[g, u, v] == dist[g, i, j] - 1 >= 0                  # free, one step closer
                first = next(p for p in neighbours(i, j, b1, b2, wrap) if dist[g][p] == dist[g, i, j] - 1)
                assert first == (u, v)                                          # the first such neighbour
            if valid and length[q] == int(dist[g].flat[s]) + 1:
                assert dist[g].flat[path[q, length[q] - 1]] == 0                # ends on a goal
