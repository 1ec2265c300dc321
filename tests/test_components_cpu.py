"""Free-space components without a device: ag_cspace_components' argument validation, and the numpy labeller and lookup
rule of tests/components_reference.py that tests/test_components_gpu.py holds the kernels to."""
import collections
import math

import numpy as np
import pytest

from components_reference import component_of_numpy, grid_of_env, label_numpy, special_images


@pytest.fixture(scope="module")
def lib():
    from abstract_gym_b200 import _lib
    return _lib.load()


def test_cspace_components_argument_errors(lib):
    """every bad argument gets its status before anything touches the device, in the documented order"""
    d = 4096                                 # fake device address
    call = lambda n=1, b1=8, b2=8, wrap=3, bits=d, labels=d, nc=None: \
        lib.ag_cspace_components(bits, n, b1, b2, wrap, labels, nc, None)
    assert call(n=-1) == -2 and call(b1=0) == -2 and call(b2=0) == -2 and call(b1=-5) == -2
    assert call(n=-1, wrap=9, bits=None, labels=d + 1) == -2                     # shape before everything else
    assert call(b1=46341, b2=46341) == -2 and call(b1=1 << 16, b2=1 << 15) == -2  # b1 * b2 > INT32_MAX
    assert call(n=1 << 40, b1=1 << 15, b2=1 << 15, wrap=9) == -2                 # n_grids * b1 * b2 beyond int64
    assert call(n=1 << 32, b1=1 << 15, b2=1 << 15, wrap=9) == -3                 # 2^62 poses fit: the mode is next
    assert call(wrap=4) == -3 and call(wrap=-1) == -3 and call(wrap=9, bits=None) == -3
    assert call(n=0, bits=None, labels=None, nc=d + 4) == 0                      # nothing to do, nothing touched
    assert call(bits=None) == -1 and call(labels=None) == -1 and call(labels=None, bits=d + 2) == -1
    assert call(bits=d + 2) == -4 and call(labels=d + 1) == -4 and call(nc=d + 4) == -4


def test_cspace_components_without_device_is_a_cuda_error(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present: valid arguments would launch on the fake addresses")
    for wrap in range(4):
        for nc in (None, 4096):
            st = lib.ag_cspace_components(4096, 3, 40, 70, wrap, 8192, nc, None)
            assert st in (100, 35), st                                          # cudaErrorNoDevice / cudaErrorInsufficientDriver


def bfs(free, wrap):
    """plain BFS from each unlabelled free pose in row-major order: the first pose reached is the component's minimum"""
    b1, b2 = free.shape
    lab = np.full((b1, b2), -1, dtype=np.int64)
    for s in range(b1 * b2):
        i, j = divmod(s, b2)
        if not free[i, j] or lab[i, j] >= 0:
            continue
        lab[i, j] = s
        q = collections.deque([(i, j)])
        while q:
            x, y = q.popleft()
            for u, v in ((x + 1, y), (x - 1, y), (x, y + 1), (x, y - 1)):
                if wrap & 1:
                    u %= b1
                if wrap & 2:
                    v %= b2
                if 0 <= u < b1 and 0 <= v < b2 and free[u, v] and lab[u, v] < 0:
                    lab[u, v] = s
                    q.append((u, v))
    return lab


def test_numpy_labeller_equals_bfs_random():
    rng = np.random.default_rng(11)
    for _ in range(300):
        b1, b2 = (int(v) for v in rng.integers(1, 41, 2))
        f = rng.uniform(0.3, 0.9)
        free = rng.random((b1, b2)) < f
        for wrap in range(4):
            assert np.array_equal(label_numpy(free, wrap), bfs(free, wrap)), (b1, b2, f, wrap)


@pytest.mark.parametrize("wrap", range(4))
def test_numpy_labeller_equals_bfs_special(wrap):
    img = special_images(14, 18)                        # even sizes: no seam joins two checkerboard poses
    for name, free in img.items():
        assert np.array_equal(label_numpy(free, wrap), bfs(free, wrap)), (name, wrap)
    cb = label_numpy(img["checkerboard"], wrap)
    assert np.array_equal(cb[img["checkerboard"]], np.flatnonzero(img["checkerboard"]))   # no diagonal joins
    assert (label_numpy(img["spiral"], wrap)[img["spiral"]] == 0).all()
    c = label_numpy(img["corners"], wrap)
    assert len(np.unique(c[c >= 0])) == {0: 4, 1: 2, 2: 2, 3: 1}[wrap]


def test_numpy_labeller_keeps_grids_apart():
    rng = np.random.default_rng(3)
    free = rng.random((5, 9, 7)) < 0.7
    free[:, 0, :] = free[:, -1, :] = True                # grid g's last row next to grid g+1's first row in memory
    for wrap in range(4):
        got = label_numpy(free, wrap)
        for g in range(5):
            assert np.array_equal(got[g], bfs(free[g], wrap))


def test_component_of_rule():
    """k = floor((q - lo) / step + 0.5) per axis; mod b on a wrapping axis, -1 off a non-wrapping one; NaN / inf -> -1"""
    b1, b2 = 8, 6
    labels = np.arange(2 * b1 * b2, dtype=np.int32).reshape(2, b1, b2)
    st = (2 * math.pi / b1, 2 * math.pi / b2)
    q = np.array([[0.0, 0.0], [st[0] * 0.49, st[1] * 0.51], [-st[0] * 0.6, 2 * math.pi], [1e6, -1e6], [math.nan, 0.0],
                  [0.0, math.inf], [st[0] * 7.4, st[1] * 5.6]])
    grids = np.array([0, 1, 0, 1, 0, 1, 1])
    got = component_of_numpy(labels, q, grids, (0.0, 0.0), st, 3)
    k1 = [0, 0, 7, int(np.fmod(np.floor(1e6 / st[0] + 0.5), b1)), 0, 0, 7]
    k2 = [0, 1, 0, int(np.fmod(np.floor(-1e6 / st[1] + 0.5), b2)) % b2, 0, 0, 0]
    want = [labels[g, a, b] for g, a, b in zip(grids, k1, k2)]
    want[4] = want[5] = -1
    assert got.tolist() == want
    off = component_of_numpy(labels, q, grids, (0.0, 0.0), st, 0)
    assert off.tolist() == [0, 48 + 1, -1, -1, -1, -1, -1]
    assert grid_of_env(6, 3, 2, 4).tolist() == [1, 2, 2, 3, 3, 0]
