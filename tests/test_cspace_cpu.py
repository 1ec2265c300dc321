"""Configuration-space occupancy without a device: ag_cspace_occupancy's argument validation, and the reference lattice
and oracle composition that tests/test_cspace_gpu.py holds the kernel to (tests/cspace_reference.py)."""
import math

import numpy as np
import pytest

from cspace_reference import default_step, lattice, oracle_image, pack


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


def test_cspace_occupancy_argument_errors(lib):
    """every bad argument gets its status before anything touches the device, in the documented order"""
    from abstract_gym_b200 import _lib
    p, g = _lib.default_params(), _grid()
    d = 4096                                 # fake device address
    call = lambda b1=8, b2=8, lo1=0.0, st1=0.1, lo2=0.0, st2=0.1, bits=d, fc=None, engine=_lib.ENGINE_FAST, p=p, g=g: \
        lib.ag_cspace_occupancy(p, g, lo1, st1, b1, lo2, st2, b2, bits, fc, engine, None)
    assert call(b1=0) == -2 and call(b2=0) == -2 and call(b1=-3) == -2          # b1, b2 >= 1
    assert call(b1=0, p=None, engine=9) == -2                                   # ... before anything else
    assert call(p=None) == -1 and call(g=None) == -1
    bad = _grid()
    bad.words_per_row = 2
    assert call(g=bad) == -2                                                    # inconsistent grid
    bad = _grid()
    bad.bits = None
    assert call(g=bad) == -1
    long_links = _lib.default_params()
    long_links.link_1 = 1.5
    assert call(p=long_links, lo1=math.inf) == -3                               # outside the FAST engine's error budget
    for kw in (dict(lo1=math.nan), dict(st1=math.inf), dict(lo2=-math.inf), dict(st2=math.nan)):
        assert call(bits=None, **kw) == -2                                      # lo, step finite, before the pointers
    many = _grid()
    many.n_grids, many.envs_per_grid = 1 << 30, 256
    assert call(g=many, b1=1 << 30, b2=1 << 30, bits=None) == -2                # n_grids * b1 * W overflows int64
    assert call(bits=None) == -1
    assert call(bits=d + 2) == -4 and call(fc=d + 4) == -4                      # word / int64 alignment
    assert call(engine=9, fc=d + 4) == -4 and call(engine=9) == -3 and call(engine=-1) == -3


def test_cspace_occupancy_without_device_is_a_cuda_error(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is present: valid arguments would launch on the fake addresses")
    from abstract_gym_b200 import _lib
    for engine in (_lib.ENGINE_EXACT, _lib.ENGINE_FAST, _lib.ENGINE_BRUTE):
        for fc in (None, 4096):
            st = lib.ag_cspace_occupancy(_lib.default_params(), _grid(), 0.0, 0.1, 8, 0.0, 0.1, 40, 4096, fc, engine, None)
            assert st in (100, 35), st                                          # cudaErrorNoDevice / cudaErrorInsufficientDriver


def test_lattice_is_lo_plus_i_times_step():
    """the test-side lattice is lo + i * step with one rounding per operation (no FMA, no accumulation)"""
    for lo, step, b in ((0.0, default_step(4096), 4096), (0.5 * default_step(512), default_step(512), 512),
                        (2.0 ** 21, -0.37, 1000), (-1.234567, 1e-3, 777)):
        q = lattice(lo, step, b)
        assert q.dtype == np.float64 and q.shape == (b,)
        assert all(q[i] == lo + float(i) * step for i in range(b))
    assert default_step(7) == 2.0 * math.pi / 7
    # the axis rows of a default lattice: q1 = 0 exactly, the others within a few ulp of pi/2, pi, 3 pi/2
    q = lattice(0.0, default_step(1024), 1024)
    assert q[0] == 0.0
    for k, ang in ((256, math.pi / 2), (512, math.pi), (768, 1.5 * math.pi)):
        assert abs(q[k] - ang) <= 4 * math.ulp(ang)


def test_pack_bit_order():
    rng = np.random.default_rng(4)
    for b2 in (1, 31, 32, 33, 100):
        img = rng.random((3, 5, b2)) < 0.5
        w = pack(img)
        assert w.dtype == np.uint32 and w.shape == (3, 5, (b2 + 31) // 32)
        for j in range(b2):
            assert np.array_equal((w[..., j // 32] >> np.uint32(j % 32)) & 1, img[..., j].astype(np.uint32))
        pad = w[..., -1] >> np.uint32(b2 % 32) if b2 % 32 else np.zeros_like(w[..., -1])
        assert not pad.any()                                                    # padding bits are zero


@pytest.mark.parametrize("offset", [0.0, 0.5])
def test_oracle_image_is_collision_batch_pose_by_pose(oracle, offset):
    """the composition's image of a small scene_0 lattice, against the oracle called one pose at a time"""
    sq, ci = oracle.manual_grid()
    b1, b2 = 24, 20
    st = (default_step(b1), default_step(b2))
    lo = (offset * st[0], offset * st[1])
    img = oracle_image(oracle, (sq, ci), lo, st, b1, b2)
    assert img.shape == (b1, b2) and 0 < img.sum() < img.size
    for i in range(b1):
        for j in range(b2):
            hit, _, _ = oracle.collision_batch(np.array([lo[0] + i * st[0]]), np.array([lo[1] + j * st[1]]), sq,
                                               want_first_hit=False)
            assert bool(hit[0]) == img[i, j], (i, j)
