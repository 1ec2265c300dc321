"""Free-space components on the device (ag_cspace_components / torch.ops.abstract_gym_b200.cspace_components /
BatchedScene.cspace_components / cspace_component_of) against tests/components_reference.py, bit for bit: the numpy
labeller up to 1024^2 poses per grid, the torch composed form beyond (which the smaller cases hold to numpy first)."""
import math
import os

import numpy as np
import pytest

from components_reference import (component_of_numpy, composed_components, grid_of_env, label_numpy, pack_words,
                                  special_images)

pytestmark = pytest.mark.gpu

ENGINES = ["fast", "exact", "brute"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ag():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import abstract_gym_b200 as ag
    return ag


@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


def scene(ag, torch, grid, n=1, env_id0=0, engine="fast"):
    z = torch.zeros(n, dtype=torch.float64, device="cuda")
    return ag.BatchedScene(ag.BatchedTwoJointRobot(z, z.clone()), grid, engine=engine, env_id0=env_id0)


def op(torch, words, b1, b2, wrap):
    """labels and counts through the torch op"""
    from abstract_gym_b200 import ops
    n = words.numel() // (b1 * ((b2 + 31) // 32))
    labels = torch.empty(n, b1, b2, dtype=torch.int32, device="cuda")
    nc = torch.empty(n, dtype=torch.int64, device="cuda")
    ops.cspace_components(words, b1, b2, wrap, labels, nc)
    return labels, nc


def counts(labels):
    """components per grid of canonical labels: the poses whose label is their own index"""
    lab = np.asarray(labels).reshape(labels.shape[0], -1)
    return (lab == np.arange(lab.shape[1])).sum(axis=1)


def assert_labels(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    want = want.cpu().numpy() if hasattr(want, "cpu") else np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    diff = got != want
    assert not diff.any(), "%s: %d of %d labels differ, first at %s: %d vs %d" % (
        what, diff.sum(), diff.size, np.argwhere(diff)[0], got[diff][0], want[diff][0])


def check_image(torch, free, wrap, what, reference="numpy"):
    """free: bool torch [n, b1, b2] on the device; the op's labels and counts equal the reference's"""
    n, b1, b2 = free.shape
    labels, nc = op(torch, pack_words(~free), b1, b2, wrap)
    if reference == "numpy":
        want = label_numpy(free.cpu().numpy(), wrap)
    else:
        want = composed_components(free, wrap)[0].cpu().numpy()
    assert_labels(labels, want, what)
    assert np.array_equal(nc.cpu().numpy(), counts(want)), what
    return labels, nc


FRACTIONS = [0.3, 0.55, 0.593, 0.65, 0.9]


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (37, 1), (31, 33), (256, 256), (1000, 1000), (4096, 4096)])
def test_synthetic_images(ag, torch_, shape):
    torch = torch_
    b1, b2 = shape
    gen = torch.Generator(device="cuda").manual_seed(b1 * 7919 + b2)
    for f in FRACTIONS:
        free = torch.rand(1, b1, b2, device="cuda", generator=gen) < f
        for wrap in range(4):
            check_image(torch, free, wrap, "%dx%d f=%g wrap=%d" % (b1, b2, f, wrap),
                        "numpy" if b1 * b2 <= 1 << 20 else "composed")


def test_composed_form_equals_numpy(ag, torch_):
    """the 4096^2 cases' reference, held to numpy at 1024^2 near the percolation threshold"""
    torch = torch_
    free = torch.rand(2, 1024, 1024, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) < 0.6
    for wrap in range(4):
        assert_labels(composed_components(free, wrap)[0], label_numpy(free.cpu().numpy(), wrap), "composed %d" % wrap)


@pytest.mark.parametrize("shape", [(6, 6), (300, 500), (1000, 1000)])
def test_adversarial_images(ag, torch_, shape):
    torch = torch_
    b1, b2 = shape
    for name, img in special_images(b1, b2).items():
        free = torch.as_tensor(img, device="cuda")[None]
        for wrap in range(4):
            labels, nc = check_image(torch, free, wrap, "%s %dx%d wrap=%d" % (name, b1, b2, wrap))
            lab = labels[0].cpu().numpy()
            if name == "spiral":
                assert (lab[img] == 0).all() and int(nc) == 1
            elif name == "checkerboard":                 # even sizes: every free pose is its own component
                assert np.array_equal(lab[img], np.flatnonzero(img)) and int(nc) == img.sum()
            elif name == "all_free":
                assert (lab == 0).all() and int(nc) == 1
            elif name == "all_colliding":
                assert (lab == -1).all() and int(nc) == 0
            elif name == "seams":
                assert (lab[0, 3] == lab[-1, 3]) == bool(wrap & 1)
                assert (lab[b1 // 2, 0] == lab[b1 // 2, -1]) == bool(wrap & 2)
                assert int(nc) == 4 - bool(wrap & 1) - bool(wrap & 2)
            elif name == "corners":
                assert int(nc) == {0: 4, 1: 2, 2: 2, 3: 1}[wrap]


def test_padding_bits_are_ignored(ag, torch_):
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(4)
    for b1, b2 in ((37, 45), (100, 100), (5, 1), (64, 33)):
        free = torch.rand(3, b1, b2, device="cuda", generator=gen) < 0.6
        words = pack_words(~free)
        garbage = torch.randint(-2 ** 31, 2 ** 31, words.shape, dtype=torch.int64, device="cuda", generator=gen)
        if b2 % 32:
            pad = (~((1 << (b2 % 32)) - 1)) & 0xFFFFFFFF
            mask = torch.zeros_like(garbage)
            mask[..., -1] = pad - (1 << 32) if pad >= 1 << 31 else pad
            dirty = (words.to(torch.int64) | (garbage & mask)).to(torch.int32)   # int64 -> int32 keeps the low 32 bits
            assert not torch.equal(dirty, words)
        else:
            dirty = words
        for wrap in range(4):
            clean, nc = op(torch, words, b1, b2, wrap)
            got, nc2 = op(torch, dirty, b1, b2, wrap)
            assert_labels(got, clean, "padding %dx%d wrap %d" % (b1, b2, wrap))
            assert torch.equal(nc, nc2)
            assert_labels(clean, label_numpy(free.cpu().numpy(), wrap), "padding reference")


def test_many_grids(ag, torch_):
    """1024 grids of 256^2 with distinct content; the last row of every grid and the first of the next are free, next
    to each other in memory: grids never join"""
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(6)
    f = torch.linspace(0.3, 0.9, 1024, device="cuda").view(-1, 1, 1)
    free = torch.rand(1024, 256, 256, device="cuda", generator=gen) < f
    free[:, 0, :] = free[:, -1, :] = True
    for wrap in range(4):
        labels, nc = check_image(torch, free, wrap, "1024 x 256^2 wrap %d" % wrap, "composed")
        some = [0, 1, 511, 1023]
        assert_labels(labels[some], label_numpy(free[some].cpu().numpy(), wrap), "1024 x 256^2 numpy")
        assert (labels[:, -1, :] >= 0).all() and (labels[1:, 0, 0] == 0).all()


def bool_occupancy_reference(sc, b1, b2, lo, step, wrap, engine, reference):
    img = sc.cspace_occupancy(b1, b2, lo=lo, step=step, engine=engine)
    if reference == "numpy":
        return img, label_numpy(~img.cpu().numpy(), wrap)
    return img, composed_components(~img, wrap)[0].cpu().numpy()


def check_scene(sc, b1, b2, engine, lo=(0.0, 0.0), step=None, wrap=None, what=""):
    import torch
    st = (2 * math.pi / b1, 2 * math.pi / b2) if step is None else step
    w = (3 if step is None else 0) if wrap is None else int(wrap[0]) | int(wrap[1]) << 1
    labels, nc = sc.cspace_components(b1, b2, lo=lo, step=step, wrap=wrap, count=True, engine=engine)
    img, want = bool_occupancy_reference(sc, b1, b2, lo, st, w, engine, "numpy" if b1 * b2 <= 1 << 20 else "composed")
    assert labels.dtype == torch.int32 and nc.dtype == torch.int64
    assert labels.shape == img.shape and nc.shape == (img.shape[0],)
    assert_labels(labels, want, "%s %s" % (what, engine))
    assert torch.equal(labels < 0, img), what                   # -1 exactly where a pose collides
    assert np.array_equal(nc.cpu().numpy(), counts(want)), what
    return labels


@pytest.mark.parametrize("b", [1024, 4096])
def test_scene0_default_lattice(ag, torch_, b):
    sc = scene(ag, torch_, ag.OccupancyGrid(size=9, random_obstacle=False))
    for engine in ENGINES:
        check_scene(sc, b, b, engine, what="scene_0 %d^2" % b)
    print("scene_0 %d^2: %d components" % (b, int(sc.cspace_components(b, count=True)[1])))


def test_config4_grid(ag, torch_):
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    g.load_from_matrix((np.random.default_rng(4).random((1024, 1024)) < 0.002).astype(np.uint8))
    sc = scene(ag, torch_, g)
    for engine in ENGINES:
        b = 256 if engine == "brute" else 1024
        check_scene(sc, b, b, engine, what="config 4 %d^2" % b)


def test_config5_grids(ag, torch_):
    torch = torch_
    grid = ag.BatchedOccupancyGrid.random(64, 256, 0.008, 256, device="cuda",
                                          generator=torch.Generator(device="cuda").manual_seed(5), clear_base_cells=2)
    sc = scene(ag, torch, grid)
    for engine in ENGINES:
        check_scene(sc, 256, 256, engine, what="64 config-5 grids")


def test_offset_lattice_without_wrap(ag, torch_):
    sc = scene(ag, torch_, ag.OccupancyGrid(size=9, random_obstacle=False))
    st = (2 * math.pi / 512, 2 * math.pi / 384)
    for engine in ENGINES:
        a = check_scene(sc, 512, 384, engine, lo=(0.5 * st[0], 0.5 * st[1]), step=st, wrap=(False, False),
                        what="offset, no wrap")
        b = sc.cspace_components(512, 384, lo=(0.5 * st[0], 0.5 * st[1]), step=st, engine=engine)   # wrap=None: none
        assert torch_.equal(a, b)


def test_graph_capture(ag, torch_):
    torch = torch_
    sc = scene(ag, torch, ag.OccupancyGrid(size=9, random_obstacle=False))
    want, want_nc = sc.cspace_components(1024, count=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            labels, nc = sc.cspace_components(1024, count=True)
    for _ in range(2):                                       # replays rewrite the counts
        g.replay()
        torch.cuda.synchronize()
        assert_labels(labels, want, "captured")
        assert torch.equal(nc, want_nc)


def test_torch_op_equals_object_api(ag, torch_):
    torch = torch_
    from abstract_gym_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(9)
    grid = ag.BatchedOccupancyGrid.random(3, 48, 0.02, envs_per_grid=256, device="cuda", generator=gen)
    sc = scene(ag, torch, grid)
    b1, b2 = 70, 90
    words = sc.cspace_occupancy(b1, b2, packed=True)
    for wrap in range(4):
        want, want_nc = sc.cspace_components(b1, b2, wrap=(bool(wrap & 1), bool(wrap & 2)), count=True)
        labels, nc = op(torch, words, b1, b2, wrap)
        assert_labels(labels, want, "torch op wrap %d" % wrap)
        assert torch.equal(nc, want_nc)
        again = torch.empty_like(labels)
        ops.cspace_components(words, b1, b2, wrap, again, None)
        assert_labels(again, want, "torch op, no counts")
    labels = torch.empty(3, b1, b2, dtype=torch.int32, device="cuda")
    for bad in (lambda: ops.cspace_components(words, b1, b2, 0, labels[:2], None),
                lambda: ops.cspace_components(words[:, :, :2].contiguous(), b1, b2, 0, labels, None),
                lambda: ops.cspace_components(words, b1, b2, 0, labels, torch.empty(2, dtype=torch.int64, device="cuda")),
                lambda: ops.cspace_components(words, b1, b2, 4, labels, None),
                lambda: ops.cspace_components(words, b1, b2, 0, labels.to(torch.int64), None)):
        with pytest.raises(RuntimeError):
            bad()
    with pytest.raises((NotImplementedError, RuntimeError)):
        ops.cspace_components(words.cpu(), b1, b2, 0, labels.cpu(), None)


@pytest.mark.parametrize("wrap", [None, (False, False), (True, False)])
def test_component_of(ag, torch_, wrap):
    """the lookup equals the numpy rule on a multi-grid scene with env_id0 != 0: far-away, negative, NaN and infinite
    angles, and poses off a non-wrapping lattice"""
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(12)
    grid = ag.BatchedOccupancyGrid.random(3, 31, 0.05, envs_per_grid=5, device="cuda", generator=gen)
    n, env_id0 = 40, 7
    sc = scene(ag, torch, grid, n=n, env_id0=env_id0)
    b1, b2 = 64, 48
    if wrap is None:
        lo, step, w = (0.0, 0.0), None, 3
        st = (2 * math.pi / b1, 2 * math.pi / b2)
    else:
        lo, st, w = (-1.0, 0.3), (0.05, 0.07), int(wrap[0]) | int(wrap[1]) << 1
        step = st
    labels = sc.cspace_components(b1, b2, lo=lo, step=step, wrap=wrap)
    rng = np.random.default_rng(3)
    q = rng.uniform(-8.0, 8.0, (n, 2))
    q[0] = (1e7, -3e5)
    q[1] = (-1e15, 2.5e9)
    q[2] = (math.nan, 0.1)
    q[3] = (0.2, math.inf)
    q[4] = (-math.inf, math.nan)
    q[5] = (lo[0] - 0.49 * st[0], lo[1] + (b2 - 0.51) * st[1])           # just inside the lattice's ends
    q[6] = (lo[0] - 0.51 * st[0], lo[1] + (b2 - 0.49) * st[1])           # just outside
    q[7] = (1e300, -1e300)
    sc.robot.joint_1.copy_(torch.as_tensor(rng.uniform(0, 7, n), device="cuda"))
    sc.robot.joint_2.copy_(torch.as_tensor(rng.uniform(-7, 0, n), device="cuda"))
    grids = grid_of_env(n, env_id0, 5, 3)
    lab = labels.cpu().numpy()
    got = sc.cspace_component_of(labels, torch.as_tensor(q, device="cuda"), lo=lo, step=step, wrap=wrap)
    assert got.dtype == torch.int32 and got.shape == (n,)
    want = component_of_numpy(lab, q, grids, lo, st, w)
    assert np.array_equal(got.cpu().numpy(), want), (got.cpu().numpy(), want)
    assert (want[2:5] == -1).all() and (want >= 0).any()
    cur = np.stack([sc.robot.joint_1.cpu().numpy(), sc.robot.joint_2.cpu().numpy()], axis=1)
    assert np.array_equal(sc.cspace_component_of(labels, lo=lo, step=step, wrap=wrap).cpu().numpy(),
                          component_of_numpy(lab, cur, grids, lo, st, w))
    m = 7                                                                  # M != N
    assert np.array_equal(sc.cspace_component_of(labels, torch.as_tensor(q[:m], device="cuda"), lo=lo, step=step,
                                                 wrap=wrap).cpu().numpy(),
                          component_of_numpy(lab, q[:m], grid_of_env(m, env_id0, 5, 3), lo, st, w))


_DEBUG_CHILD = r'''
import sys
import numpy as np, torch
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import abstract_gym_b200 as ag
from abstract_gym_b200 import _lib, ops
from components_reference import label_numpy, pack_words, special_images
assert _lib.lib_path().endswith("_debug.so"), _lib.lib_path()
gen = torch.Generator(device="cuda").manual_seed(1)
cases = [torch.rand(3, 300, 500, device="cuda", generator=gen) < 0.6,
         torch.rand(64, 64, 70, device="cuda", generator=gen) < 0.593,
         torch.as_tensor(special_images(130, 260)["spiral"], device="cuda")[None]]
for free in cases:
    n, b1, b2 = free.shape
    words = pack_words(~free)
    for wrap in range(4):
        labels = torch.empty(n, b1, b2, dtype=torch.int32, device="cuda")
        nc = torch.empty(n, dtype=torch.int64, device="cuda")
        ops.cspace_components(words, b1, b2, wrap, labels, nc)
        want = label_numpy(free.cpu().numpy(), wrap)
        assert np.array_equal(labels.cpu().numpy(), want), (free.shape, wrap)
        per = want.reshape(n, -1)
        assert np.array_equal(nc.cpu().numpy(), (per == np.arange(per.shape[1])).sum(axis=1))
z = torch.zeros(1, dtype=torch.float64, device="cuda")
sc = ag.BatchedScene(ag.BatchedTwoJointRobot(z, z.clone()), ag.OccupancyGrid(size=9, random_obstacle=False))
img = sc.cspace_occupancy(256)
assert np.array_equal(sc.cspace_components(256).cpu().numpy(), label_numpy(~img.cpu().numpy(), 3))
print("debug components ok")
'''


def test_debug_bounds_build_components(ag, torch_):
    """the -DAG_DEBUG_BOUNDS library gives the reference's labels (child process); each k_ccl_* kernel of it carries the
    index traps and the release library none (read from the machine code: no test sets a trap off)"""
    import subprocess
    import sys
    from abstract_gym_b200 import build as ag_build
    from test_gpu_parity import _traps_per_kernel
    lib = ag_build.build_debug()
    code = _DEBUG_CHILD % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, AG_LIB_PATH=lib), stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "debug components ok" in r.stdout, r.stdout[-3000:]
    debug, release = _traps_per_kernel(lib), _traps_per_kernel(ag_build.LIB)
    kernels = [k for k in debug if "k_ccl_" in k]
    assert len(kernels) == 3 and all(debug[k] > 0 for k in kernels), {k: debug[k] for k in kernels}
    assert all(release[k] == 0 for k in kernels)
