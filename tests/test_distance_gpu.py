"""Free-space distance and lattice descent on the device (ag_cspace_distance / ag_cspace_descend, their torch ops,
BatchedScene.cspace_distance / cspace_distance_of / cspace_path) against tests/distance_reference.py, bit for bit: the
scipy BFS up to 1024^2 poses per grid, the composed torch BFS beyond (which is held to scipy at 1024^2 first)."""
import math
import os

import numpy as np
import pytest

from components_reference import grid_of_env, pack_words, special_images
from distance_reference import composed_distance, descend_numpy, distance_numpy

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


def op(torch, words, goal_words, b1, b2, wrap):
    """distances and per-grid maxima through the torch op"""
    from abstract_gym_b200 import ops
    n = words.numel() // (b1 * ((b2 + 31) // 32))
    dist = torch.empty(n, b1, b2, dtype=torch.int32, device="cuda")
    md = torch.empty(n, dtype=torch.int32, device="cuda")
    ops.cspace_distance(words, goal_words, b1, b2, wrap, dist, md)
    return dist, md


def maxima(dist):
    d = np.asarray(dist).reshape(dist.shape[0], -1)
    return np.where((d >= 0).any(axis=1), d.max(axis=1), -1)


def assert_dist(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    want = want.cpu().numpy() if hasattr(want, "cpu") else np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    diff = got != want
    assert not diff.any(), "%s: %d of %d distances differ, first at %s: %d vs %d" % (
        what, diff.sum(), diff.size, np.argwhere(diff)[0], got[diff][0], want[diff][0])


def check_image(torch, free, goals, wrap, what, reference="numpy", goal_words=None):
    """free, goals: bool torch [n, b1, b2]; the op's distances and maxima equal the reference's"""
    n, b1, b2 = free.shape
    dist, md = op(torch, pack_words(~free), pack_words(goals) if goal_words is None else goal_words, b1, b2, wrap)
    if reference == "numpy":
        want = distance_numpy(free.cpu().numpy(), goals.cpu().numpy(), wrap)
    else:
        want = composed_distance(free, goals, wrap)[0].cpu().numpy()
    assert_dist(dist, want, what)
    assert np.array_equal(md.cpu().numpy(), maxima(want)), what
    return dist, md


def goal_sets(torch, free, gen):
    """0, 1 and many goals, some on colliding poses"""
    n, b1, b2 = free.shape
    one = torch.zeros_like(free)
    one.view(n, -1)[:, (b1 * b2) // 3] = True
    many = torch.rand(free.shape, device="cuda", generator=gen) < 0.001
    many.view(n, -1)[:, 0] = True
    return {"none": torch.zeros_like(free), "one": one, "many": many}


@pytest.mark.parametrize("shape", [(1, 1), (1, 37), (37, 1), (31, 33), (256, 256), (1000, 1000)])
def test_synthetic_images(ag, torch_, shape):
    torch = torch_
    b1, b2 = shape
    gen = torch.Generator(device="cuda").manual_seed(b1 * 7919 + b2)
    for f in (0.3, 0.6, 0.9, 1.0):
        free = torch.rand(1, b1, b2, device="cuda", generator=gen) < f
        for gname, goals in goal_sets(torch, free, gen).items():
            for wrap in range(4):
                check_image(torch, free, goals, wrap, "%dx%d f=%g %s wrap=%d" % (b1, b2, f, gname, wrap))


def test_composed_form_equals_numpy(ag, torch_):
    """the 4096^2 cases' reference, held to scipy at 1024^2"""
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(2)
    free = torch.rand(2, 1024, 1024, device="cuda", generator=gen) < 0.65
    goals = torch.rand(2, 1024, 1024, device="cuda", generator=gen) < 2e-5
    for wrap in range(4):
        assert_dist(composed_distance(free, goals, wrap)[0],
                    distance_numpy(free.cpu().numpy(), goals.cpu().numpy(), wrap), "composed %d" % wrap)


def test_4096(ag, torch_):
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(40)
    for f, wrap in ((0.6, 3), (0.8, 0), (0.95, 1)):
        free = torch.rand(1, 4096, 4096, device="cuda", generator=gen) < f
        goals = torch.rand(1, 4096, 4096, device="cuda", generator=gen) < 1e-6
        goals[0, 2048, 2048] = True
        check_image(torch, free, goals, wrap, "4096^2 f=%g wrap %d" % (f, wrap), "composed")


@pytest.mark.parametrize("shape", [(6, 6), (300, 500), (1000, 1000)])
def test_adversarial_images(ag, torch_, shape):
    """the spiral and the serpentine give very long distances and many relaxation passes"""
    torch = torch_
    b1, b2 = shape
    for name, img in special_images(b1, b2).items():
        free = torch.as_tensor(img, device="cuda")[None]
        ends = torch.zeros_like(free)
        ends[0, 0, 0] = True                                   # the spiral's and the serpentine's first pose
        for gname, goals in (("corner", ends), ("all", torch.ones_like(free))):
            for wrap in range(4):
                dist, _ = check_image(torch, free, goals, wrap, "%s %s %dx%d wrap=%d" % (name, gname, b1, b2, wrap))
                if gname == "all":
                    assert torch.equal(dist, torch.where(free, 0, -1).int())
        if name == "spiral":
            dist, md = op(torch, pack_words(~free), pack_words(ends), b1, b2, 0)
            assert int(md) == int(img.sum()) - 1                # one corridor


def test_padding_and_colliding_goals_seed_nothing(ag, torch_):
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(4)
    for b1, b2 in ((37, 45), (100, 100), (5, 1), (64, 33)):
        free = torch.rand(3, b1, b2, device="cuda", generator=gen) < 0.6
        goals = torch.rand(3, b1, b2, device="cuda", generator=gen) < 0.02
        words, gw = pack_words(~free), pack_words(goals)
        if b2 % 32:
            pad = (~((1 << (b2 % 32)) - 1)) & 0xFFFFFFFF
            pad = pad - (1 << 32) if pad >= 1 << 31 else pad
            gw[..., -1] |= pad                                  # a goal on every padding bit
        on_colliding = pack_words(goals | ~free)                # and on every colliding pose
        for wrap in range(4):
            clean, md = check_image(torch, free, goals, wrap, "padding %dx%d wrap %d" % (b1, b2, wrap))
            for dirty in (gw, on_colliding | gw):
                got, md2 = op(torch, words, dirty, b1, b2, wrap)
                assert_dist(got, clean, "dirty goals %dx%d wrap %d" % (b1, b2, wrap))
                assert torch.equal(md, md2)


def test_many_grids(ag, torch_):
    """1024 grids of 256^2 (config-5-like batches) with distinct content, and a ragged 37 grids of 70 x 45: grids never
    join"""
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(6)
    f = torch.linspace(0.4, 0.95, 1024, device="cuda").view(-1, 1, 1)
    free = torch.rand(1024, 256, 256, device="cuda", generator=gen) < f
    free[:, 0, :] = free[:, -1, :] = True
    goals = torch.zeros_like(free)
    goals[::2, 128, 128] = True                                 # odd grids have no goal
    for wrap in (0, 3):
        dist, md = check_image(torch, free, goals, wrap, "1024 x 256^2 wrap %d" % wrap, "composed")
        some = [0, 1, 511, 1022]
        assert_dist(dist[some], distance_numpy(free[some].cpu().numpy(), goals[some].cpu().numpy(), wrap), "numpy")
        assert (md[1::2] == -1).all() and (dist[1::2] < 0).all()
    free = torch.rand(37, 70, 45, device="cuda", generator=gen) < 0.7
    goals = torch.rand(37, 70, 45, device="cuda", generator=gen) < 0.003
    for wrap in range(4):
        check_image(torch, free, goals, wrap, "37 x 70x45 wrap %d" % wrap)


def test_consistent_with_components(ag, torch_):
    """dist >= 0 exactly where the pose's component label is the label of a free goal; adjacent free poses differ by at
    most 1"""
    torch = torch_
    from abstract_gym_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(13)
    for b1, b2, f in ((512, 512, 0.6), (300, 200, 0.75)):
        free = torch.rand(2, b1, b2, device="cuda", generator=gen) < f
        goals = torch.rand(2, b1, b2, device="cuda", generator=gen) < 3e-5
        for wrap in range(4):
            words = pack_words(~free)
            dist, _ = op(torch, words, pack_words(goals), b1, b2, wrap)
            labels = torch.empty(2, b1, b2, dtype=torch.int32, device="cuda")
            ops.cspace_components(words, b1, b2, wrap, labels, None)
            for g in range(2):
                goal_labels = torch.unique(labels[g][goals[g] & free[g]])
                assert torch.equal(dist[g] >= 0, torch.isin(labels[g], goal_labels) & free[g])
            d = dist.to(torch.int64)
            for dim, bit in ((1, 1), (2, 2)):
                a, b = d, torch.roll(d, -1, dim)
                both = (a >= 0) & (b >= 0)
                if not wrap & bit:
                    both.narrow(dim, d.shape[dim] - 1, 1).fill_(False)
                assert ((a - b).abs()[both] <= 1).all()


def check_scene_distance(sc, b1, b2, engine, goals, want_goal_img, what, lo=(0.0, 0.0), step=None, wrap=None):
    import torch
    st = (2 * math.pi / b1, 2 * math.pi / b2) if step is None else step
    w = (3 if step is None else 0) if wrap is None else int(wrap[0]) | int(wrap[1]) << 1
    dist, md = sc.cspace_distance(b1, b2, goals=goals, lo=lo, step=step, wrap=wrap, max_dist=True, engine=engine)
    img = sc.cspace_occupancy(b1, b2, lo=lo, step=st, engine=engine)
    assert dist.dtype == torch.int32 and md.dtype == torch.int32 and dist.shape == img.shape
    if b1 * b2 <= 1 << 20:
        want = distance_numpy(~img.cpu().numpy(), want_goal_img.cpu().numpy(), w)
    else:
        want = composed_distance(~img, want_goal_img, w)[0].cpu().numpy()
    assert_dist(dist, want, "%s %s" % (what, engine))
    assert torch.equal(dist == -1, img), what
    assert np.array_equal(md.cpu().numpy(), maxima(want)), what
    return dist


def goal_image(torch, poses, n_grids, b1, b2, lo, st, w):
    """bool goal image of [G, 2] or [n_grids, G, 2] poses by the numpy snapping rule"""
    from components_reference import component_of_numpy
    p = np.asarray(poses, dtype=np.float64)
    if p.ndim == 2:
        p = np.broadcast_to(p, (n_grids,) + p.shape)
    idx = np.arange(n_grids * b1 * b2, dtype=np.int32).reshape(n_grids, b1, b2)
    img = np.zeros(n_grids * b1 * b2, dtype=bool)
    for g in range(n_grids):
        k = component_of_numpy(idx, p[g], np.full(len(p[g]), g), lo, st, w)
        img[k[k >= 0]] = True
    return torch.as_tensor(img.reshape(n_grids, b1, b2), device="cuda")


def test_scene0_every_goal_form(ag, torch_):
    torch = torch_
    sc = scene(ag, torch, ag.OccupancyGrid(size=9, random_obstacle=False))
    b = 1024
    st = (2 * math.pi / b,) * 2
    valid, s1, s2 = sc.robot.inverse_kinematic([[sc.target_c.x, sc.target_c.y]], corrected=True)
    ik = torch.cat([s1[valid], s2[valid]]).cpu().numpy()
    assert len(ik) == 2
    for engine in ENGINES:
        check_scene_distance(sc, b, b, engine, None, goal_image(torch, ik, 1, b, b, (0, 0), st, 3), "scene_0 cartesian")
    sc.choose_j_tar = True
    tj = np.array([[1.1, -0.2]])
    check_scene_distance(sc, b, b, "fast", None, goal_image(torch, tj, 1, b, b, (0, 0), st, 3), "scene_0 joint target")
    sc.choose_j_tar = False
    poses = np.array([[0.1, 0.2], [3.0, -1.0], [math.nan, 0.0], [1e300, 0.0], [2.0, 2.0]])
    check_scene_distance(sc, b, b, "fast", torch.as_tensor(poses, device="cuda"),
                         goal_image(torch, poses, 1, b, b, (0, 0), st, 3), "scene_0 poses")
    img = torch.zeros(1, b, b, dtype=torch.bool, device="cuda")
    img[0, 5, 900] = img[0, 700, 3] = True
    check_scene_distance(sc, b, b, "exact", img, img, "scene_0 image")
    check_scene_distance(sc, 4096, 4096, "fast", None, goal_image(torch, ik, 1, 4096, 4096, (0, 0), (2 * math.pi / 4096,) * 2, 3),
                         "scene_0 4096^2")


def test_random_grids_per_grid_goals(ag, torch_):
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(9)
    grid = ag.BatchedOccupancyGrid.random(3, 48, 0.02, envs_per_grid=256, device="cuda", generator=gen)
    sc = scene(ag, torch, grid)
    b1, b2 = 200, 150
    lo, st = (-0.3, 0.2), (0.031, 0.04)
    rng = np.random.default_rng(2)
    per_grid = rng.uniform(-1, 6, (3, 4, 2))
    for engine in ENGINES:
        for wrap in ((False, False), (True, False), (True, True)):
            w = int(wrap[0]) | int(wrap[1]) << 1
            check_scene_distance(sc, b1, b2, engine, torch.as_tensor(per_grid, device="cuda"),
                                 goal_image(torch, per_grid, 3, b1, b2, lo, st, w), "random grids", lo=lo, step=st,
                                 wrap=wrap)
    with pytest.raises(ValueError):
        sc.cspace_distance(b1, b2, goals=torch.zeros(2, b1, b2, dtype=torch.bool, device="cuda"))
    with pytest.raises(ValueError):
        sc.cspace_distance(b1, b2, goals=torch.zeros(2, 4, 2, dtype=torch.float64, device="cuda"))


@pytest.mark.parametrize("wrap", [None, (False, False), (True, False)])
def test_distance_of_and_path(ag, torch_, wrap):
    """cspace_distance_of and cspace_path against numpy on a multi-grid scene with env_id0 != 0: colliding,
    unreachable, off-lattice and NaN starts, max_len 1 and shorter than the path"""
    torch = torch_
    from components_reference import component_of_numpy
    gen = torch.Generator(device="cuda").manual_seed(12)
    grid = ag.BatchedOccupancyGrid.random(3, 31, 0.05, envs_per_grid=5, device="cuda", generator=gen)
    n, env_id0 = 400, 7
    sc = scene(ag, torch, grid, n=n, env_id0=env_id0)
    b1, b2 = 96, 80
    if wrap is None:
        lo, step, w = (0.0, 0.0), None, 3
        st = (2 * math.pi / b1, 2 * math.pi / b2)
    else:
        lo, st, w = (-1.0, 0.3), (0.05, 0.07), int(wrap[0]) | int(wrap[1]) << 1
        step = st
    goals = np.array([[1.0, 1.5], [3.0, 2.0]])
    dist = sc.cspace_distance(b1, b2, goals=torch.as_tensor(goals, device="cuda"), lo=lo, step=step, wrap=wrap)
    d = dist.cpu().numpy()
    rng = np.random.default_rng(3)
    q = rng.uniform(-2.0, 7.0, (n, 2))
    q[0] = (math.nan, 0.1)
    q[1] = (0.2, math.inf)
    q[2] = (1e300, -1e300)
    q[3] = (lo[0] - 0.51 * st[0], lo[1])
    grids = grid_of_env(n, env_id0, 5, 3)
    got = sc.cspace_distance_of(dist, torch.as_tensor(q, device="cuda"), lo=lo, step=step, wrap=wrap)
    want = component_of_numpy(d, q, grids, lo, st, w)
    assert got.dtype == torch.int32 and np.array_equal(got.cpu().numpy(), want)
    assert (want == -1).any() and (want > 0).any()
    idx = np.arange(b1 * b2, dtype=np.int32).reshape(1, b1, b2).repeat(3, axis=0)
    start = component_of_numpy(idx, q, np.zeros(n, dtype=np.int64), lo, st, w)
    longest = int(want.max()) + 1
    for max_len in (1, 7, longest, longest + 5):
        path, length = sc.cspace_path(dist, max_len, torch.as_tensor(q, device="cuda"), lo=lo, step=step, wrap=wrap)
        wp, wl = descend_numpy(d, start, grids, max_len, w)
        assert path.shape == (n, max_len) and path.dtype == torch.int32 and length.dtype == torch.int32
        assert np.array_equal(length.cpu().numpy(), wl) and np.array_equal(path.cpu().numpy(), wp), max_len
        assert (wl[:4] == 0).all()
    path, length = sc.cspace_path(dist, 50, lo=lo, step=step, wrap=wrap)            # the current joints
    cur = np.stack([sc.robot.joint_1.cpu().numpy(), sc.robot.joint_2.cpu().numpy()], axis=1)
    wp, wl = descend_numpy(d, component_of_numpy(idx, cur, np.zeros(n, dtype=np.int64), lo, st, w), grids, 50, w)
    assert np.array_equal(path.cpu().numpy(), wp) and np.array_equal(length.cpu().numpy(), wl)


def test_descend_op_bad_device_data(ag, torch_):
    """out-of-range grid indices and starts are device data: length 0, path -1"""
    torch = torch_
    from abstract_gym_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(3)
    free = torch.rand(2, 50, 60, device="cuda", generator=gen) < 0.8
    goals = torch.zeros_like(free)
    goals[:, 25, 30] = True
    for wrap in range(4):
        dist, _ = op(torch, pack_words(~free), pack_words(goals), 50, 60, wrap)
        start = torch.tensor([0, 3000, -1, 2999, 1234, 1234, 1234, 7], dtype=torch.int32, device="cuda")
        grid = torch.tensor([0, 1, 0, 1, -1, 2, 1 << 40, 1], dtype=torch.int64, device="cuda")
        for max_len in (1, 3, 200):
            path = torch.empty(8, max_len, dtype=torch.int32, device="cuda")
            length = torch.empty(8, dtype=torch.int32, device="cuda")
            ops.cspace_descend(dist, 50, 60, wrap, start, grid, max_len, path, length)
            wp, wl = descend_numpy(dist.cpu().numpy(), start.cpu().numpy(), grid.cpu().numpy(), max_len, wrap)
            assert np.array_equal(path.cpu().numpy(), wp) and np.array_equal(length.cpu().numpy(), wl)
            assert (wl[[1, 2, 4, 5, 6]] == 0).all()
        with pytest.raises(RuntimeError):
            ops.cspace_descend(dist, 50, 60, wrap, start, grid, 0, path, length)
        with pytest.raises(RuntimeError):
            ops.cspace_descend(dist, 50, 60, wrap, start, grid.int(), 200, path, length)


def test_graph_capture(ag, torch_):
    """descent captures and replays; the distance call inside a capture fails with the CUDA error before enqueuing
    anything, and the capture still ends cleanly"""
    torch = torch_
    from abstract_gym_b200 import _lib
    sc = scene(ag, torch, ag.OccupancyGrid(size=9, random_obstacle=False), n=4096)
    sc.robot.joint_1.uniform_(0, 6.28)
    sc.robot.joint_2.uniform_(0, 6.28)
    dist = sc.cspace_distance(512)
    want = sc.cspace_path(dist, 300)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            path, length = sc.cspace_path(dist, 300)
            with pytest.raises(_lib.AgError) as err:
                sc.cspace_distance(64, goals=torch.zeros(1, 64, 64, dtype=torch.bool, device="cuda"))
    assert err.value.status == 900                                          # cudaErrorStreamCaptureUnsupported
    path.fill_(-7)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(path, want[0]) and torch.equal(length, want[1])
    assert torch.equal(sc.cspace_distance(512), dist)                       # the stream works after the capture


def test_torch_ops(ag, torch_):
    torch = torch_
    from abstract_gym_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(9)
    grid = ag.BatchedOccupancyGrid.random(3, 48, 0.02, envs_per_grid=256, device="cuda", generator=gen)
    sc = scene(ag, torch, grid)
    b1, b2 = 70, 90
    words = sc.cspace_occupancy(b1, b2, packed=True)
    gimg = torch.zeros(3, b1, b2, dtype=torch.bool, device="cuda")
    gimg[:, 10, 10] = gimg[1, 60, 80] = True
    gw = pack_words(gimg)
    for wrap in range(4):
        want, want_md = sc.cspace_distance(b1, b2, goals=gimg, wrap=(bool(wrap & 1), bool(wrap & 2)), max_dist=True)
        dist, md = op(torch, words, gw, b1, b2, wrap)
        assert_dist(dist, want, "torch op wrap %d" % wrap)
        assert torch.equal(md, want_md)
        again = torch.empty_like(dist)
        ops.cspace_distance(words, gw, b1, b2, wrap, again, None)
        assert_dist(again, want, "torch op, no maxima")
    dist = torch.empty(3, b1, b2, dtype=torch.int32, device="cuda")
    for bad in (lambda: ops.cspace_distance(words, gw, b1, b2, 0, dist[:2], None),
                lambda: ops.cspace_distance(words, gw[:2], b1, b2, 0, dist, None),
                lambda: ops.cspace_distance(words[:, :, :2].contiguous(), gw, b1, b2, 0, dist, None),
                lambda: ops.cspace_distance(words, gw, b1, b2, 0, dist, torch.empty(2, dtype=torch.int32, device="cuda")),
                lambda: ops.cspace_distance(words, gw, b1, b2, 4, dist, None),
                lambda: ops.cspace_distance(words, gw, b1, b2, 0, dist.to(torch.int64), None)):
        with pytest.raises(RuntimeError):
            bad()
    with pytest.raises((NotImplementedError, RuntimeError)):
        ops.cspace_distance(words.cpu(), gw.cpu(), b1, b2, 0, dist.cpu(), None)


_DEBUG_CHILD = r'''
import sys
import numpy as np, torch
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import abstract_gym_b200 as ag
from abstract_gym_b200 import _lib, ops
from components_reference import pack_words, special_images
from distance_reference import descend_numpy, distance_numpy
assert _lib.lib_path().endswith("_debug.so"), _lib.lib_path()
gen = torch.Generator(device="cuda").manual_seed(1)
cases = [torch.rand(3, 300, 500, device="cuda", generator=gen) < 0.7,
         torch.rand(64, 33, 70, device="cuda", generator=gen) < 0.8,
         torch.as_tensor(special_images(130, 260)["spiral"], device="cuda")[None]]
for free in cases:
    n, b1, b2 = free.shape
    goals = torch.zeros_like(free)
    goals[:, 0, 0] = goals[:, b1 // 2, b2 // 3] = True
    for wrap in range(4):
        dist = torch.empty(n, b1, b2, dtype=torch.int32, device="cuda")
        md = torch.empty(n, dtype=torch.int32, device="cuda")
        ops.cspace_distance(pack_words(~free), pack_words(goals), b1, b2, wrap, dist, md)
        want = distance_numpy(free.cpu().numpy(), goals.cpu().numpy(), wrap)
        assert np.array_equal(dist.cpu().numpy(), want), (free.shape, wrap)
        m = 300
        start = torch.randint(-5, b1 * b2 + 5, (m,), dtype=torch.int32, device="cuda", generator=gen)
        grid = torch.randint(-1, n + 1, (m,), dtype=torch.int64, device="cuda", generator=gen)
        path = torch.empty(m, 64, dtype=torch.int32, device="cuda")
        length = torch.empty(m, dtype=torch.int32, device="cuda")
        ops.cspace_descend(dist, b1, b2, wrap, start, grid, 64, path, length)
        wp, wl = descend_numpy(want, start.cpu().numpy(), grid.cpu().numpy(), 64, wrap)
        assert np.array_equal(path.cpu().numpy(), wp) and np.array_equal(length.cpu().numpy(), wl)
print("debug distance ok")
'''


def test_debug_bounds_build_distance(ag, torch_):
    """the -DAG_DEBUG_BOUNDS library gives the reference's distances and paths (child process); each new kernel of it
    carries the index traps and the release library none (read from the machine code: no test sets a trap off)"""
    import subprocess
    import sys
    from abstract_gym_b200 import build as ag_build
    from test_gpu_parity import _traps_per_kernel
    lib = ag_build.build_debug()
    code = _DEBUG_CHILD % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, AG_LIB_PATH=lib), stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "debug distance ok" in r.stdout, r.stdout[-3000:]
    debug, release = _traps_per_kernel(lib), _traps_per_kernel(ag_build.LIB)
    kernels = [k for k in debug if "k_dist_" in k]
    assert len(kernels) == 4 and all(debug[k] > 0 for k in kernels), {k: debug[k] for k in kernels}
    assert all(release[k] == 0 for k in kernels)
