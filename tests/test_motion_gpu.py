"""Motion checking on the device (ag_check_motion / BatchedScene.check_motion / torch.ops.abstract_gym_b200.check_motion)
against the reference composition of tests/motion_reference.py: move_to_joint_pose's poses and the oracle's
collision check at each.  first_collision, first_hit and last_free must match bit for bit, for every engine."""
import os

import numpy as np
import pytest

from motion_reference import reference_motion

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


def grid_of(ag, occ):
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    if occ is not None:
        g.load_from_matrix(occ)
    return g


def scene(ag, torch, grid, m, env_id0=0, engine="fast"):
    rb = ag.BatchedTwoJointRobot(torch.zeros(m, dtype=torch.float64, device="cuda"), torch.zeros(m, dtype=torch.float64, device="cuda"))
    return ag.BatchedScene(rb, grid, engine=engine, env_id0=env_id0)


def run(torch, sc, start, goal, steps, engine):
    st = torch.as_tensor(np.asarray(steps, np.int32), device="cuda") if not np.isscalar(steps) else int(steps)
    fc, extra = sc.check_motion(torch.as_tensor(goal, device="cuda"), start=torch.as_tensor(start, device="cuda"), steps=st,
                                first_hit=True, last_free=True, engine=engine)
    return fc.cpu().numpy(), extra["first_hit"].cpu().numpy(), extra["last_free"].cpu().numpy()


def assert_same(got, ref, what=""):
    for name, g, r in zip(("first_collision", "first_hit", "last_free"), got, ref):
        same = (g == r) | (np.isnan(g) & np.isnan(r)) if g.dtype.kind == "f" else g == r
        assert same.all(), "%s %s: %d of %d differ, first at %d: %r vs %r" % (
            what, name, (~same).sum(), same.size, np.argwhere(~same)[0][0], g[~same][:3], r[~same][:3])


def scene0_motions(oracle, m, seed):
    """half the starts collision-free (rejection-sampled on the oracle), half uniform; goals uniform in [0, 2 pi)"""
    rng = np.random.default_rng(seed)
    sq, ci = oracle.manual_grid()
    start = rng.uniform(0.0, 2 * np.pi, (m, 2))
    bad = np.arange(m) < m // 2
    while bad.any():
        start[bad] = rng.uniform(0.0, 2 * np.pi, (bad.sum(), 2))
        hit, _, _ = oracle.collision_batch(start[:, 0].copy(), start[:, 1].copy(), sq, want_first_hit=False)
        bad &= hit != 0
    return start, rng.uniform(0.0, 2 * np.pi, (m, 2)), [(sq, ci)]


@pytest.fixture(scope="module")
def scene0_case(oracle):
    start, goal, grids = scene0_motions(oracle, 1 << 16, 1)
    return start, goal, grids, reference_motion(oracle, start, goal, np.full(len(start), 100), grids)


@pytest.mark.parametrize("engine", ENGINES)
def test_scene0_motions(ag, torch_, oracle, scene0_case, engine):
    """2^16 motions of 100 steps on scene_0's map (the configuration-space map form for FAST)"""
    start, goal, grids, ref = scene0_case
    sc = scene(ag, torch_, grid_of(ag, None), len(start))
    got = run(torch_, sc, start, goal, 100, engine)
    assert_same(got, ref, engine)
    assert (ref[0] > 0).sum() > 1000 and (ref[0] == -1).sum() > 1000 and (ref[0] == 1).sum() > 100


def test_free_motions_end_at_move_to_joint_pose(ag, torch_, scene0_case):
    start, goal, _, ref = scene0_case
    free = np.nonzero(ref[0] == -1)[0]
    rb = ag.BatchedTwoJointRobot(torch_.as_tensor(start[free, 0], device="cuda"), torch_.as_tensor(start[free, 1], device="cuda"))
    rb.move_to_joint_pose(torch_.as_tensor(goal[free], device="cuda"), steps=100)
    sc = scene(ag, torch_, grid_of(ag, None), len(start))
    _, _, lf = run(torch_, sc, start, goal, 100, "fast")
    assert np.array_equal(lf[free, 0], rb.joint_1.cpu().numpy()) and np.array_equal(lf[free, 1], rb.joint_2.cpu().numpy())


def special_motions(rng, m):
    """per-motion steps including 1, 7, 100, 1000, 0 and negative ones; start == goal; |q| > 2^20; NaN goals"""
    start = rng.uniform(-2 * np.pi, 2 * np.pi, (m, 2))
    goal = rng.uniform(-2 * np.pi, 2 * np.pi, (m, 2))
    steps = rng.choice(np.array([1, 7, 100, 1000, 0, -3, 13], np.int32), m, p=[.2, .2, .25, .05, .1, .1, .1])
    sel = rng.random(m)
    goal[sel < 0.05] = start[sel < 0.05]
    big = (sel >= 0.05) & (sel < 0.08)
    start[big] += rng.choice([-1.0, 1.0], (big.sum(), 2)) * 3.0e6
    goal[big] = start[big] + rng.uniform(-1.0, 1.0, (big.sum(), 2))
    goal[(sel >= 0.08) & (sel < 0.1), 1] = np.nan
    return start, goal, steps


GRIDS = {
    "scene0": None,
    "rand31": lambda rng: (rng.random((31, 31)) < 0.006).astype(np.uint8),   # sparse: obstacle list and map form
    "rand31_dense": lambda rng: (rng.random((31, 31)) < 0.05).astype(np.uint8),
    "rand64": lambda rng: (rng.random((64, 64)) < 0.02).astype(np.uint8),
}


@pytest.mark.parametrize("m", [1, 31, 257, 5000])
@pytest.mark.parametrize("name", sorted(GRIDS))
def test_special_motions_every_engine(ag, torch_, oracle, name, m):
    rng = np.random.default_rng(m + len(name))
    occ = None if GRIDS[name] is None else GRIDS[name](rng)
    grids = [oracle.manual_grid()] if occ is None else [oracle.grid_squares(occ)]
    start, goal, steps = special_motions(rng, m)
    ref = reference_motion(oracle, start, goal, steps, grids)
    sc = scene(ag, torch_, grid_of(ag, occ), m)
    for engine in ENGINES:
        assert_same(run(torch_, sc, start, goal, steps, engine), ref, "%s %s" % (name, engine))
    assert (ref[0] == -2).sum() == (steps < 1).sum()


@pytest.mark.parametrize("env_id0", [0, 300])
def test_grid_per_motion(ag, torch_, oracle, env_id0):
    """three 256 x 256 grids, motion i on grid ((env_id0 + i) / envs_per_grid) % 3"""
    rng = np.random.default_rng(7 + env_id0)
    occs = [(rng.random((256, 256)) < 0.004).astype(np.uint8) for _ in range(3)]
    m, epg = 1500, 256
    grid = ag.BatchedOccupancyGrid(torch_.as_tensor(np.stack(occs), device="cuda"), epg)
    start = rng.uniform(0.0, 2 * np.pi, (m, 2))
    goal = rng.uniform(0.0, 2 * np.pi, (m, 2))
    steps = rng.integers(1, 60, m).astype(np.int32)
    ref = reference_motion(oracle, start, goal, steps, [oracle.grid_squares(o) for o in occs], ((env_id0 + np.arange(m)) // epg) % 3)
    sc = scene(ag, torch_, grid, m, env_id0=env_id0)
    for engine in ENGINES:
        assert_same(run(torch_, sc, start, goal, steps, engine), ref, "256 x3 %s" % engine)
    assert (ref[0] > 0).sum() > 100


def test_1024_map(ag, torch_, oracle):
    rng = np.random.default_rng(8)
    occ = (rng.random((1024, 1024)) < 0.002).astype(np.uint8)
    m = 96
    start, goal = rng.uniform(0.0, 2 * np.pi, (m, 2)), rng.uniform(0.0, 2 * np.pi, (m, 2))
    ref = reference_motion(oracle, start, goal, np.full(m, 100), [oracle.grid_squares(occ)])
    sc = scene(ag, torch_, grid_of(ag, occ), m)
    for engine in ENGINES:
        assert_same(run(torch_, sc, start, goal, 100, engine), ref, "1024 %s" % engine)


@pytest.mark.parametrize("cached", [True, False])
def test_graph_capture(ag, torch_, oracle, cached):
    """a captured call equals the uncaptured one: on a grid whose map is cached, and on a fresh grid (no cache entry
    can be made inside a capture: the general form runs)"""
    torch = torch_
    start, goal, grids = scene0_motions(oracle, 4096, 9)
    grid = grid_of(ag, None)
    sc = scene(ag, torch, grid, len(start))
    st = torch.as_tensor(start, device="cuda")
    gl = torch.as_tensor(goal, device="cuda")
    steps = torch.full((len(start),), 100, dtype=torch.int32, device="cuda")
    if cached:
        ref = run(torch, sc, start, goal, 100, "fast")
    else:   # parameters no earlier call used (the target is part of the map's key): no cache entry exists
        sc.target_c = ag.Point(0.0123, -0.0456)
        ref = reference_motion(oracle, start, goal, np.full(len(start), 100), grids)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            fc, extra = sc.check_motion(gl, start=st, steps=steps, first_hit=True, last_free=True)
    g.replay()
    torch.cuda.synchronize()
    assert_same((fc.cpu().numpy(), extra["first_hit"].cpu().numpy(), extra["last_free"].cpu().numpy()), ref, "captured")


def test_torch_op_equals_object_api(ag, torch_, oracle):
    torch = torch_
    from abstract_gym_b200 import ops
    rng = np.random.default_rng(10)
    start, goal, steps = special_motions(rng, 3000)
    sc = scene(ag, torch, grid_of(ag, None), len(start))
    want = run(torch, sc, start, goal, steps, "fast")
    j1 = torch.as_tensor(start[:, 0].copy(), device="cuda")
    j2 = torch.as_tensor(start[:, 1].copy(), device="cuda")
    gl = torch.as_tensor(goal, device="cuda")
    stt = torch.as_tensor(steps, device="cuda")
    fc = torch.empty(len(start), dtype=torch.int32, device="cuda")
    fh = torch.empty_like(fc)
    lf = torch.empty(len(start), 2, dtype=torch.float64, device="cuda")
    ops.check_motion(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), j1, j2, gl, stt, fc, fh, lf, 0, ag.ENGINES["fast"])
    assert_same((fc.cpu().numpy(), fh.cpu().numpy(), lf.cpu().numpy()), want, "torch op")
    fc2 = torch.empty_like(fc)
    ops.check_motion(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), j1, j2, gl, stt, fc2, None, None, 0, ag.ENGINES["exact"])
    assert torch.equal(fc2, fc)
    with pytest.raises((NotImplementedError, RuntimeError)):
        ops.check_motion(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), j1.cpu(), j2.cpu(), gl.cpu(), stt.cpu(),
                         fc.cpu(), None, None, 0, 1)


_DEBUG_CHILD = r'''
import sys
import numpy as np, torch
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import abstract_gym_b200 as ag
from abstract_gym_b200 import _lib
from oracle import oracle as orc
from motion_reference import reference_motion
assert _lib.lib_path().endswith("_debug.so"), _lib.lib_path()
rng = np.random.default_rng(12)
m = 2048
for name, occs in (("scene0", None), ("rand64", [(rng.random((64, 64)) < 0.02).astype(np.uint8)]),
                   ("rand300", [(rng.random((300, 300)) < 0.004).astype(np.uint8) for _ in range(2)])):
    start, goal = rng.uniform(0, 2 * np.pi, (m, 2)), rng.uniform(0, 2 * np.pi, (m, 2))
    steps = rng.integers(-1, 80, m).astype(np.int32)
    if occs is None:
        grid, grids, which = ag.OccupancyGrid(size=9, random_obstacle=False), [orc.manual_grid()], None
    else:
        grid = ag.BatchedOccupancyGrid(torch.as_tensor(np.stack(occs), device="cuda"), m // len(occs))
        grids, which = [orc.grid_squares(o) for o in occs], np.arange(m) // (m // len(occs))
    ref = reference_motion(orc, start, goal, steps, grids, which)
    rb = ag.BatchedTwoJointRobot(torch.zeros(m, dtype=torch.float64, device="cuda"), torch.zeros(m, dtype=torch.float64, device="cuda"))
    sc = ag.BatchedScene(rb, grid)
    for engine in ("fast", "exact", "brute"):
        if engine == "brute" and name == "rand300":
            continue
        fc, ex = sc.check_motion(torch.as_tensor(goal, device="cuda"), start=torch.as_tensor(start, device="cuda"),
                                 steps=torch.as_tensor(steps, device="cuda"), first_hit=True, last_free=True, engine=engine)
        got = (fc.cpu().numpy(), ex["first_hit"].cpu().numpy(), ex["last_free"].cpu().numpy())
        for g, r in zip(got, ref):
            assert np.array_equal(g, r), (name, engine)
print("debug motion ok")
'''


def test_debug_bounds_build_motion(ag, torch_):
    """the -DAG_DEBUG_BOUNDS library gives the same motion results (child process); every motion kernel of it carries
    the index traps and the release library none (read from the machine code: no test sets a trap off)"""
    import subprocess
    import sys
    from abstract_gym_b200 import build as ag_build
    from test_gpu_parity import _traps_per_kernel
    lib = ag_build.build_debug()
    code = _DEBUG_CHILD % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, AG_LIB_PATH=lib), stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "debug motion ok" in r.stdout, r.stdout[-3000:]
    debug, release = _traps_per_kernel(lib), _traps_per_kernel(ag_build.LIB)
    motion = [k for k in debug if "k_check_motion" in k]
    assert len(motion) == 4 and all(debug[k] > 0 for k in motion), {k: debug[k] for k in motion}
    assert all(release[k] == 0 for k in motion)
