"""CPU-only checks of the C-ABI boundary: the library loads, exports every symbol the header
declares, and its host-only helpers agree with the reference goldens.  No device compute here."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from abstract_gym_b200 import _lib
    return _lib.load()


def test_header_symbols_exported(lib):
    from abstract_gym_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "abstract_gym_b200.h")).read()
    declared = set(re.findall(r"AG_API[^;(]*?\b(ag_\w+)\s*\(", hdr))
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), "library does not export %s" % name
    assert declared == set(_lib.SYMBOLS), "ctypes table and header disagree: %s" % (declared ^ set(_lib.SYMBOLS))


def test_struct_layouts_match_header():
    from abstract_gym_b200 import _lib
    assert C.sizeof(_lib.Params) == 11 * 8 + 2 * 4
    assert C.sizeof(_lib.Grid) == 3 * 8 + 2 * 8 + 4 * 4 + 2 * 8 + 8 + 8
    assert C.sizeof(_lib.RolloutArgs) == 8 + 8 + 4 + 4 + 8 + 8 + 8 + 4 + 4 + 14 * 8 + 8 + 8 + 8 + 4 + 4


def test_default_params_are_the_reference_literals(lib):
    from abstract_gym_b200 import _lib
    p = _lib.default_params()
    assert (p.link_1, p.link_2) == (0.4, 0.3)                 # robot/two_joint_robot.py:12-13
    assert (p.target_x, p.target_y) == (-0.2, -0.3)           # scenario/scene_0.py:17
    assert (p.target_j1, p.target_j2) == (1.1, -0.2)          # scenario/scene_0.py:30
    assert p.reach_eps == 2e-3 and p.section_eps == 1e-10
    assert (p.reward_collision, p.reward_reach) == (-1e3, 1e4)
    assert p.action_scale == 0.1 and p.choose_j_tar == 0


def test_status_strings(lib):
    from abstract_gym_b200 import _lib
    assert _lib.status_string(0) == "ok"
    assert _lib.status_string(-5) == "The matrix is not square."   # occupancy_grid.py:81
    assert "NULL" in _lib.status_string(-1)


@pytest.mark.parametrize("S", [2, 5, 9, 31, 32, 33, 64, 201, 256, 1024])
def test_grid_tables_match_oracle(lib, oracle, S):
    from abstract_gym_b200 import _lib
    spad = (S + 1) & ~1
    mx, my = np.zeros(spad), np.zeros(spad)
    side = C.c_double()
    assert lib.ag_grid_tables_host(S, 1.6, mx.ctypes.data_as(C.c_void_p), my.ctypes.data_as(C.c_void_p), C.byref(side)) == 0
    occ = np.eye(S, dtype=np.uint8)          # obstacle (r=c=i): min_x = table_x[i], min_y = table_y[i]
    sq, _ = oracle.grid_squares(occ)
    assert np.array_equal(sq[:, 0], mx[:S]) and np.array_equal(sq[:, 1], my[:S])
    assert np.array_equal(sq[:, 2], mx[:S] + side.value) and np.array_equal(sq[:, 3], my[:S] + side.value)
    assert side.value == 1.6 / (S - 1)
    assert lib.ag_grid_words_per_row(S) == (S + 31) // 32
    assert lib.ag_grid_stride_words(S) % 4 == 0 and lib.ag_grid_stride_words(S) >= S * ((S + 31) // 32)


def test_grid_tables_match_reference_goldens(lib, golden_dir):
    z = np.load(os.path.join(golden_dir, "scene_cases.npz"))
    for name in ("manual9", "rand9", "rand31", "rand64", "rand6", "matrix5"):
        occ, sq = z[name + "/occ"], z[name + "/squares"]
        S = occ.shape[0]
        spad = (S + 1) & ~1
        mx, my = np.zeros(spad), np.zeros(spad)
        side = C.c_double()
        lib.ag_grid_tables_host(S, float(z[name + "/env_size"]), mx.ctypes.data_as(C.c_void_p),
                                my.ctypes.data_as(C.c_void_p), C.byref(side))
        ci = z[name + "/cell_index"]
        r, c = ci // S, ci % S
        assert np.array_equal(sq[:, 0], mx[c]) and np.array_equal(sq[:, 1], my[r])
        assert np.array_equal(sq[:, 2], mx[c] + side.value) and np.array_equal(sq[:, 3], my[r] + side.value)


def test_grid_pack_host(lib):
    rng = np.random.default_rng(3)
    for S in (5, 9, 32, 33, 70):
        occ = (rng.random((S, S)) < 0.3).astype(np.uint8)
        words = np.zeros(lib.ag_grid_stride_words(S), dtype=np.uint32)
        assert lib.ag_grid_pack_host(occ.ctypes.data_as(C.c_void_p), S, S, words.ctypes.data_as(C.c_void_p)) == 0
        wpr = (S + 31) // 32
        for r in range(S):
            for c in range(S):
                assert ((words[r * wpr + c // 32] >> (c % 32)) & 1) == occ[r, c]
    occ = np.zeros((4, 5), dtype=np.uint8)
    words = np.zeros(64, dtype=np.uint32)
    assert lib.ag_grid_pack_host(occ.ctypes.data_as(C.c_void_p), 4, 5, words.ctypes.data_as(C.c_void_p)) == -5
    assert lib.ag_grid_pack_host(None, 4, 4, words.ctypes.data_as(C.c_void_p)) == -1


def test_argument_validation_without_device(lib):
    """bad arguments are rejected before anything touches the device"""
    from abstract_gym_b200 import _lib
    p = _lib.default_params()
    g = _lib.Grid()
    assert lib.ag_collision_check(p, g, None, None, None, None, 4, 0, 0, None) == -1      # NULL grid pointers
    g.bits = g.min_x = g.min_y = 256
    g.S, g.words_per_row, g.n_grids, g.grid_stride_words, g.envs_per_grid = 9, 1, 1, 12, 1
    g.side, g.env_size = 0.2, 1.6
    assert lib.ag_collision_check(p, g, None, None, None, None, -1, 0, 0, None) == -2     # n < 0
    assert lib.ag_collision_check(p, g, None, None, None, None, 0, 0, 0, None) == 0       # empty batch is fine
    assert lib.ag_collision_check(p, g, None, None, None, None, 4, 0, 0, None) == -1      # NULL arrays
    g.words_per_row = 2
    assert lib.ag_collision_check(p, g, None, None, None, None, 0, 0, 0, None) == -2      # inconsistent grid
    g.words_per_row = 1
    a = _lib.RolloutArgs()
    a.n, a.K = 4, 0
    assert lib.ag_rollout(p, g, C.byref(a), None) == -2                                   # K < 1
    a.K = 8
    assert lib.ag_rollout(p, g, C.byref(a), None) == -1                                   # NULL state
    assert lib.ag_rollout(p, g, None, None) == -1
    assert lib.ag_launch_count() == 0


OK, NULL, SHAPE, MODE, ALIGN = 0, -1, -2, -3, -4
EXACT, FAST, BAD_ENGINE = 0, 1, 9
D = 4096                                     # fake device address, 16-byte aligned; D + k is misaligned for k < 16


def _grid():
    from abstract_gym_b200 import _lib
    g = _lib.Grid()
    g.bits = g.min_x = g.min_y = 256
    g.S, g.words_per_row, g.n_grids, g.grid_stride_words, g.envs_per_grid = 9, 1, 1, 12, 1
    g.side, g.env_size = 0.2, 1.6
    return g


def _rollout(lib, p, g, args=True, **fields):
    from abstract_gym_b200 import _lib
    if args is None:
        return lib.ag_rollout(p, g, None, None)
    a = _lib.RolloutArgs()
    a.n, a.K, a.engine = 4, 8, FAST
    a.j1 = a.j2 = a.reward = a.flags = a.step_ctr = a.reset_ctr = a.ep_len = a.stats = D
    for k, v in fields.items():
        setattr(a, k, v)
    return lib.ag_rollout(p, g, C.byref(a), None)


# Each entry point with valid arguments on fake device addresses; a case overrides some of them.  Unchanged, every
# call would launch (or, for ag_cspace_map, allocate), so every case must be rejected before the CUDA runtime.
CALLS = {
    "ag_collision_check": lambda lib, p, g, j1=D, j2=D, hit=D, first_hit=None, n=4, engine=FAST:
        lib.ag_collision_check(p, g, j1, j2, hit, first_hit, n, 0, engine, None),
    "ag_check_motion": lambda lib, p, g, j1=D, j2=D, goal=D, steps=D, fc=D, last_free=None, m=4, engine=FAST:
        lib.ag_check_motion(p, g, j1, j2, goal, steps, fc, None, last_free, m, 0, engine, None),
    "ag_cspace_occupancy": lambda lib, p, g, lo1=0.0, step1=0.1, b1=8, lo2=0.0, step2=0.1, b2=8, bits=D, fc=None,
                                  engine=FAST:
        lib.ag_cspace_occupancy(p, g, lo1, step1, b1, lo2, step2, b2, bits, fc, engine, None),
    "ag_cspace_components": lambda lib, p, g, bits=D, n_grids=1, b1=8, b2=8, wrap=3, labels=D, nc=None:
        lib.ag_cspace_components(bits, n_grids, b1, b2, wrap, labels, nc, None),
    "ag_cspace_map": lambda lib, p, g, cmap=D: lib.ag_cspace_map(p, g, cmap, None),
    "ag_step": lambda lib, p, g, j1=D, actions=D, f32=0, flags=D, ee=None, targets=None, n=4, engine=FAST:
        lib.ag_step(p, g, j1, D, actions, f32, D, flags, ee, None, None, None, targets, n, 0, engine, None),
    "ag_reset": lambda lib, p, g, reward=None, reset_ctr=D, reset_u=None, R=0, clear_flags=0, n=4, engine=FAST:
        lib.ag_reset(p, g, D, D, reward, D, reset_ctr, None, reset_u, R, 0, clear_flags, None, n, 0, engine, None),
    "ag_step_obs": lambda lib, p, g, actions=D, obs=D, collision=D, final_obs=None, crop=None, crop_size=0, n=4,
                          engine=FAST:
        lib.ag_step_obs(p, g, D, D, actions, 0, D, D, D, D, None, obs, D, D, collision, final_obs, crop, crop_size, None,
                        0, 1, n, 0, engine, None),
    "ag_rollout": _rollout,
}


def _case(entry, status, **kw):
    parts = []
    for k, v in kw.items():
        parts += ["%s.%s=%s" % (k, f, x) for f, x in v.items()] if isinstance(v, dict) else ["%s=%s" % (k, v)]
    return pytest.param(entry, kw, status, id="%s:%s" % (entry, ",".join(parts)))


BAD_GRID, NO_GRID_BITS, LONG_LINKS = {"words_per_row": 2}, {"bits": None}, {"link_1": 1.5}

# (entry point, status, arguments): one bad argument, then pairs whose status shows which check comes first.  grid /
# params set fields of the fake grid / the default parameters; LONG_LINKS is outside the FAST engine's error budget.
STATUS_TABLE = [
    _case("ag_collision_check", SHAPE, n=-1),
    _case("ag_collision_check", SHAPE, n=-1, p=None, engine=BAD_ENGINE),
    _case("ag_collision_check", NULL, p=None),
    _case("ag_collision_check", NULL, g=None),
    _case("ag_collision_check", NULL, grid=NO_GRID_BITS, n=0),
    _case("ag_collision_check", SHAPE, grid=BAD_GRID, n=0),
    _case("ag_collision_check", MODE, params=LONG_LINKS, n=0),
    _case("ag_collision_check", OK, params=LONG_LINKS, n=0, engine=EXACT),
    _case("ag_collision_check", OK, n=0, j1=None, engine=BAD_ENGINE),
    _case("ag_collision_check", NULL, j1=None),
    _case("ag_collision_check", NULL, hit=None, engine=BAD_ENGINE),
    _case("ag_collision_check", MODE, engine=BAD_ENGINE),
    _case("ag_collision_check", MODE, engine=-1),

    _case("ag_check_motion", SHAPE, m=-1, p=None, engine=BAD_ENGINE),
    _case("ag_check_motion", NULL, p=None),
    _case("ag_check_motion", NULL, g=None),
    _case("ag_check_motion", SHAPE, grid=BAD_GRID, m=0),
    _case("ag_check_motion", MODE, params=LONG_LINKS, m=0),
    _case("ag_check_motion", OK, m=0, goal=None, engine=BAD_ENGINE),
    _case("ag_check_motion", NULL, steps=None),
    _case("ag_check_motion", NULL, fc=None, goal=D + 8),
    _case("ag_check_motion", ALIGN, goal=D + 8),
    _case("ag_check_motion", ALIGN, last_free=D + 8, engine=BAD_ENGINE),
    _case("ag_check_motion", MODE, engine=BAD_ENGINE),

    _case("ag_cspace_occupancy", SHAPE, b1=0, p=None, engine=BAD_ENGINE),
    _case("ag_cspace_occupancy", SHAPE, b2=0),
    _case("ag_cspace_occupancy", NULL, g=None),
    _case("ag_cspace_occupancy", NULL, grid=NO_GRID_BITS, lo1=math.nan),
    _case("ag_cspace_occupancy", MODE, params=LONG_LINKS, lo1=math.inf),
    _case("ag_cspace_occupancy", SHAPE, step2=math.nan, bits=None),
    _case("ag_cspace_occupancy", SHAPE, grid={"n_grids": 1 << 30, "envs_per_grid": 256}, b1=1 << 30, b2=1 << 30,
          bits=None),
    _case("ag_cspace_occupancy", NULL, bits=None, fc=D + 4),
    _case("ag_cspace_occupancy", ALIGN, bits=D + 2),
    _case("ag_cspace_occupancy", ALIGN, fc=D + 4, engine=BAD_ENGINE),
    _case("ag_cspace_occupancy", MODE, engine=BAD_ENGINE),

    _case("ag_cspace_components", SHAPE, n_grids=-1, wrap=9, bits=None),
    _case("ag_cspace_components", SHAPE, b1=46341, b2=46341, wrap=9),
    _case("ag_cspace_components", SHAPE, n_grids=1 << 40, b1=1 << 15, b2=1 << 15, wrap=9),
    _case("ag_cspace_components", MODE, wrap=4, bits=None),
    _case("ag_cspace_components", MODE, wrap=9, n_grids=0),
    _case("ag_cspace_components", OK, n_grids=0, bits=None, nc=D + 4),
    _case("ag_cspace_components", NULL, labels=None, bits=D + 2),
    _case("ag_cspace_components", ALIGN, labels=D + 1),
    _case("ag_cspace_components", ALIGN, nc=D + 4),

    _case("ag_cspace_map", NULL, cmap=None, grid={"n_grids": 2}),
    _case("ag_cspace_map", NULL, p=None),
    _case("ag_cspace_map", SHAPE, grid={"n_grids": 2}, cmap=D + 8),
    _case("ag_cspace_map", SHAPE, grid={"S": 33, "words_per_row": 2, "bits": None}),
    _case("ag_cspace_map", ALIGN, cmap=D + 8, grid=NO_GRID_BITS),
    _case("ag_cspace_map", NULL, grid=NO_GRID_BITS),
    _case("ag_cspace_map", SHAPE, grid=BAD_GRID),
    _case("ag_cspace_map", MODE, params=LONG_LINKS),

    _case("ag_step", SHAPE, n=-1, p=None),
    _case("ag_step", NULL, g=None),
    _case("ag_step", SHAPE, grid=BAD_GRID, n=0),
    _case("ag_step", OK, n=0, actions=None, engine=BAD_ENGINE),
    _case("ag_step", NULL, flags=None, actions=D + 8),
    _case("ag_step", ALIGN, actions=D + 8),
    _case("ag_step", MODE, actions=D + 8, f32=1, engine=BAD_ENGINE),
    _case("ag_step", ALIGN, ee=D + 8, engine=BAD_ENGINE),
    _case("ag_step", ALIGN, targets=D + 8),
    _case("ag_step", MODE, engine=BAD_ENGINE),

    _case("ag_reset", SHAPE, n=-1, g=None),
    _case("ag_reset", NULL, p=None),
    _case("ag_reset", MODE, params=LONG_LINKS, n=0),
    _case("ag_reset", OK, n=0, reset_ctr=None),
    _case("ag_reset", NULL, clear_flags=1),
    _case("ag_reset", MODE, clear_flags=0, engine=BAD_ENGINE),
    _case("ag_reset", NULL, reset_ctr=None, reset_u=D, R=0),
    _case("ag_reset", SHAPE, reset_u=D + 8, R=0),
    _case("ag_reset", ALIGN, reset_u=D + 8, R=1, engine=BAD_ENGINE),
    _case("ag_reset", MODE, reset_u=D, R=1, engine=BAD_ENGINE),

    _case("ag_step_obs", SHAPE, crop=D, crop_size=4, p=None),
    _case("ag_step_obs", SHAPE, crop=D, crop_size=65),
    _case("ag_step_obs", MODE, crop=None, crop_size=4, engine=BAD_ENGINE),
    _case("ag_step_obs", NULL, g=None),
    _case("ag_step_obs", SHAPE, grid=BAD_GRID, n=0),
    _case("ag_step_obs", OK, n=0, obs=None),
    _case("ag_step_obs", NULL, collision=None, final_obs=D + 8),
    _case("ag_step_obs", ALIGN, final_obs=D + 8, engine=BAD_ENGINE),
    _case("ag_step_obs", ALIGN, actions=D + 8),
    _case("ag_step_obs", MODE, crop=D, crop_size=5, engine=BAD_ENGINE),

    _case("ag_rollout", NULL, args=None),
    _case("ag_rollout", NULL, p=None, K=0),
    _case("ag_rollout", SHAPE, K=0),
    _case("ag_rollout", SHAPE, K=65537),
    _case("ag_rollout", SHAPE, n=-1, j1=None),
    _case("ag_rollout", OK, n=0, j1=None, grid=BAD_GRID),
    _case("ag_rollout", NULL, stats=None),
    _case("ag_rollout", NULL, rec_j1=D),
    _case("ag_rollout", MODE, rec_j1=D, rec_j2=D, engine=BAD_ENGINE),
    _case("ag_rollout", NULL, events=D),
    _case("ag_rollout", SHAPE, reset_u=D, R=0, actions=D + 4),
    _case("ag_rollout", ALIGN, actions=D + 4, grid=BAD_GRID),
    _case("ag_rollout", ALIGN, targets=D + 8),
    _case("ag_rollout", SHAPE, grid=BAD_GRID),
    _case("ag_rollout", MODE, params=LONG_LINKS),
    _case("ag_rollout", MODE, engine=BAD_ENGINE),
]


@pytest.mark.parametrize("entry,args,status", STATUS_TABLE)
def test_status_table(lib, entry, args, status):
    """each entry point's status for rejected arguments, and which check comes first; nothing reaches the device"""
    from abstract_gym_b200 import _lib
    args = dict(args)
    p, g = _lib.default_params(), _grid()
    for k, v in args.pop("params", {}).items():
        setattr(p, k, v)
    for k, v in args.pop("grid", {}).items():
        setattr(g, k, v)
    p, g = args.pop("p", p), args.pop("g", g)
    assert CALLS[entry](lib, p, g, **args) == status


def test_product_does_not_touch_the_oracle():
    """the oracle is test infrastructure: nothing under abstract_gym_b200/ may reference it"""
    pkg = os.path.join(ROOT, "abstract_gym_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.lower() or f == "__none__", "%s mentions the oracle" % f


def test_no_device_means_loud_failure():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import abstract_gym_b200 as ag
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ag.BatchedTwoJointRobot([0.1], [0.2])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ag.TwoJointRobot(0.1, 0.2).end_effector()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ag.OccupancyGrid(size=9, random_obstacle=False).device_grid()


def test_reference_host_api_shapes(golden_dir):
    """OccupancyGrid keeps the reference's attributes, order and corner values (host, setup-time)."""
    import abstract_gym_b200 as ag
    z = np.load(os.path.join(golden_dir, "scene_cases.npz"))
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    occ, coord, obs, side = g.get_occupancy_grid()
    got = np.array([[o.min_x, o.min_y, o.max_x, o.max_y] for o in obs])
    assert np.array_equal(got, z["manual9/squares"]) and side == 0.2 and occ.shape == (9, 9)
    assert coord[0].tolist() == [0.40000000000000013, -0.19999999999999996]
    for name, S, p, seed in (("rand9", 9, 0.1, 11), ("rand31", 31, 0.01, 12), ("rand64", 64, 0.02, 13)):
        np.random.seed(seed)
        g = ag.OccupancyGrid(size=S, random_obstacle=True, obstacle_probability=p)
        got = np.array([[o.min_x, o.min_y, o.max_x, o.max_y] for o in g.obstacle_list])
        assert np.array_equal(got, z[name + "/squares"]) and np.array_equal(g.occ != 0, z[name + "/occ"] != 0)
    mat = np.array([[0, 0, 1, 0, 0], [0, 1, 1, 0, 0], [0, 1, 1, 0, 0], [0, 0, 0, 0, 0], [0, 1, 0, 0, 1]])
    g.load_from_matrix(mat)
    got = np.array([[o.min_x, o.min_y, o.max_x, o.max_y] for o in g.obstacle_list])
    assert np.array_equal(got, z["matrix5/squares"]) and g.size == 5
    g.load_from_matrix(np.zeros((3, 4)))      # prints "The matrix is not square." and leaves the grid alone
    assert g.size == 5
    g.load_from_matrix(np.zeros((4, 4)))      # empty grid accepted (the reference raises ValueError)
    assert g.obstacle_list == [] and g.size == 4


def test_ik_known_answer(golden_dir):
    import json
    import abstract_gym_b200 as ag
    k = json.load(open(os.path.join(golden_dir, "reference_goldens.json")))["known"]
    s1, s2 = ag.TwoJointRobot(0.0, 0.0).inverse_kinematic(ag.Point(0.5, 0.0))   # two_joint_robot.py:115-120
    assert s1.tolist() == k["ik_s1"] and s2.tolist() == k["ik_s2"]
