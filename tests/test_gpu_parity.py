"""GPU parity: the CUDA path (called through the C ABI via the Python host) against the CPU oracle
and the committed reference goldens.

Bar (BASELINE.json north_star): collision flags and first-hit cell indices bit-exact; joints,
end-effector positions and rewards within 1e-5 relative (TOL below; observed ~1e-16).
"""
import hashlib
import json
import os
import struct

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-5   # relative, north_star
ENGINES = ["exact", "fast", "brute"]


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


def rel_close(a, b, tol=TOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= tol * np.maximum(np.abs(b), 1e-3))


def random_grid(rng, S, p):
    occ = (rng.random((S, S)) < p).astype(np.uint8)
    return occ


def make_scene(ag, torch, occ_or_grid, j1, j2, **kw):
    if isinstance(occ_or_grid, np.ndarray):
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
        g.load_from_matrix(occ_or_grid)
    else:
        g = occ_or_grid
    rb = ag.BatchedTwoJointRobot(torch.as_tensor(j1, device="cuda"), torch.as_tensor(j2, device="cuda"))
    return ag.BatchedScene(rb, g, **kw)


# ------------------------------------------------------------------ goldens from the reference

def test_predicate_goldens(ag, golden_dir):
    z = np.load(os.path.join(golden_dir, "predicate_cases.npz"))
    out = ag.segment_square_arrays(z["seg"], z["sq"], want_abc=True, want_corner_values=True)
    nan_ok = np.isnan(z["abc"]) & np.isnan(out["abc"])
    assert np.all((out["abc"] == z["abc"]) | nan_ok)
    assert np.array_equal(np.sign(out["v"]), z["signs"])
    crash = z["out"] == 2
    assert np.array_equal(out["hit"][~crash], z["out"][~crash] == 1)
    assert out["axis_aligned"] == int(crash.sum())


def test_fk_goldens(ag, golden_dir):
    z = np.load(os.path.join(golden_dir, "fk_cases.npz"))
    fk = ag.forward_kinematics(z["j"][:, 0], z["j"][:, 1]).cpu().numpy()
    assert rel_close(fk, z["fk"])
    assert np.abs(fk - z["fk"]).max() < 1e-14   # CUDA sincos vs glibc: a few ulp


def test_collision_checker_main_block(ag):
    c = ag.CollisionChecker(ag.Line(ag.Point(0, 0), ag.Point(1, 2)), ag.Square(ag.Point(0, 0.8), ag.Point(0.9, 1.4)))
    assert c.collision_check() is True                      # utils/collision_checker.py:94-96
    assert (c.a, c.b, c.c) == (1.0, -0.5, 0.0)
    rb = ag.TwoJointRobot(0.3, 1.2)
    assert rel_close([rb.end_effector().x, rb.end_effector().y], [0.4908419219932445, 0.39781980845470366], 1e-14)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["manual9", "rand9", "rand31", "rand64", "rand6", "matrix5"])
def test_scene_step_goldens(ag, torch_, golden_dir, name, engine):
    z = np.load(os.path.join(golden_dir, "scene_cases.npz"))
    occ = z[name + "/occ"]
    j0, acts, out, fh, ee = (z[name + "/" + k] for k in ("j0", "actions", "out", "first_hit", "ee"))
    sc = make_scene(ag, torch_, occ, j0[:, 0], j0[:, 1], engine=engine)
    for t in range(acts.shape[1]):
        j1, j2, rw, done, coll, extra = sc.step(torch_.as_tensor(acts[:, t], device="cuda"), want_ee=True,
                                                want_first_hit=(engine != "fast"))
        assert np.array_equal(j1.cpu().numpy(), out[:, t, 0]) and np.array_equal(j2.cpu().numpy(), out[:, t, 1])
        assert np.array_equal(rw.cpu().numpy().astype(np.float64), out[:, t, 2])
        assert np.array_equal(done.cpu().numpy(), out[:, t, 3] != 0)
        assert np.array_equal(coll.cpu().numpy(), out[:, t, 4] != 0)
        assert rel_close(extra["ee"].cpu().numpy(), ee[:, t])
        if engine != "fast":
            hit_now, fh_now = sc.collision_check(first_hit=True)
            assert np.array_equal(fh_now.cpu().numpy(), fh[:, t])
            assert np.array_equal(extra["first_hit"].cpu().numpy(), fh[:, t])


@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_reach_sequences(ag, torch_, golden_dir, engine):
    z = np.load(os.path.join(golden_dir, "scene_cases.npz"))
    start, seq = z["reach/start"], z["reach/seq"]
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sc = make_scene(ag, torch_, g, start[:, 0], start[:, 1], engine=engine)
    for t in range(seq.shape[1]):
        j1, j2, rw, done, coll = sc.step(torch_.as_tensor(seq[:, t, 0:2].copy(), device="cuda"))
        assert np.array_equal(j1.cpu().numpy(), seq[:, t, 2])
        assert np.array_equal(rw.cpu().numpy().astype(np.float64), seq[:, t, 4])
        assert np.array_equal(done.cpu().numpy(), seq[:, t, 5] != 0)
        assert np.array_equal(coll.cpu().numpy(), seq[:, t, 6] != 0)
    assert (seq[:, :, 5] != 0).any()


@pytest.mark.parametrize("idx", [0, 1, 2])
def test_scene_dropin_reproduces_reference_digest(ag, golden_dir, idx):
    """experiment/experiment_0.py:13-34 run through OUR Scene/TwoJointRobot/OccupancyGrid with the
    reference's seed must give the reference's sha256 (SURVEY.md section 8c goldens)."""
    g = json.load(open(os.path.join(golden_dir, "reference_goldens.json")))["experiment0"][idx]
    steps = 6000 if idx else g["steps"]          # full 20 000 steps for seed 0, a prefix check for the others
    np.random.seed(g["seed"])
    rob = ag.TwoJointRobot(joint_1=1.0, joint_2=2.5)
    occ = ag.OccupancyGrid(size=9, random_obstacle=False)
    s = ag.Scene(robot=rob, env=occ, visualize=False)
    s.random_valid_pose()
    h = hashlib.sha256()
    resets = []
    for i in range(steps):
        a = s.sample_action(scale_factor=0.1)
        j1, j2, r, d, c = s.step(a)
        h.update(struct.pack("<5d2B", j1, j2, a[0], a[1], r, d, c))
        if i == 0:
            assert [float(j1), float(j2), float(a[0]), float(a[1])] == g["first_record"][:4]
        if d or c:
            resets.append(i)
            s.reset()
    assert resets == [r for r in g["resets"] if r < steps]
    if steps == g["steps"]:
        assert h.hexdigest() == g["sha256"]
        assert [float(rob.joint_1), float(rob.joint_2)] == g["final_joints"]


# ------------------------------------------------------------------ config 2: 4096 envs, 1 step, vs oracle

@pytest.mark.parametrize("engine", ENGINES)
def test_config2_4096_envs_one_step(ag, torch_, oracle, engine):
    rng = np.random.default_rng(42)
    n = 4096
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = (rng.random((n, 2)) - 0.5) * 0.1
    sq, ci = oracle.manual_grid()
    o1, o2 = j1.copy(), j2.copy()
    rw, fl = np.zeros(n), np.zeros(n, dtype=np.uint8)
    ref = oracle.step_batch(o1, o2, acts, rw, fl, sq, ci)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sc = make_scene(ag, torch_, g, j1, j2, engine=engine)
    d1, d2, drw, ddone, dcoll, extra = sc.step(torch_.as_tensor(acts, device="cuda"), want_ee=True,
                                               want_first_hit=(engine != "fast"))
    assert np.array_equal(d1.cpu().numpy(), o1) and np.array_equal(d2.cpu().numpy(), o2)
    assert np.array_equal(dcoll.cpu().numpy(), (fl & 1) != 0)          # bit-exact flags
    assert np.array_equal(ddone.cpu().numpy(), (fl & 2) != 0)
    assert np.array_equal(drw.cpu().numpy().astype(np.float64), rw)
    assert rel_close(extra["ee"].cpu().numpy(), ref["ee"]) and rel_close(extra["dist"].cpu().numpy(), ref["dist"])
    if engine != "fast":
        assert np.array_equal(extra["first_hit"].cpu().numpy(), ref["first_hit"])   # bit-exact cell indices
    assert 300 < int((fl & 1).sum()) < 800


# ------------------------------------------------------------------ engines agree at scale (size-independent property)

@pytest.mark.parametrize("S,p,n", [(9, None, 1 << 21), (9, 0.1, 1 << 20), (31, 0.01, 1 << 20), (6, 0.06, 1 << 19),
                                   (64, 0.02, 1 << 20), (256, 0.008, 1 << 19), (1024, 0.002, 1 << 18)])
def test_engines_agree_at_scale(ag, torch_, S, p, n):
    """EXACT traversal == FAST filter == BRUTE (every occupied cell, the reference's loop) on millions
    of uniform poses: 0 mismatches allowed."""
    rng = np.random.default_rng(S * 1000 + 7)
    if p is None:
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
    else:
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
        g.load_from_matrix(random_grid(rng, S, p))
    gen = torch_.Generator(device="cuda").manual_seed(S)
    rb = ag.BatchedTwoJointRobot.random(n, device="cuda", generator=gen)
    sc = ag.BatchedScene(rb, g)
    hit_e, fh_e = sc.collision_check(first_hit=True, engine="exact")
    hit_f = sc.collision_check(engine="fast")
    nb = n if S <= 256 else 1 << 15
    sc_b = ag.BatchedScene(ag.BatchedTwoJointRobot(rb.joint_1[:nb], rb.joint_2[:nb]), g)
    hit_b, fh_b = sc_b.collision_check(first_hit=True, engine="brute")
    assert int((hit_e != hit_f).sum().item()) == 0
    assert int((hit_e[:nb] != hit_b).sum().item()) == 0
    assert int((fh_e[:nb] != fh_b).sum().item()) == 0
    frac = float(hit_e.float().mean().item())
    assert 0.01 < frac < 0.99, frac


@pytest.mark.parametrize("S,p", [(9, None), (31, 0.01), (256, 0.008)])
def test_collision_vs_oracle_large(ag, torch_, oracle, S, p):
    rng = np.random.default_rng(S + 1)
    n = 200000 if S <= 31 else 20000
    if p is None:
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
        sq, ci = oracle.manual_grid()
    else:
        occ = random_grid(rng, S, p)
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
        g.load_from_matrix(occ)
        sq, ci = oracle.grid_squares(occ)
    j1, j2 = rng.uniform(-10, 10, n), rng.uniform(-10, 10, n)
    hit, fh, mg = oracle.collision_batch(j1, j2, sq, ci, want_margin=True)
    sc = make_scene(ag, torch_, g, j1, j2)
    for engine in ("exact", "fast"):
        dh, dfh = sc.collision_check(first_hit=True, engine=engine)
        bad = dh.cpu().numpy() != (hit != 0)
        # north_star accounting: mismatches with an oracle decision margin < 1e-6 m are boundary-excused
        hard = int((bad & (mg >= 1e-6)).sum())
        assert hard == 0 and int(bad.sum()) == 0, (engine, int(bad.sum()), hard)
        assert np.array_equal(dfh.cpu().numpy(), fh)


# ------------------------------------------------------------------ K4 rollouts vs oracle

def _rollout_case(ag, torch, oracle, occs, n, K, engine, scripted, envs_per_grid=None, seed=9, R=24, p_manual=False):
    rng = np.random.default_rng(1000 + n + K)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    if p_manual:
        grids_sq = [oracle.manual_grid()[0]]
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
    elif len(occs) == 1:
        grids_sq = [oracle.grid_squares(occs[0])[0]]
        g = ag.OccupancyGrid(size=9, random_obstacle=False)
        g.load_from_matrix(occs[0])
    else:
        grids_sq = [oracle.grid_squares(o)[0] for o in occs]
        g = ag.BatchedOccupancyGrid(torch.as_tensor(np.stack(occs), device="cuda"), envs_per_grid)
    actions = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32) if scripted else None
    reset_u = rng.random((n, R, 2)) if scripted else None
    # oracle
    st = oracle.RolloutState(j1, j2)
    p = oracle.default_params()
    rec, stats = oracle.rollout(st, K, grids_sq, envs_per_grid=envs_per_grid, env_id0=0, seed=seed,
                                actions_f32=actions, reset_u=reset_u, params=p)
    # device
    sc = make_scene(ag, torch, g, j1, j2, engine=engine, seed=seed)
    drec = sc.rollout(K, actions=None if actions is None else torch.as_tensor(actions, device="cuda"),
                      reset_u=None if reset_u is None else torch.as_tensor(reset_u, device="cuda"))
    torch.cuda.synchronize()
    assert np.array_equal(drec["flags"].cpu().numpy(), rec["flags"])
    assert np.array_equal(drec["reward"].cpu().numpy(), rec["reward"])
    assert np.array_equal(drec["j1"].cpu().numpy(), rec["j1"]) and np.array_equal(drec["j2"].cpu().numpy(), rec["j2"])
    assert np.array_equal(sc.robot.joint_1.cpu().numpy(), st.j1) and np.array_equal(sc.robot.joint_2.cpu().numpy(), st.j2)
    assert np.array_equal(sc.step_ctr.cpu().numpy().view(np.uint32), st.step_ctr)
    assert np.array_equal(sc.reset_ctr.cpu().numpy().view(np.uint32), st.reset_ctr)
    assert np.array_equal(sc.ep_len.cpu().numpy().view(np.uint32), st.ep_len)
    assert np.array_equal(sc.flags.cpu().numpy(), st.flags)
    assert np.array_equal(sc.stats.cpu().numpy(), stats)
    return stats


@pytest.mark.parametrize("engine", ["exact", "fast"])
@pytest.mark.parametrize("scripted", [True, False])
def test_rollout_scene0_vs_oracle(ag, torch_, oracle, engine, scripted):
    stats = _rollout_case(ag, torch_, oracle, None, 4096, 64, engine, scripted, p_manual=True)
    assert stats[oracle.ST_ENV_STEPS] == 4096 * 64 and stats[oracle.ST_EPISODES] > 100


@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_rollout_ragged_and_tiny(ag, torch_, oracle, engine):
    for n, K in ((1, 5), (31, 3), (257, 17), (1000, 1)):
        _rollout_case(ag, torch_, oracle, None, n, K, engine, True, p_manual=True)


@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_rollout_config4_highres_grid(ag, torch_, oracle, engine):
    rng = np.random.default_rng(4)
    occ = random_grid(rng, 1024, 0.002)
    stats = _rollout_case(ag, torch_, oracle, [occ], 1024, 8, engine, False, seed=3)
    assert stats[oracle.ST_EPISODES] > 0


@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_rollout_config5_heterogeneous_grids(ag, torch_, oracle, engine):
    rng = np.random.default_rng(5)
    occs = [random_grid(rng, 256, 0.008) for _ in range(8)]
    stats = _rollout_case(ag, torch_, oracle, occs, 2048, 16, engine, False, envs_per_grid=256, seed=11)
    assert stats[oracle.ST_EPISODES] > 0
    # envs_per_grid not a multiple of the block: per-thread grid lookup path
    _rollout_case(ag, torch_, oracle, occs[:3], 900, 6, engine, True, envs_per_grid=100, seed=12)


def test_rollout_dense_grid_counts_stuck_resets(ag, torch_, oracle):
    rng = np.random.default_rng(6)
    occ = random_grid(rng, 31, 0.5)          # almost no free pose: bounded rejection sampling gives up and counts
    stats = _rollout_case(ag, torch_, oracle, [occ], 512, 4, "fast", False, seed=2)
    assert stats[oracle.ST_STUCK_RESETS] > 0


def test_empty_grid_never_collides(ag, torch_):
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    g.load_from_matrix(np.zeros((9, 9)))     # the reference raises ValueError here (occupancy_grid.py:64)
    rb = ag.BatchedTwoJointRobot.random(10000, device="cuda")
    sc = ag.BatchedScene(rb, g)
    for e in ENGINES:
        assert int(sc.collision_check(engine=e).sum().item()) == 0
    sc.rollout(8, record=False)
    st = sc.stats_dict()
    assert st["collisions"] == 0 and st["env_steps"] == 80000


# ------------------------------------------------------------------ K3 / K5 / pipeline / sharding

def test_reset_kernel_vs_reference_semantics(ag, torch_, oracle):
    rng = np.random.default_rng(8)
    n, R = 5000, 16
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    u = rng.random((n, R, 2))
    sq, ci = oracle.manual_grid()
    hit, _, _ = oracle.collision_batch(j1, j2, sq, ci)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sc = make_scene(ag, torch_, g, j1, j2)
    sc.flags.fill_(3); sc.step_reward.fill_(-1000.0)
    mask = (np.arange(n) % 3 != 0)
    sc.reset(mask=torch_.as_tensor(mask, device="cuda"), reset_u=torch_.as_tensor(u, device="cuda"))
    d1, d2 = sc.robot.joint_1.cpu().numpy(), sc.robot.joint_2.cpu().numpy()
    rc = sc.reset_ctr.cpu().numpy()
    # expected: scene_0.py:179-181 -- resample only while colliding, candidates in order, (u*pi)*2.0
    e1, e2, erc = j1.copy(), j2.copy(), np.zeros(n, dtype=np.int32)
    for e in np.nonzero(mask & (hit != 0))[0]:
        k = 0
        while True:
            e1[e], e2[e] = u[e, k, 0] * np.pi * 2.0, u[e, k, 1] * np.pi * 2.0
            k += 1
            if not oracle.collision_batch(e1[e:e + 1], e2[e:e + 1], sq, ci)[0][0]:
                break
        erc[e] = k
    assert np.array_equal(d1, e1) and np.array_equal(d2, e2) and np.array_equal(rc, erc)
    fl = sc.flags.cpu().numpy()
    assert np.all(fl[mask] == 0) and np.all(fl[~mask] == 3)      # a non-colliding pose is kept, flags cleared
    assert int(sc.collision_check().cpu().numpy()[mask].sum()) == 0


def test_device_grid_pack_matches_host(ag, torch_):
    rng = np.random.default_rng(9)
    for S in (5, 9, 33, 256):
        occ = (rng.random((3, S, S)) < 0.2).astype(np.uint8)
        dg = ag.DeviceGrid.from_device_matrices(torch_.as_tensor(occ, device="cuda"))
        assert np.array_equal(dg.unpack(), occ)
        hg = ag.DeviceGrid.from_host_matrix(occ[1], device="cuda")
        assert np.array_equal(hg.unpack()[0], occ[1])


def test_rollout_host_pipeline_equals_device_rollout(ag, torch_):
    n, K = 5000, 12
    rng = np.random.default_rng(10)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    a = make_scene(ag, torch_, g, j1, j2, seed=4)
    b = make_scene(ag, torch_, g, j1, j2, seed=4)
    ra = a.rollout(K, actions=torch_.as_tensor(acts, device="cuda"))
    hact = torch_.as_tensor(acts).pin_memory()
    out = b.alloc_records(K, pinned_host=True)
    st = b.rollout_host(K, hact, out, chunk_envs=1024)
    for k in ("j1", "j2", "reward", "flags"):
        assert np.array_equal(ra[k].cpu().numpy(), out[k].numpy()), k
    assert np.array_equal(a.robot.joint_1.cpu().numpy(), b.robot.joint_1.cpu().numpy())
    assert a.stats_dict() == b.stats_dict() == st
    # statistics-only, in-kernel actions
    a.rollout(K, record=False); b.rollout_host(K, None, None, chunk_envs=2048)
    assert a.stats_dict() == b.stats_dict()
    assert np.array_equal(a.robot.joint_2.cpu().numpy(), b.robot.joint_2.cpu().numpy())


def test_shard_invariance_on_device(ag, torch_):
    """two shards with global env ids == one launch over all envs (Philox keyed by global id)"""
    n, K = 6000, 20
    rng = np.random.default_rng(11)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    occs = np.stack([random_grid(rng, 64, 0.02) for _ in range(6)])
    g = ag.BatchedOccupancyGrid(torch_.as_tensor(occs, device="cuda"), envs_per_grid=512)
    full = make_scene(ag, torch_, g, j1, j2, seed=21)
    rf = full.rollout(K)
    from abstract_gym_b200.sharding import shard_range
    tot = torch_.zeros_like(full.stats)
    for r in range(3):
        lo, hi = shard_range(n, r, 3)
        sh = make_scene(ag, torch_, g, j1[lo:hi], j2[lo:hi], seed=21, env_id0=lo)
        rs = sh.rollout(K)
        assert torch_.equal(rs["flags"], rf["flags"][:, lo:hi]) and torch_.equal(rs["j1"], rf["j1"][:, lo:hi])
        tot += sh.stats
    assert torch_.equal(tot, full.stats)


def test_fast_fk_error_budget(ag, torch_):
    """the float32 FK of the FAST engine stays inside AG_DELTA_P = 3e-7 m of the float64 FK;
    checked indirectly: FAST == EXACT on 2^22 poses of a dense-ish grid (0 mismatches)"""
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    rng = np.random.default_rng(12)
    g.load_from_matrix(random_grid(rng, 48, 0.05))
    gen = torch_.Generator(device="cuda").manual_seed(99)
    u = torch_.rand(2, 1 << 22, dtype=torch_.float64, device="cuda", generator=gen)
    rb = ag.BatchedTwoJointRobot((u[0] - 0.5) * 2000.0, (u[1] - 0.5) * 2000.0)     # |j| up to 1000 rad
    sc = ag.BatchedScene(rb, g)
    assert int((sc.collision_check(engine="exact") != sc.collision_check(engine="fast")).sum().item()) == 0


# ------------------------------------------------------------------ the reference's data product (SURVEY 8f.1)

@pytest.mark.gpu
@pytest.mark.parametrize("name,seed", [("dense9_seed3", 3), ("dense9_seed4", 4)])
def test_dropin_loop_reproduces_reference_data_list(ag, golden_dir, tmp_path, name, seed):
    """experiment_0.py:11-37,54-57 with the drop-in classes, seeded like oracle/make_golden_datalist.py:
    the exported data_list.txt equals the file the UNMODIFIED reference wrote, byte for byte."""
    from abstract_gym_b200.experiment.experiment_0 import Trajectories
    occ_m = np.load(os.path.join(golden_dir, "data_list_dense9_occ.npy"))
    np.random.seed(seed)
    rob = ag.TwoJointRobot(joint_1=1.0, joint_2=2.5)
    occ = ag.OccupancyGrid(size=9, random_obstacle=False, obstacle_probability=0.01)
    occ.load_from_matrix(occ_m)
    s = ag.Scene(robot=rob, env=occ, visualize=False)
    s.random_valid_pose()
    rows = []
    for i in range(400):
        action = s.sample_action(scale_factor=0.1)
        j1, j2, step_reward, done, collision = s.step(action)
        rows.append([j1, j2, action[0], action[1], step_reward, (1 if collision else 0) | (2 if done else 0)])
        if done or collision:
            s.reset()
    a = np.array(rows, dtype=np.float64)
    col = lambda i: a[:, i:i + 1].copy()
    tr = Trajectories(col(0), col(1), col(2), col(3), col(4), a[:, 5:6].astype(np.uint8))
    out = tmp_path / "data_list.txt"
    tr.export_text(str(out), numpy2=True)
    assert out.read_bytes() == open(os.path.join(golden_dir, "data_list_%s.txt" % name), "rb").read()


@pytest.mark.gpu
def test_experiment_drivers_fast_equals_exact(ag, torch_):
    """run_experiment (fused rollout, float32 records) and run_experiment_exact (step + masked reset, float64)
    produce the same episodes on the same actions and reset candidates"""
    from abstract_gym_b200.experiment.experiment_0 import run_experiment, run_experiment_exact
    n, K, R = 3000, 40, 24
    rng = np.random.default_rng(21)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    fast = run_experiment(make_scene(ag, torch_, g, j1, j2, seed=6), K, chunk_steps=16, actions=acts)
    exact = run_experiment_exact(make_scene(ag, torch_, g, j1, j2, seed=6), K, actions=acts.astype(np.float64))
    assert np.array_equal(fast.flags, exact.flags) and np.array_equal(fast.reward, exact.reward)
    assert np.array_equal(fast.j1, exact.j1.astype(np.float32)) and np.array_equal(fast.j2, exact.j2.astype(np.float32))
    assert fast.episode_index().tolist() == exact.episode_index().tolist() and len(fast.episode_index()) > 20
    # in-kernel actions through the zero-H2D event path: the recorded float64 actions replay to the same episodes
    fast2 = run_experiment(make_scene(ag, torch_, g, j1, j2, seed=6), K, chunk_steps=16)
    acts64 = np.stack([fast2.a0, fast2.a1], axis=-1)
    exact2 = run_experiment_exact(make_scene(ag, torch_, g, j1, j2, seed=6), K, actions=acts64)
    assert np.array_equal(fast2.flags, exact2.flags) and np.array_equal(fast2.reward, exact2.reward)
    assert np.array_equal(fast2.j1, exact2.j1.astype(np.float32)) and len(fast2.episode_index()) > 20


@pytest.mark.gpu
def test_checkpoint_resume_is_bit_exact(ag, torch_, tmp_path):
    """state_dict -> torch.save -> load_state_dict: the resumed rollout (in-kernel Philox actions and resets)
    equals the uninterrupted one"""
    n = 4096
    rng = np.random.default_rng(31)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    a = make_scene(ag, torch_, g, j1, j2, seed=8, env_id0=1000)
    a.rollout(24, record=False)
    path = str(tmp_path / "ckpt.pt")
    torch_.save(a.state_dict(), path)
    ra = a.rollout(40)
    b = make_scene(ag, torch_, g, np.zeros(n), np.zeros(n), seed=0)
    b.load_state_dict(torch_.load(path))
    rb = b.rollout(40)
    for k in ("j1", "j2", "reward", "flags"):
        assert torch_.equal(ra[k], rb[k]), k
    assert torch_.equal(a.robot.joint_1, b.robot.joint_1) and torch_.equal(a.reset_ctr, b.reset_ctr)
    assert a.stats_dict() == b.stats_dict() and a.stats_dict()["episodes"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_vector_env_matches_scene_loop(ag, torch_, oracle, graph):
    """VectorEnv.step == BatchedScene.step + masked reset (the experiment_0 loop), eager and as a CUDA graph;
    observations carry the float64 end effector and the goal distance of check_target_reached"""
    n, T = 2048, 30
    env = ag.VectorEnv(n, device="cuda", seed=5)
    ref = ag.VectorEnv(n, device="cuda", seed=5)
    obs0, obs0r = env.reset().clone(), ref.reset().clone()
    assert torch_.equal(obs0, obs0r)
    assert not bool(env.scene.collision_check().any())
    ex, ey, gx, gy = oracle.forward_kinematics(float(obs0[7, 0]), float(obs0[7, 1]))
    assert rel_close(obs0[7, 2:4].cpu().numpy(), np.array([gx, gy]))
    assert rel_close(obs0[7, 4:6].cpu().numpy(), np.abs(np.array([-0.2 - gx, -0.3 - gy])))
    if graph:
        env.capture()
    gen = torch_.Generator(device="cuda").manual_seed(17)
    sc = ref.scene
    n_term = 0
    for t in range(T):
        a = (torch_.rand(n, 2, dtype=torch_.float64, device="cuda", generator=gen) - 0.5) * 0.1
        obs, rw, term, trunc, info = env.step(a)
        j1, j2, r2, done, coll = sc.step(a)
        assert torch_.equal(rw, r2) and torch_.equal(term, done | coll) and torch_.equal(info["collision"], coll)
        assert torch_.equal(info["final_obs"][:, 0], j1) and not bool(trunc.any())
        m = sc.flags != 0
        n_term += int(m.sum().item())
        sc.reset(mask=m)
        assert torch_.equal(obs[:, 0], sc.robot.joint_1) and torch_.equal(obs[:, 1], sc.robot.joint_2)
    assert n_term > 20 and env.stats()["episodes"] == n_term and env.stats()["env_steps"] == ref.stats()["env_steps"]


@pytest.mark.gpu
def test_batched_ik_and_move_to_joint_pose_vs_reference(ag, torch_, golden_dir):
    """robot/two_joint_robot.py:49-113 over arrays vs fixtures from the live reference: reachability flags
    equal, joint solutions within 1e-12 (north_star asks 1e-5 relative), move_to_joint_pose bit-exact"""
    z = np.load(os.path.join(golden_dir, "ik_cases.npz"))
    rb = ag.BatchedTwoJointRobot(torch_.zeros(1, dtype=torch_.float64, device="cuda"),
                                 torch_.zeros(1, dtype=torch_.float64, device="cuda"))
    valid, s1, s2 = rb.inverse_kinematic(torch_.as_tensor(z["target"], device="cuda"))
    v = valid.cpu().numpy()
    assert np.array_equal(v, z["valid"] != 0)
    sol = np.concatenate([s1.cpu().numpy(), s2.cpu().numpy()], axis=1)
    assert np.max(np.abs(sol[v] - z["sol"][v])) < 1e-12 and np.all(sol[~v] == 0)
    # corrected variant: FK of the solution lands on the target also for y < 0
    tgt = z["target"][v]
    _, c1, c2 = rb.inverse_kinematic(torch_.as_tensor(tgt, device="cuda"), corrected=True)
    for c in (c1, c2):
        ee = ag.forward_kinematics(c[:, 0].contiguous(), c[:, 1].contiguous())[:, 2:4].cpu().numpy()
        assert np.max(np.abs(ee - tgt)) < 1e-7      # acos is ill-conditioned at the rim of the annulus (sqrt(eps))
    # one launch per distinct step count (steps is a launch parameter)
    for st in np.unique(z["steps"]):
        sel = np.nonzero(z["steps"] == st)[0]
        sub = ag.BatchedTwoJointRobot(torch_.as_tensor(z["start"][sel, 0].copy(), device="cuda"),
                                      torch_.as_tensor(z["start"][sel, 1].copy(), device="cuda"))
        sub.move_to_joint_pose(torch_.as_tensor(z["goal"][sel].copy(), device="cuda"), steps=int(st))
        assert np.array_equal(sub.joint_1.cpu().numpy(), z["end"][sel, 0])
        assert np.array_equal(sub.joint_2.cpu().numpy(), z["end"][sel, 1])


@pytest.mark.gpu
def test_tangency_band_all_engines_and_oracle(ag, torch_, oracle):
    """scene_0's link 1 (0.4 m) is tangent to the squares starting at x = 0.40000000000000013 and y = 0.4: poses
    within a few mrad of j1 = 0 / pi/2 are where the float32 filter cannot decide and the float64 filter
    (narrow_f64) takes over.  FAST == EXACT == BRUTE == oracle on a dense sample of that band, including
    the exactly axis-aligned poses."""
    rng = np.random.default_rng(123)
    n = 1 << 18
    base = rng.choice([0.0, np.pi / 2, np.pi, -np.pi / 2, 2 * np.pi, 5 * np.pi / 2], n)
    eps = rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-13, -2.3, n)
    eps[: n // 64] = 0.0
    j1 = base + eps
    j2 = rng.uniform(0, 2 * np.pi, n)
    j2[::7] = j1[::7] + rng.choice([0.0, np.pi / 2, np.pi], len(j1[::7])) + rng.normal(0, 1e-6, len(j1[::7]))
    sq, ci = oracle.manual_grid()
    hit, fh, mg = oracle.collision_batch(j1, j2, sq, ci, want_margin=True)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sc = make_scene(ag, torch_, g, j1, j2)
    res = {e: sc.collision_check(engine=e).cpu().numpy() for e in ("exact", "fast", "brute")}
    assert np.array_equal(res["exact"], res["brute"])
    assert np.array_equal(res["fast"], res["exact"])
    # vs the CPU oracle: the only difference left is glibc sin/cos (the reference's) vs CUDA sincos, <= 2 ulp, which
    # can flip a decision that sits within ~1e-16 m of its threshold -- this sample is built on exactly those
    # thresholds.  north_star accounting: mismatches with an oracle margin < 1e-6 m are counted, others forbidden.
    bad = res["exact"] != (hit != 0)
    hard = bad & (mg >= 1e-6)
    print("tangency band: %d boundary-excused mismatches of %d poses (max margin %.3g m), %d hard"
          % (int(bad.sum()), n, float(mg[bad].max()) if bad.any() else 0.0, int(hard.sum())))
    assert int(hard.sum()) == 0 and int(bad.sum()) <= 32 and (not bad.any() or float(mg[bad].max()) < 1e-12)
    assert 0.05 < res["exact"].mean() < 0.95


@pytest.mark.gpu
def test_torch_custom_ops_equal_object_api(ag, torch_):
    """torch.ops.abstract_gym_b200.* -- the COMPILED op library (csrc/ag_torch_ops.cpp over the same C symbols) ==
    BatchedScene, on scene_0's map and on per-batch 256x256 maps in the two-level form, scripted reset candidates,
    per-env targets, a statistics-only rollout and the filter diagnostics; CPU tensors are refused."""
    import time
    from abstract_gym_b200 import ops, build
    assert os.path.exists(build.OPS_LIB)
    O = torch_.ops.abstract_gym_b200
    n, K = 3072, 20
    rng = np.random.default_rng(41)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = torch_.as_tensor(((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32), device="cuda")
    ru = torch_.as_tensor(rng.random((n, 12, 2)), device="cuda")
    tg = torch_.as_tensor(np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.5, 0.5, n)], axis=1), device="cuda")
    occs = [random_grid(rng, 256, 0.008) for _ in range(n // 256)]
    for kind in ("scene0", "c5"):
        g = ag.OccupancyGrid(size=9, random_obstacle=False) if kind == "scene0" else \
            ag.BatchedOccupancyGrid(torch_.as_tensor(np.stack(occs), device="cuda"), 256)
        ref = make_scene(ag, torch_, g, j1, j2, seed=3)
        rec = ref.rollout(K, actions=acts, reset_u=ru, targets=tg)
        sc = make_scene(ag, torch_, g, j1, j2, seed=3)         # only used as a bag of correctly typed state tensors
        dg = sc.grid
        assert (dg.hier is not None) == (kind == "c5")
        P, GA = ops.pack_params(sc.params()), ops.grid_args(dg)
        out = sc.alloc_records(K)
        hit = torch_.empty(n, dtype=torch_.uint8, device="cuda")
        O.collision_check(P, *GA, sc.robot.joint_1, sc.robot.joint_2, hit, None, 0, 1)
        assert torch_.equal(hit != 0, make_scene(ag, torch_, g, j1, j2).collision_check())
        diag = torch_.zeros(3, dtype=torch_.int64, device="cuda")
        O.rollout(P, *GA, sc.robot.joint_1, sc.robot.joint_2, sc.step_reward, sc.flags, sc.step_ctr, sc.reset_ctr, sc.ep_len,
                  acts, ru, tg, out["j1"], out["j2"], out["reward"], out["flags"], sc.stats, diag, None, None, K, 3, 0, 1)
        for k in ("j1", "j2", "reward", "flags"):
            assert torch_.equal(rec[k], out[k]), (kind, k)
        assert torch_.equal(ref.stats, sc.stats) and torch_.equal(ref.robot.joint_1, sc.robot.joint_1)
        assert torch_.equal(ref.reset_ctr, sc.reset_ctr)
        # statistics only, in-kernel actions
        ref.rollout(K, record=False)
        O.rollout(P, *GA, sc.robot.joint_1, sc.robot.joint_2, sc.step_reward, sc.flags, sc.step_ctr, sc.reset_ctr, sc.ep_len,
                  None, None, None, None, None, None, None, sc.stats, None, None, None, K, 3, 0, 1)
        assert torch_.equal(ref.stats, sc.stats) and torch_.equal(ref.robot.joint_2, sc.robot.joint_2)
        # one step + masked reset through the ops == through the object API
        a1 = (torch_.rand(n, 2, dtype=torch_.float64, device="cuda") - 0.5) * 0.1
        ref.step(a1, targets=tg); m = (ref.flags != 0).to(torch_.uint8); ref.reset(mask=m)
        O.step(P, *GA, sc.robot.joint_1, sc.robot.joint_2, a1, sc.step_reward, sc.flags, None, None, None, sc.stats, tg, 0, 1)
        m2 = (sc.flags != 0).to(torch_.uint8)
        O.reset(P, *GA, sc.robot.joint_1, sc.robot.joint_2, sc.step_reward, sc.flags, sc.reset_ctr, m2, None, sc.stats, 3, True, 0, 1)
        assert torch_.equal(m, m2) and torch_.equal(ref.robot.joint_1, sc.robot.joint_1) and torch_.equal(ref.stats, sc.stats)
    with pytest.raises((RuntimeError, NotImplementedError)):
        O.collision_check(P, *GA, sc.robot.joint_1.cpu(), sc.robot.joint_2.cpu(), hit.cpu(), None, 0, 1)
    with pytest.raises(RuntimeError):
        O.collision_check(P, *GA, sc.robot.joint_1.float(), sc.robot.joint_2, hit, None, 0, 1)
    # host overhead of one op call (validation + stream lookup + the launch itself), tiny kernel
    small = make_scene(ag, torch_, ag.OccupancyGrid(size=9, random_obstacle=False), j1[:64], j2[:64])
    GS, h64 = ops.grid_args(small.grid), torch_.empty(64, dtype=torch_.uint8, device="cuda")
    for _ in range(200):
        O.collision_check(P, *GS, small.robot.joint_1, small.robot.joint_2, h64, None, 0, 1)
    torch_.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2000):
        O.collision_check(P, *GS, small.robot.joint_1, small.robot.joint_2, h64, None, 0, 1)
    dt_op = (time.perf_counter() - t0) / 2000
    torch_.cuda.synchronize()
    print("torch op call: %.1f us per call (host side, includes the kernel launch)" % (dt_op * 1e6))
    assert dt_op < 50e-6


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_vector_env_vs_oracle(ag, torch_, oracle, graph):
    """VectorEnv (one fused K6 launch per step) against the oracle's Scene.step + the reference's reset rule
    (scene_0.py:105-113,174-181 with Philox stream-1 candidates) for 40 steps, eager and as a CUDA graph: joints,
    reward, terminated, collision, observations of restarted envs, the occupancy crop and the episode statistics."""
    n, T, seed = 4096, 40, 21
    env = ag.VectorEnv(n, device="cuda", seed=seed, crop_size=3)
    obs = env.reset().clone()
    sq, ci = oracle.manual_grid()
    j1, j2 = env.scene.robot.joint_1.cpu().numpy().copy(), env.scene.robot.joint_2.cpu().numpy().copy()
    rc = env.scene.reset_ctr.cpu().numpy().view(np.uint32).astype(np.int64).copy()
    rw, fl = np.zeros(n), np.zeros(n, dtype=np.uint8)
    if graph:
        env.capture()
        assert torch_.equal(env._obs, obs)                    # capture() leaves the caller's observation untouched
    rng = np.random.default_rng(33)
    episodes = 0
    occ = np.zeros((9, 9), dtype=np.uint8)
    for r, c in ag.OccupancyGrid.MANUAL_CELLS:
        occ[r, c] = 1
    for t in range(T):
        a = (rng.random((n, 2)) - 0.5) * 0.3
        o, r_dev, term, trunc, info = env.step(torch_.as_tensor(a, device="cuda"))
        res = oracle.step_batch(j1, j2, a, rw, fl, sq, ci)
        assert np.array_equal(info["final_obs"][:, 0].cpu().numpy(), j1) and np.array_equal(info["final_obs"][:, 1].cpu().numpy(), j2)
        assert np.array_equal(r_dev.cpu().numpy(), rw.astype(np.float32))
        assert np.array_equal(term.cpu().numpy(), fl != 0) and np.array_equal(info["collision"].cpu().numpy(), (fl & 1) != 0)
        assert rel_close(info["final_obs"][:, 2:4].cpu().numpy(), res["ee"]) and rel_close(info["final_obs"][:, 4:6].cpu().numpy(), res["dist"])
        for e in np.flatnonzero(fl != 0):                     # Scene.reset(): resample only while colliding
            episodes += 1
            if fl[e] & 1:
                for _ in range(64):
                    u0, u1 = oracle.philox_uniform2(seed, int(e), int(rc[e]), 1)
                    rc[e] += 1
                    j1[e], j2[e] = (u0 * np.pi) * 2.0, (u1 * np.pi) * 2.0
                    h = oracle.collision_batch(j1[e:e + 1].copy(), j2[e:e + 1].copy(), sq, want_first_hit=False)
                    h = h[0] if isinstance(h, tuple) else h
                    if not h[0]:
                        break
            rw[e], fl[e] = 0.0, 0
        assert np.array_equal(o[:, 0].cpu().numpy(), j1) and np.array_equal(o[:, 1].cpu().numpy(), j2)
        # the crop: 3x3 cells around the end effector's cell of the observation the env continues from
        gx, gy = o[:, 2].cpu().numpy(), o[:, 3].cpu().numpy()
        col = np.floor((gx + 0.8) / 0.2).astype(int); row = (np.floor((0.8 - gy) / 0.2) + 1).astype(int)
        crop = info["crop"].cpu().numpy()
        for e in range(0, n, 97):
            for dr in range(3):
                for dc in range(3):
                    r_, c_ = row[e] - 1 + dr, col[e] - 1 + dc
                    want = 2 if not (0 <= r_ < 9 and 0 <= c_ < 9) else int(occ[r_, c_])
                    assert crop[e, dr, dc] == want
    st = env.stats()
    assert episodes > 200 and st["episodes"] == episodes and st["env_steps"] == n * T
    assert np.array_equal(env.scene.reset_ctr.cpu().numpy().view(np.uint32).astype(np.int64), rc)


@pytest.mark.gpu
def test_rollout_host_compact_records(ag, torch_):
    """rollout_host without the reward plane: same j1 / j2 / flags, and reward_from_flags reproduces the plane"""
    n, K = 4096, 16
    rng = np.random.default_rng(51)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = torch_.as_tensor(((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)).pin_memory()
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    a, b = make_scene(ag, torch_, g, j1, j2, seed=4), make_scene(ag, torch_, g, j1, j2, seed=4)
    full, compact = a.alloc_records(K, pinned_host=True), b.alloc_records(K, pinned_host=True, reward=False)
    assert "reward" not in compact
    a.rollout_host(K, acts, full, chunk_envs=1024); b.rollout_host(K, acts, compact, chunk_envs=1024)
    for k in ("j1", "j2", "flags"):
        assert torch_.equal(full[k], compact[k])
    assert torch_.equal(b.reward_from_flags(compact["flags"]), full["reward"]) and int((full["flags"] != 0).sum()) > 5
    from abstract_gym_b200.experiment.experiment_0 import Trajectories
    assert np.array_equal(Trajectories.from_rollout(compact, acts).reward, full["reward"].numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_steps", [1, 5, 64])
def test_rollout_host_step_sliced_pipeline(ag, torch_, chunk_steps):
    """the step-sliced host pipeline (contiguous copies, dependent kernels) == one device rollout, records and state;
    also with in-kernel Philox actions / statistics only"""
    n, K = 5000, 12
    rng = np.random.default_rng(10)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    a = make_scene(ag, torch_, g, j1, j2, seed=4)
    b = make_scene(ag, torch_, g, j1, j2, seed=4)
    ra = a.rollout(K, actions=torch_.as_tensor(acts, device="cuda"))
    hact = torch_.as_tensor(acts).pin_memory()
    out = b.alloc_records(K, pinned_host=True)
    st = b.rollout_host(K, hact, out, chunk_steps=chunk_steps)
    for k in ("j1", "j2", "reward", "flags"):
        assert np.array_equal(ra[k].cpu().numpy(), out[k].numpy()), k
    assert np.array_equal(a.robot.joint_1.cpu().numpy(), b.robot.joint_1.cpu().numpy())
    assert torch_.equal(a.step_ctr, b.step_ctr) and torch_.equal(a.ep_len, b.ep_len)
    assert a.stats_dict() == b.stats_dict() == st
    a.rollout(K, record=False); b.rollout_host(K, None, None, chunk_steps=chunk_steps)
    assert a.stats_dict() == b.stats_dict()
    assert np.array_equal(a.robot.joint_2.cpu().numpy(), b.robot.joint_2.cpu().numpy())


def _compare_rollout(ag, torch, oracle, sc, st, K, actions, params, grids_sq):
    rec, stats0 = oracle.rollout(st, K, grids_sq, seed=sc.seed, actions_f32=actions, params=params)
    drec = sc.rollout(K, actions=torch.as_tensor(actions, device="cuda"))
    torch.cuda.synchronize()
    for k in ("flags", "reward", "j1", "j2"):
        assert np.array_equal(drec[k].cpu().numpy(), rec[k]), k
    assert np.array_equal(sc.robot.joint_1.cpu().numpy(), st.j1) and np.array_equal(sc.flags.cpu().numpy(), st.flags)
    assert np.array_equal(sc.ep_len.cpu().numpy().view(np.uint32), st.ep_len)
    assert np.array_equal(sc.reset_ctr.cpu().numpy().view(np.uint32), st.reset_ctr)
    return rec, stats0


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_rollout_joint_target_mode(ag, torch_, oracle, engine):
    """choose_j_tar (scene_0.py:123-127): done when both joints are within 2e-3 of target_j; envs start around it"""
    n, K = 4096, 32
    rng = np.random.default_rng(61)
    tj = np.array([2.3, 4.1])
    j1, j2 = tj[0] + rng.normal(0, 0.02, n), tj[1] + rng.normal(0, 0.02, n)
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.02).astype(np.float32)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sc = make_scene(ag, torch_, g, j1, j2, engine=engine, seed=13)
    sc.choose_j_tar, sc.target_j = True, tj
    p = oracle.default_params()
    p.choose_j_tar, p.target_j1, p.target_j2 = 1, tj[0], tj[1]
    st = oracle.RolloutState(j1, j2)
    rec, _ = _compare_rollout(ag, torch_, oracle, sc, st, K, acts, p, [oracle.manual_grid()[0]])
    assert int(((rec["flags"] & 2) != 0).sum()) > 50                  # the target is actually reached
    assert sc.stats_dict()["successes"] == int(((rec["flags"] & 2) != 0).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_rollout_entered_with_sticky_state_and_huge_angles(ag, torch_, oracle, engine):
    """a rollout entered with sticky reward / flags left by earlier step() calls (scene_0.py:95-100 never clears
    them) records them on its first step and resets; joints beyond the float32 filter's range (|j| >= 2^20 rad) go
    through the float64 path"""
    n, K = 4096, 24
    rng = np.random.default_rng(62)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    j1[::5] += 2 * np.pi * np.round(rng.uniform(2e5, 3e6, len(j1[::5])))   # same poses, many turns away
    pre = (rng.random((3, n, 2)) - 0.5) * 0.6                               # big pre-steps: many collisions, no reset
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sq, ci = oracle.manual_grid()
    sc = make_scene(ag, torch_, g, j1, j2, engine=engine, seed=14)
    st = oracle.RolloutState(j1, j2)
    rw = np.zeros(n); fl = np.zeros(n, dtype=np.uint8)
    for t in range(3):
        sc.step(torch_.as_tensor(pre[t], device="cuda"))
        oracle.step_batch(st.j1, st.j2, pre[t], rw, fl, sq, ci)
    assert np.array_equal(sc.flags.cpu().numpy(), fl) and 200 < int((fl != 0).sum()) < n
    st.reward[:] = rw.astype(np.float32); st.flags[:] = fl
    rec, _ = _compare_rollout(ag, torch_, oracle, sc, st, K, acts, oracle.default_params(), [sq])
    assert np.array_equal(rec["flags"][0] != 0, (fl != 0) | (rec["flags"][0] != 0))   # sticky flags show on step 0


@pytest.mark.gpu
def test_rollout_full_size_config3_vs_oracle(ag, torch_, oracle):
    """BASELINE config 3 at its full size -- 2^20 envs x 64 fused steps, scene_0 map, FAST engine, trajectory
    records -- against the CPU oracle on the same scripted actions: every flag, reward and recorded joint of the
    6.7e7 env-steps bit-exact, final state and episode counters equal (the oracle needs a few seconds on the host)."""
    n, K = 1 << 20, 64
    rng = np.random.default_rng(2026)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = ((rng.random((K, n, 2), dtype=np.float32) - np.float32(0.5)) * np.float32(0.1))
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sc = make_scene(ag, torch_, g, j1, j2, engine="fast", seed=77)
    st = oracle.RolloutState(j1, j2)
    rec, stats = oracle.rollout(st, K, [oracle.manual_grid()[0]], seed=77, actions_f32=acts)
    drec = sc.rollout(K, actions=torch_.as_tensor(acts, device="cuda"))
    torch_.cuda.synchronize()
    for k in ("flags", "reward", "j1", "j2"):
        assert np.array_equal(drec[k].cpu().numpy(), rec[k]), k
    assert np.array_equal(sc.robot.joint_1.cpu().numpy(), st.j1) and np.array_equal(sc.robot.joint_2.cpu().numpy(), st.j2)
    assert np.array_equal(sc.reset_ctr.cpu().numpy().view(np.uint32), st.reset_ctr)
    assert np.array_equal(sc.stats.cpu().numpy(), stats)
    assert stats[oracle.ST_ENV_STEPS] == n * K and stats[oracle.ST_EPISODES] > 50000 and stats[oracle.ST_SUCCESSES] > 100


@pytest.mark.gpu
def test_integration_md_ctypes_stub_runs(ag, torch_):
    """the reference-side ctypes stub printed in INTEGRATION.md is executable as written (struct layouts match the
    header) and steps a batch exactly like BatchedScene.step"""
    import re
    from abstract_gym_b200 import _lib
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "INTEGRATION.md")).read()
    m = re.search(r"```python\n(# abstract_gym/scenario/scene_0_b200\.py.*?)```", text, re.S)
    assert m, "stub not found in INTEGRATION.md"
    code = m.group(1).replace('C.CDLL("libabstract_gym_b200.so")', "C.CDLL(%r)" % _lib.lib_path())
    ns = {}
    exec(compile(code, "INTEGRATION.md", "exec"), ns)
    env = ag.OccupancyGrid(size=9, random_obstacle=False)         # has .occ and .environment_size like the reference's
    grid, keep = ns["pack_grid"](env)
    n = 2048
    rng = np.random.default_rng(71)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = (rng.random((n, 2)) - 0.5) * 0.6
    ref = make_scene(ag, torch_, env, j1, j2, engine="fast")
    ref.step(torch_.as_tensor(acts, device="cuda"))

    class _S:                                                     # what the stub reads from a reference Scene
        robot = ag.TwoJointRobot(0.0, 0.0)
        target_c = ag.Point(-0.2, -0.3)
    t = lambda a, dt: torch_.as_tensor(a, device="cuda").to(dt).contiguous()
    d1, d2 = t(j1, torch_.float64), t(j2, torch_.float64)
    rw, fl = torch_.zeros(n, dtype=torch_.float32, device="cuda"), torch_.zeros(n, dtype=torch_.uint8, device="cuda")
    ns["step_batch"](_S, grid, d1, d2, t(acts, torch_.float64), rw, fl)
    torch_.cuda.synchronize()
    assert torch_.equal(d1, ref.robot.joint_1) and torch_.equal(fl, ref.flags) and torch_.equal(rw, ref.step_reward)
    assert int((fl != 0).sum()) > 100


@pytest.mark.gpu
def test_per_env_targets(ag, torch_):
    """per-env cartesian targets (gym-style callers): done fires exactly for the envs whose own target is reached,
    goal distance is measured to the own target; VectorEnv carries them through its (captured) step"""
    n = 2048
    rng = np.random.default_rng(81)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = (rng.random((n, 2)) - 0.5) * 0.1
    ee_next = ag.forward_kinematics(torch_.as_tensor(j1 + acts[:, 0], device="cuda"),
                                    torch_.as_tensor(j2 + acts[:, 1], device="cuda"))[:, 2:4]
    targets = ee_next.clone()
    far = torch_.arange(n, device="cuda") % 2 == 1
    targets[far] += 0.05                                              # odd envs: target 5 cm away in x and y
    sc = make_scene(ag, torch_, g, j1, j2)
    _, _, rw, done, coll, extra = sc.step(torch_.as_tensor(acts, device="cuda"), want_ee=True, targets=targets)
    assert torch_.equal(done, ~far)
    assert bool((rw[~far] == 1e4).all()) and bool((rw[far & ~coll] == 0).all())
    assert float(extra["dist"][~far].max()) < 1e-12 and float((extra["dist"][far] - 0.05).abs().max()) < 1e-12
    # VectorEnv: same targets, eager and captured
    for graph in (False, True):
        env = ag.VectorEnv(n, device="cuda", seed=3, targets=torch_.zeros(n, 2, dtype=torch_.float64, device="cuda"))
        obs = env.reset().clone()
        a = (torch_.rand(n, 2, dtype=torch_.float64, device="cuda") - 0.5) * 0.1
        nxt = ag.forward_kinematics((obs[:, 0] + a[:, 0]).contiguous(), (obs[:, 1] + a[:, 1]).contiguous())[:, 2:4]
        tg = nxt.clone(); tg[far] += 0.05
        if graph:
            env.capture()
        env.set_targets(tg)
        _, r, term, _, info = env.step(a)
        assert torch_.equal(term & ~info["collision"], ~far & ~info["collision"]) and bool(term[~far].all())


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_steps,chunk_envs", [(0, 512), (3, 1 << 17)])
def test_rollout_host_heterogeneous_grids(ag, torch_, chunk_steps, chunk_envs):
    """host-buffer pipeline on per-batch 64x64 maps (the lane-asynchronous kernel, staged grids): both slicing modes
    equal one device rollout"""
    n, K = 2048, 10
    rng = np.random.default_rng(91)
    occs = np.stack([random_grid(rng, 64, 0.01) for _ in range(8)])
    g = ag.BatchedOccupancyGrid(torch_.as_tensor(occs, device="cuda"), 256)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    a, b = make_scene(ag, torch_, g, j1, j2, seed=5), make_scene(ag, torch_, g, j1, j2, seed=5)
    ra = a.rollout(K, actions=torch_.as_tensor(acts, device="cuda"))
    out = b.alloc_records(K, pinned_host=True)
    b.rollout_host(K, torch_.as_tensor(acts).pin_memory(), out, chunk_envs=chunk_envs, chunk_steps=chunk_steps)
    for k in ("j1", "j2", "reward", "flags"):
        assert np.array_equal(ra[k].cpu().numpy(), out[k].numpy()), k
    assert a.stats_dict() == b.stats_dict() and a.stats_dict()["episodes"] > 100
    assert torch_.equal(a.robot.joint_1, b.robot.joint_1) and torch_.equal(a.reset_ctr, b.reset_ctr)


@pytest.mark.gpu
def test_clustered_grid_generator(ag, torch_, oracle):
    """clustered-obstacle maps: a usable fraction of poses stays free, and rollouts on them equal the oracle"""
    gen = torch_.Generator(device="cuda").manual_seed(7)
    bg = ag.BatchedOccupancyGrid.clustered(4, 128, n_blobs=10, blob_radius_cells=4, envs_per_grid=256, generator=gen)
    occ = bg.device_grid().unpack()
    assert occ.shape == (4, 128, 128) and 0.005 < occ.mean() < 0.2
    n, K = 1024, 12
    rng = np.random.default_rng(92)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    sc = make_scene(ag, torch_, bg, j1, j2, seed=9)
    free = 1.0 - float(sc.collision_check().float().mean().item())
    assert free > 0.15, free
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    st = oracle.RolloutState(j1, j2)
    rec, stats = oracle.rollout(st, K, [oracle.grid_squares(o)[0] for o in occ], envs_per_grid=256, seed=9, actions_f32=acts)
    drec = sc.rollout(K, actions=torch_.as_tensor(acts, device="cuda"))
    assert np.array_equal(drec["flags"].cpu().numpy(), rec["flags"]) and np.array_equal(sc.stats.cpu().numpy(), stats)


@pytest.mark.gpu
def test_rollout_random_grids_sweep(ag, torch_, oracle):
    """24 random maps of every class (obstacle-list, traversal, staged with transposed bits, per-batch) x scripted /
    Philox draws: FAST rollouts equal the oracle record for record"""
    rng = np.random.default_rng(2027)
    cases = 0
    for i in range(24):
        S = int(rng.choice([5, 7, 9, 12, 17, 31, 33, 48, 64, 100, 128]))
        p = float(rng.choice([0.01, 0.03, 0.08])) if S <= 31 else float(rng.choice([0.004, 0.01]))
        n = int(rng.choice([96, 256, 1000, 2048]))
        K = int(rng.integers(2, 20))
        if i % 3 == 2 and S > 9:
            occs = [random_grid(rng, S, p) for _ in range(max(1, n // 256))]
            _rollout_case(ag, torch_, oracle, occs, (n // 256) * 256 or 256, K, "fast", bool(i % 2), envs_per_grid=256, seed=100 + i)
        else:
            _rollout_case(ag, torch_, oracle, [random_grid(rng, S, p)], n, K, "fast", bool(i % 2), seed=100 + i)
        cases += 1
    assert cases == 24


# ------------------------------------------------------------------ round 2: config-size parity, sinks, filters

def _sampled_fullsize(ag, torch, oracle, scene, grid_squares_of_chunk, n, K, chunk, n_chunks, seed, epg=None):
    """Launch the whole batch (in-kernel Philox actions and resets), then re-run `n_chunks` random contiguous chunks of
    `chunk` global env ids on the oracle: Philox is keyed by the global id, so every recorded flag / reward / joint of
    the sampled envs, their final state and counters must match bit for bit."""
    j1_0, j2_0 = scene.robot.joint_1.cpu().numpy().copy(), scene.robot.joint_2.cpu().numpy().copy()
    rc0 = scene.reset_ctr.cpu().numpy().view(np.uint32).copy()
    rec = scene.rollout(K, actions=None, record=True)
    torch.cuda.synchronize()
    rng = np.random.default_rng(seed)
    starts = rng.choice(n // chunk, size=n_chunks, replace=False) * chunk
    fl, rw = rec["flags"].cpu().numpy(), rec["reward"].cpu().numpy()
    r1, r2 = rec["j1"].cpu().numpy(), rec["j2"].cpu().numpy()
    fin1, fin2 = scene.robot.joint_1.cpu().numpy(), scene.robot.joint_2.cpu().numpy()
    rcn = scene.reset_ctr.cpu().numpy().view(np.uint32)
    eln = scene.ep_len.cpu().numpy().view(np.uint32)
    episodes = 0
    for s0 in starts:
        sl = slice(int(s0), int(s0) + chunk)
        st = oracle.RolloutState(j1_0[sl], j2_0[sl])
        st.reset_ctr[:] = rc0[sl]
        orec, ostats = oracle.rollout(st, K, [grid_squares_of_chunk(int(s0))], envs_per_grid=None, env_id0=scene.env_id0 + int(s0),
                                      seed=scene.seed)
        assert np.array_equal(fl[:, sl], orec["flags"]), "flags differ in chunk %d" % s0
        assert np.array_equal(rw[:, sl], orec["reward"])
        assert np.array_equal(r1[:, sl], orec["j1"]) and np.array_equal(r2[:, sl], orec["j2"])
        assert np.array_equal(fin1[sl], st.j1) and np.array_equal(fin2[sl], st.j2)
        assert np.array_equal(rcn[sl], st.reset_ctr) and np.array_equal(eln[sl], st.ep_len)
        episodes += int(ostats[oracle.ST_EPISODES])
    return episodes


@pytest.mark.gpu
def test_fullsize_config4_sampled_vs_oracle(ag, torch_, oracle):
    """BASELINE config 4 at its full size (2^20 envs x 64 steps on the bench's 1024x1024 Bernoulli(0.002) map, FAST
    engine, lane-asynchronous kernel): 16 x 256 = 4096 sampled global env ids against the oracle, all 64 steps."""
    n, K = 1 << 20, 64
    occ = (np.random.default_rng(4).random((1024, 1024)) < 0.002).astype(np.uint8)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    g.load_from_matrix(occ)
    gen = torch_.Generator(device="cuda").manual_seed(1234)
    sc = ag.BatchedScene(ag.BatchedTwoJointRobot.random(n, device="cuda", generator=gen), g, engine="fast", seed=0)
    sc.random_valid_pose()
    sq = oracle.grid_squares(occ)[0]
    episodes = _sampled_fullsize(ag, torch_, oracle, sc, lambda s0: sq, n, K, 256, 16, seed=44)
    assert episodes > 50000                                  # ~57 % of the env-steps end an episode on this map
    assert sc.stats_dict()["env_steps"] == n * K


@pytest.mark.gpu
def test_fullsize_config5_sampled_vs_oracle(ag, torch_, oracle):
    """BASELINE config 5 at its full size: 4096 distinct 256x256 Bernoulli(0.008) maps (bench generator), 2^20 envs x
    64 steps, auto-reset; 16 sampled batches of 256 envs (each on its own map) against the oracle."""
    n, K = 1 << 20, 64
    ggen = torch_.Generator(device="cuda").manual_seed(5)
    grid = ag.BatchedOccupancyGrid.random(n // 256, 256, 0.008, 256, device="cuda", generator=ggen, clear_base_cells=2)
    gen = torch_.Generator(device="cuda").manual_seed(1234)
    sc = ag.BatchedScene(ag.BatchedTwoJointRobot.random(n, device="cuda", generator=gen), grid, engine="fast", seed=0)
    sc.random_valid_pose()
    dg = grid.device_grid()

    def squares(s0):
        occ = dg.unpack([s0 // 256])[0]
        assert occ[126:131, 125:130].sum() == 0              # the cells around the base are free
        return oracle.grid_squares(occ)[0]

    episodes = _sampled_fullsize(ag, torch_, oracle, sc, squares, n, K, 256, 16, seed=55)
    assert episodes > 20000 and sc.stats_dict()["stuck_resets"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("grid_kind", ["scene0", "rand64"])
def test_event_sink_equals_dense_records(ag, torch_, grid_kind):
    """joints-only records + the event list (ag_rollout_args.events) carry exactly what the four dense planes carry"""
    n, K = 8192, 48
    rng = np.random.default_rng(71)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    if grid_kind == "rand64":
        g.load_from_matrix(random_grid(rng, 64, 0.01))
    a = make_scene(ag, torch_, g, j1, j2, engine="fast", seed=5)
    b = make_scene(ag, torch_, g, j1, j2, engine="fast", seed=5)
    dense = a.rollout(K)
    sink = b.alloc_event_sink(K)
    b.rollout(K, out=dict(j1=sink["j1"], j2=sink["j2"]), events=sink)
    torch_.cuda.synchronize()
    cnt = int(sink["count_buf"][0].item())
    assert 0 < cnt <= sink["events"].shape[0]
    reward, flags = b.events_to_planes(sink, K, count=cnt)
    assert np.array_equal(flags, dense["flags"].cpu().numpy()) and np.array_equal(reward, dense["reward"].cpu().numpy())
    assert np.array_equal(sink["j1"].cpu().numpy(), dense["j1"].cpu().numpy())
    assert cnt == int((dense["flags"].cpu().numpy() != 0).sum())
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy())


@pytest.mark.gpu
def test_rollout_events_host_and_philox_actions(ag, torch_):
    """the zero-H2D host path: in-kernel actions, joints + events to pinned host memory, equal to the device rollout;
    philox_actions() reproduces on the host the actions an env drew in the kernel"""
    n, K = 1 << 14, 32
    rng = np.random.default_rng(72)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    a = make_scene(ag, torch_, g, j1, j2, engine="fast", seed=9)
    b = make_scene(ag, torch_, g, j1, j2, engine="fast", seed=9)
    a.random_valid_pose(); b.random_valid_pose()
    start1, start2 = a.robot.joint_1.cpu().numpy().copy(), a.robot.joint_2.cpu().numpy().copy()
    for call in range(2):                                     # two calls: the draw counters carry over
        dense = a.rollout(K)
        sink = b.alloc_event_sink(K, pinned_host=True)
        st = b.rollout_events_host(K, sink, chunk_steps=5)
        torch_.cuda.synchronize()
        reward, flags = b.events_to_planes(sink, K)
        assert np.array_equal(flags, dense["flags"].cpu().numpy()) and np.array_equal(reward, dense["reward"].cpu().numpy())
        assert np.array_equal(sink["j1"].numpy(), dense["j1"].cpu().numpy()) and np.array_equal(sink["j2"].numpy(), dense["j2"].cpu().numpy())
        assert st["env_steps"] == n * K
        if call == 0:
            quiet = np.flatnonzero((flags != 0).sum(axis=0) == 0)[:512]     # envs without an episode end
            acts = b.philox_actions(quiet, np.zeros(len(quiet), dtype=np.uint64), K)   # [K, m, 2] float64
            q1, q2 = start1[quiet].copy(), start2[quiet].copy()
            for t in range(K):
                q1 = q1 + acts[t, :, 0]; q2 = q2 + acts[t, :, 1]
                assert np.array_equal(q1.astype(np.float32), sink["j1"].numpy()[t, quiet])
                assert np.array_equal(q2.astype(np.float32), sink["j2"].numpy()[t, quiet])
    assert np.array_equal(a.robot.joint_1.cpu().numpy(), b.robot.joint_1.cpu().numpy())
    assert np.array_equal(a.stats.cpu().numpy(), b.stats.cpu().numpy())


@pytest.mark.gpu
def test_fast_filter_band_1e3_to_2p20_rad(ag, torch_, oracle):
    """FAST == EXACT == oracle for joint angles between 1e3 and 2^20 rad, the range where the float32 filter trusts its
    float64 range reduction most (beyond 2^20 it hands over to float64): same poses, many whole turns away."""
    n = 1 << 18
    rng = np.random.default_rng(81)
    base1, base2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    turns = np.round(10.0 ** rng.uniform(np.log10(1.6e2), np.log10(1.66e5), n)) * rng.choice([-1.0, 1.0], n)   # 1e3 .. 1.04e6 rad
    j1, j2 = base1 + 2 * np.pi * turns, base2 + 2 * np.pi * np.roll(turns, 1)
    assert np.abs(j1).max() < 2 ** 20 and np.abs(j1).min() > 9e2
    g = ag.OccupancyGrid(size=9, random_obstacle=False)
    sq, ci = oracle.manual_grid()
    ref = oracle.collision_batch(j1, j2, sq, want_first_hit=False)
    ref = ref[0] if isinstance(ref, tuple) else ref
    for engine in ("fast", "exact"):
        sc = make_scene(ag, torch_, g, j1, j2, engine=engine)
        hit = sc.collision_check().cpu().numpy()
        bad = np.flatnonzero(hit != (ref != 0))
        assert len(bad) == 0, "%s: %d flags differ" % (engine, len(bad))
    # and through the fused rollout (table arm of k_rollout_lut): a short rollout from these poses
    K = 8
    acts = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
    sc = make_scene(ag, torch_, g, j1, j2, engine="fast", seed=4)
    sc.random_valid_pose()
    st = oracle.RolloutState(sc.robot.joint_1.cpu().numpy(), sc.robot.joint_2.cpu().numpy())
    st.reset_ctr[:] = sc.reset_ctr.cpu().numpy().view(np.uint32)
    _compare_rollout(ag, torch_, oracle, sc, st, K, acts, oracle.default_params(), [sq])


@pytest.mark.gpu
@pytest.mark.parametrize("S,p", [(320, 0.004), (440, 0.003)])
def test_exact_rollout_with_large_staged_grids(ag, torch_, oracle, S, p):
    """EXACT / BRUTE rollouts on grids whose staging footprint plus the kernel's static shared memory exceeds 48 KB
    (S = 320 with the transposed copy: 30.7 KB dynamic + 22.6 KB static): needs the dynamic shared-memory opt-in."""
    rng = np.random.default_rng(S)
    occ = random_grid(rng, S, p)
    occ[S // 2 - 3:S // 2 + 4, S // 2 - 3:S // 2 + 4] = 0
    for engine in ("exact", "fast"):
        _rollout_case(ag, torch_, oracle, [occ], 768, 6, engine, True, seed=8)


@pytest.mark.gpu
def test_nearly_axis_aligned_links_exact_brute_oracle(ag, torch_, oracle):
    """Links within 1e-16 .. 1e-7 rad of an axis: the reference's lambda arithmetic (collision_checker.py:79-91) divides
    by dx ~ 1e-13 there and may accept a square on the link's infinite line far beyond its end.  EXACT switches to the
    reference's loop over every occupied cell for such links, so EXACT == BRUTE == oracle also here."""
    rng = np.random.default_rng(91)
    n = 1 << 16
    occ = np.zeros((31, 31), dtype=np.uint8)
    occ[2:6, 14:17] = 1; occ[25:29, 14:17] = 1; occ[14:17, 2:6] = 1; occ[14:17, 25:29] = 1     # squares on both axes, far from the arm
    occ[rng.integers(0, 31, 40), rng.integers(0, 31, 40)] = 1
    occ[13:18, 13:18] = 0
    axis = rng.integers(0, 4, n) * (np.pi / 2)
    delta = 10.0 ** rng.uniform(-16, -7, n) * rng.choice([-1.0, 1.0], n)
    j1 = axis + delta
    j2 = np.where(rng.random(n) < 0.5, rng.integers(0, 4, n) * (np.pi / 2) + np.roll(delta, 1), rng.uniform(0, 2 * np.pi, n))
    sq = oracle.grid_squares(occ)[0]
    ref = oracle.collision_batch(j1, j2, sq, want_first_hit=False)
    ref = (ref[0] if isinstance(ref, tuple) else ref) != 0
    hits = {}
    for engine in ("exact", "brute", "fast"):
        sc = make_scene(ag, torch_, occ, j1, j2, engine=engine)
        hits[engine] = sc.collision_check().cpu().numpy()
    assert np.array_equal(hits["exact"], hits["brute"])
    bad = np.flatnonzero(hits["exact"] != ref)
    # CUDA sincos vs glibc in the last ulp moves dx by ~1e-17: only poses whose flag flips under that are excused
    assert len(bad) <= n // 200, "%d mismatches vs the oracle" % len(bad)
    print("near-axis links: exact==brute on %d poses; %d differ from the CPU oracle (sincos ulp), fast differs from exact on %d"
          % (n, len(bad), int((hits["fast"] != hits["exact"]).sum())))


_DEBUG_CHILD = r'''
import numpy as np, torch, sys
sys.path.insert(0, %r)
import abstract_gym_b200 as ag
from abstract_gym_b200 import _lib
from oracle import oracle as orc
assert _lib.lib_path().endswith("_debug.so"), _lib.lib_path()
rng = np.random.default_rng(11)
n, K = 2048, 10
cases = [("scene0", None, 9),
         ("rand64", [(rng.random((64, 64)) < 0.02).astype(np.uint8)], 64),
         ("rand300", [(rng.random((300, 300)) < 0.004).astype(np.uint8) for _ in range(2)], 300)]
for name, occs, S in cases:
    for engine in ("fast", "exact", "brute"):
        if engine == "brute" and S > 64:
            continue
        j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
        if occs is None:
            grid, squares, epg = ag.OccupancyGrid(size=9, random_obstacle=False), [orc.manual_grid()[0]], None
        else:
            epg = n // len(occs)
            grid = ag.BatchedOccupancyGrid(torch.as_tensor(np.stack(occs), device="cuda"), epg)
            squares = [orc.grid_squares(o)[0] for o in occs]
        robot = ag.BatchedTwoJointRobot(torch.as_tensor(j1, device="cuda"), torch.as_tensor(j2, device="cuda"))
        sc = ag.BatchedScene(robot, grid, engine=engine, seed=4)
        rec = sc.rollout(K)
        torch.cuda.synchronize()
        st = orc.RolloutState(j1, j2)
        kw = {} if epg is None else dict(envs_per_grid=epg)
        orec, ostats = orc.rollout(st, K, squares, seed=4, **kw)
        assert np.array_equal(rec["flags"].cpu().numpy(), orec["flags"]), (name, engine)
        assert np.array_equal(sc.stats.cpu().numpy(), ostats), (name, engine)
        assert np.array_equal(sc.robot.joint_1.cpu().numpy(), st.j1), (name, engine)
print("debug parity ok")
'''


def _traps_per_kernel(path):
    """{mangled kernel name: number of trap instructions} from the SASS of a library"""
    import re
    import subprocess
    from abstract_gym_b200 import build as ag_build
    cuobjdump = os.path.join(os.path.dirname(ag_build.find_nvcc()), "cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", path], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                          check=True).stdout
    traps, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            traps[name] = 0
        elif name is not None and "BPT.TRAP" in line:
            traps[name] += 1
    return traps


@pytest.mark.gpu
def test_debug_bounds_build_per_family(ag, torch_):
    """the -DAG_DEBUG_BOUNDS library (csrc/ag_device.cuh AG_CHECK_INDEX): same results as the oracle on list, traversal
    and brute paths with every index assertion compiled in.  That the assertions are there is read from the machine
    code instead of tripping one: a trap is a device fault that ends the CUDA context, and a test does not set one off
    on purpose.  Every rollout, step, reset and collision kernel of the debug library traps on a bad index (the brute
    collision kernel on the padding bit of a malformed grid); the release library has no trap at all.  The instantiations
    of each of those kernel families are counted exactly: the launchers build only the forms their dispatch can reach."""
    import subprocess
    import sys
    from abstract_gym_b200 import build as ag_build
    lib = ag_build.build_debug()
    code = _DEBUG_CHILD % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, AG_LIB_PATH=lib)
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=600)
    assert r.returncode == 0 and "debug parity ok" in r.stdout, r.stdout[-3000:]
    debug, release = _traps_per_kernel(lib), _traps_per_kernel(ag_build.LIB)
    assert sum(release.values()) == 0 and len(release) == len(debug) > 100
    # instantiations per family; a mangled name holds the length-prefixed identifier, then I for the template arguments
    families = {"k_rollout": 40, "k_rollout_async": 8, "k_rollout_lut": 12, "k_step": 10, "k_step_obs": 0, "k_reset": 6,
                "k_collision": 5}
    per_family = {f: [k for k in debug if "%d%sI" % (len(f), f) in k] for f in families}
    assert {f: len(ks) for f, ks in per_family.items()} == families
    checked = sum(per_family.values(), [])
    assert all(debug[k] > 0 for k in checked), [k for k in checked if debug[k] == 0]
    assert any("k_collisionILi2E" in k and debug[k] > 0 for k in debug)       # ENGINE_BRUTE


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["scene0", "scene0_long_links", "random_small"])
def test_cspace_map_clear_bins_are_uneventful(ag, torch_, case):
    """the configuration-space map of the headline rollout kernel (include/abstract_gym_b200.h ag_cspace_map): a CLEAR
    bit promises collision_check() == False and check_target_reached() == False for every pose of the bin.  Checked
    against the BRUTE engine (the reference's loop over all obstacles, float64) on 4M poses per case: uniform ones,
    poses around scene_0's tangent configurations (link 1 along an axis) and poses on bin edges."""
    import ctypes as C
    import math
    from abstract_gym_b200 import _lib
    from abstract_gym_b200._device import ptr, stream_ptr
    torch = torch_
    lib = _lib.load()
    b1, b2 = C.c_int32(), C.c_int32()
    words = lib.ag_cspace_map_words(C.byref(b1), C.byref(b2))
    b1, b2 = b1.value, b2.value
    assert words * 32 == 1 << (b1 + b2)
    rng = np.random.default_rng(21)
    link = (0.4, 0.3)
    if case == "scene0":
        grid, target = ag.OccupancyGrid(size=9, random_obstacle=False), None
    elif case == "scene0_long_links":
        grid, target, link = ag.OccupancyGrid(size=9, random_obstacle=False), (0.35, 0.55), (0.45, 0.4)
    else:
        occ = np.zeros((17, 17), np.uint8)
        occ[rng.integers(0, 17, 7), rng.integers(0, 17, 7)] = 1
        occ[8, 8] = occ[9, 8] = 0
        grid, target = ag.OccupancyGrid(size=17, random_obstacle=False), (-0.31, 0.22)
        grid.load_from_matrix(occ)
    n = 1 << 22
    q1, q2 = rng.uniform(-20.0, 20.0, n), rng.uniform(-20.0, 20.0, n)
    k = n // 4                                                    # tangent poses of link 1: k*pi/2 +- 10^-9 .. 10^-1
    q1[:k] = rng.integers(-8, 8, k) * (math.pi / 2) + rng.choice([-1.0, 1.0], k) * 10.0 ** rng.uniform(-9, -1, k)
    e = n // 8                                                    # poses on bin edges (both joints), +- a few phase units
    q1[k:k + e] = rng.integers(0, 1 << b1, e) * (2 * math.pi / (1 << b1)) + rng.uniform(-3e-9, 3e-9, e)
    q2[k:k + e] = rng.integers(0, 1 << b2, e) * (2 * math.pi / (1 << b2)) + rng.uniform(-3e-9, 3e-9, e)
    robot = ag.BatchedTwoJointRobot(torch.as_tensor(q1, device="cuda"), torch.as_tensor(q2, device="cuda"), link_1=link[0], link_2=link[1])
    kw = {} if target is None else dict(target_c=ag.Point(*target))
    sc = ag.BatchedScene(robot, grid, engine="brute", **kw)
    m = torch.zeros(words, dtype=torch.int32, device="cuda")
    _lib.check(lib.ag_cspace_map(sc.params(), sc.grid.c_struct(), ptr(m), stream_ptr(sc.device)), "ag_cspace_map")
    eventful = (sc.collision_check() | sc.check_target_reached()).cpu().numpy()
    mw = m.cpu().numpy().view(np.uint32)
    # the kernel's phase: low 32 bits of round(q * 2^32 / 2pi); numpy's product rounds twice (fma does not), which moves
    # a pose by at most one phase unit (1.5e-9 rad) -- far inside the map's 2e-6 m margin
    scale = 4294967296.0 / (2 * math.pi)
    x1 = np.rint(q1 * scale).astype(np.int64) & 0xFFFFFFFF
    x2 = np.rint(q2 * scale).astype(np.int64) & 0xFFFFFFFF
    bit = ((x1 >> (32 - b1)) << b2) | (x2 >> (32 - b2))
    is_set = ((mw[bit >> 5] >> (bit & 31).astype(np.uint32)) & 1).astype(bool)
    bad = eventful & ~is_set
    assert not bad.any(), "%d eventful poses in CLEAR bins, e.g. q = (%r, %r)" % (bad.sum(), q1[bad][0], q2[bad][0])
    uni = slice(k + e, n)
    frac = (is_set[uni] & ~eventful[uni]).sum() / max((~eventful[uni]).sum(), 1)
    print("cspace map %s: %d x %d bins, %.2f %% of them set; %.3f %% of the uneventful uniform poses sit in SET bins"
          % (case, 1 << b1, 1 << b2, 100 * is_set[uni].mean(), 100 * frac))
    assert frac < 0.03
    assert eventful.sum() > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["rows", "transposed", "hier"])
def test_grid_forms_rollout_vs_oracle(ag, torch_, oracle, form, monkeypatch):
    """the three traversal forms of the FAST engine for maps beyond the obstacle-list class -- row-major bits, rows +
    transposed copy (minor-axis walk), two-level tiles + summary bitmap (ag_grid.hier) -- each against the oracle:
    sizes that are and are not multiples of 8 / 32, one global map and staged per-batch maps, dense and sparse."""
    monkeypatch.setenv("AG_GRID_FORM", form)
    rng = np.random.default_rng(77)
    for S, p, n_maps, n, K in ((64, 0.02, 1, 2048, 10), (100, 0.01, 4, 2048, 10), (257, 0.004, 2, 1024, 8), (520, 0.002, 1, 1024, 6)):
        occs = [random_grid(rng, S, p) for _ in range(n_maps)]
        stats = _rollout_case(ag, torch_, oracle, occs, n, K, "fast", scripted=True, envs_per_grid=n // n_maps)
        assert stats[0] > 0
        g = ag.BatchedOccupancyGrid(torch_.as_tensor(np.stack(occs), device="cuda"), n // n_maps)
        dg = g.device_grid("cuda") if hasattr(g, "device_grid") else g._grid
        assert (dg.hier is not None) == (form == "hier") and (dg.bits_t is not None) == (form == "transposed")


@pytest.mark.gpu
def test_map_form_random_scenes_vs_oracle(ag, torch_, oracle):
    """the headline kernel's configuration-space map on random scene_0-class scenes: random small maps (1..8 occupied
    cells, 5..32 cells per side), random link lengths and targets -- every recorded flag, reward, joint, the
    final state and the episode counters against the oracle.  AG_SOAK=<n> runs n scenes instead of 6.
    One more scene has scene_0's obstacles and every other scripted reset candidate at u in [-1e6, -6e5]: such a pose
    (q = 2 pi u) is outside the range of the map's phase, so the map must not accept it as free."""
    rng = np.random.default_rng(2024)
    n_scenes = int(os.environ.get("AG_SOAK", "6"))
    n, K = 4096, 24
    for it in range(n_scenes + 1):
        S = int(rng.integers(5, 33))
        occ = np.zeros((S, S), np.uint8)
        m = int(rng.integers(1, 9))
        occ[rng.integers(0, S, m), rng.integers(0, S, m)] = 1
        l1, l2 = float(rng.uniform(0.15, 0.6)), float(rng.uniform(0.15, 0.6))
        ang = rng.uniform(0, 2 * np.pi)
        rad = rng.uniform(0.0, l1 + l2)
        target = (float(rad * np.cos(ang)), float(rad * np.sin(ang)))
        j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
        actions = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32)
        reset_u = rng.random((n, 40, 2))
        if it == n_scenes:
            S, m, l1, l2 = 9, 3, 0.4, 0.3
            occ = np.zeros((S, S), np.uint8)
            occ[[5, 5, 2], [6, 7, 3]] = 1
            reset_u[:, ::2] = rng.uniform(-1.0e6, -6.0e5, (n, 20, 2))
        grid = ag.OccupancyGrid(size=9, random_obstacle=False)
        grid.load_from_matrix(occ)
        robot = ag.BatchedTwoJointRobot(torch_.as_tensor(j1, device="cuda"), torch_.as_tensor(j2, device="cuda"), link_1=l1, link_2=l2)
        sc = ag.BatchedScene(robot, grid, target_c=ag.Point(*target), engine="fast", seed=5 + it)
        p = oracle.default_params()
        p.link_1, p.link_2, p.target_x, p.target_y = l1, l2, target[0], target[1]
        dp = sc.params()
        p.reach_eps = dp.reach_eps                       # whatever tolerance the scene actually uses
        rec = sc.rollout(K, actions=torch_.as_tensor(actions, device="cuda"), reset_u=torch_.as_tensor(reset_u, device="cuda"))
        torch_.cuda.synchronize()
        st = oracle.RolloutState(j1, j2)
        orec, ostats = oracle.rollout(st, K, [oracle.grid_squares(occ)[0]], seed=5 + it, actions_f32=actions, reset_u=reset_u, params=p)
        what = "scene %d: S=%d m=%d links=(%.3f, %.3f) target=(%.3f, %.3f)" % (it, S, m, l1, l2, target[0], target[1])
        assert np.array_equal(rec["flags"].cpu().numpy(), orec["flags"]), what
        assert np.array_equal(rec["reward"].cpu().numpy(), orec["reward"]), what
        assert np.array_equal(rec["j1"].cpu().numpy(), orec["j1"]) and np.array_equal(rec["j2"].cpu().numpy(), orec["j2"]), what
        assert np.array_equal(sc.robot.joint_1.cpu().numpy(), st.j1) and np.array_equal(sc.robot.joint_2.cpu().numpy(), st.j2), what
        assert np.array_equal(sc.stats.cpu().numpy(), ostats), what
