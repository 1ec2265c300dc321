"""K6 (`ag_step_obs`, csrc/ag_kernels.cu k_step_obs), the fused gym step behind VectorEnv and the torch op
`step_obs`, against the CPU oracle on every engine, action dtype, grid form and option.

Two references, both in oracle/:
  * float32 actions with auto-reset: `oracle.rollout(K=1)` per step, carrying its RolloutState -- K6's step, episode
    statistics and reset rule (Philox stream 1, keyed by the global env id and reset_ctr) exactly;
  * any float64 actions, and auto_reset off: `oracle.step_batch` per (grid, target block), then the reference's reset
    rule written out below with `oracle.philox_uniform2` and `oracle.collision_batch`.
Flags, rewards, joints, counters and crops must match bit for bit; observation geometry within 1e-5 relative and 1e-14
absolute (CUDA sincos vs glibc).  The crop reference reads the device's own end effector, so that a cell boundary never
depends on an FK ulp.
"""
import re
from collections import Counter

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-5                  # relative, the project's bar for float64 geometry
ENGINE_ID = {"exact": 0, "fast": 1, "brute": 2}
TJ = (2.3, 4.1)             # target_j of the choose_j_tar cases
N_BLOCKS = 8                # per-env targets: contiguous blocks of envs share one target


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


@pytest.fixture(scope="module")
def ops(ag):
    from abstract_gym_b200 import ops
    return ops


# ------------------------------------------------------------------ grids

def clear_base(occ, E):
    """free the cells around the arm's base at the origin: a map whose base cell is occupied has no free pose"""
    S = occ.shape[-1]
    c = int(np.floor((E / 2) / (E / (S - 1))))
    occ[..., max(c - 1, 0):c + 3, max(c - 2, 0):c + 2] = 0
    return occ


def random_occ(seed, G, S, p, E=1.6):
    rng = np.random.default_rng(seed)
    return clear_base((rng.random((G, S, S)) < p).astype(np.uint8), E)


# name -> (occ [G,S,S], environment size, envs_per_grid or None for one grid, AG_GRID_FORM)
GRIDS = {
    "scene0": lambda: (None, 1.6, None, ""),                                    # manual map: FAST's obstacle list
    "rand31": lambda: (random_occ(1, 1, 31, 0.01), 1.6, None, ""),
    "dense31": lambda: (random_occ(2, 1, 31, 0.5), 1.6, None, ""),              # stuck resets
    "rand64": lambda: (random_occ(3, 1, 64, 0.02), 1.6, None, ""),              # two-level form, staged
    "rand256": lambda: (random_occ(4, 1, 256, 0.005), 1.6, None, ""),           # two-level form, staged
    "rand256_t": lambda: (random_occ(5, 1, 256, 0.005), 1.6, None, "transposed"),
    "rand1024": lambda: (random_occ(6, 1, 1024, 0.002), 1.6, None, ""),         # two-level form, global memory
    "het256_epg256": lambda: (random_occ(7, 8, 256, 0.005), 1.6, 256, ""),      # block-uniform: staged
    "het256_epg100": lambda: (random_occ(8, 8, 256, 0.005), 1.6, 100, ""),      # per-thread grid lookup
    "edge9_e1": lambda: (random_occ(9, 1, 9, 0.3), 1.0, None, ""),              # the arm reaches past the grid
}


class Grid:
    """one GRIDS entry: the object the scene takes, its device form and the oracle's squares per grid"""

    def __init__(self, ag, torch, oracle, name, monkeypatch):
        occ, E, epg, form = GRIDS[name]()
        if form:
            monkeypatch.setenv("AG_GRID_FORM", form)
        else:
            monkeypatch.delenv("AG_GRID_FORM", raising=False)
        if occ is None:
            self.obj = ag.OccupancyGrid(size=9, random_obstacle=False)
            occ = np.zeros((1, 9, 9), dtype=np.uint8)
            for r, c in ag.OccupancyGrid.MANUAL_CELLS:
                occ[0, r, c] = 1
            self.squares = [oracle.manual_grid()[0]]
        elif epg is None:
            self.obj = ag.OccupancyGrid(size=occ.shape[1], random_obstacle=False)
            self.obj.load_from_matrix(occ[0], environment_size=E)
            self.squares = [oracle.grid_squares(occ[0], E)[0]]
        else:
            self.obj = ag.BatchedOccupancyGrid(torch.as_tensor(occ, device="cuda"), epg, environment_size=E, device="cuda")
            self.squares = [oracle.grid_squares(o, E)[0] for o in occ]
        self.dg = self.obj.device_grid("cuda")
        assert np.array_equal(self.dg.unpack(), occ)
        if form == "transposed":
            assert self.dg.bits_t is not None and self.dg.hier is None
        self.occ, self.E, self.S, self.G = occ, E, occ.shape[1], occ.shape[0]
        self.epg = epg if epg is not None else 1 << 62

    def of_env(self, gid):
        return (gid // self.epg) % self.G


# ------------------------------------------------------------------ references

def make_params(oracle, target=(-0.2, -0.3), joint=False):
    p = oracle.default_params()
    p.target_x, p.target_y = float(target[0]), float(target[1])
    if joint:
        p.choose_j_tar, p.target_j1, p.target_j2 = 1, TJ[0], TJ[1]
    return p


def fk_ref(oracle, j1, j2):
    """the oracle's forward kinematics (glibc sin / cos), batched: a zero-action step_batch on an empty map"""
    a, b = np.array(j1, dtype=np.float64), np.array(j2, dtype=np.float64)
    res = oracle.step_batch(a, b, np.zeros((len(a), 2)), np.zeros(len(a)), np.zeros(len(a), dtype=np.uint8),
                            np.zeros((0, 4)))
    assert np.array_equal(a, j1) and np.array_equal(b, j2)
    return res["ee"]


class Reference:
    """host mirror of the K6 state; step() advances it by one gym step and returns what K6 must write"""

    def __init__(self, oracle, grid, j1, j2, blocks, params, env_id0, seed, auto_reset):
        n = len(j1)
        self.o, self.grid, self.n = oracle, grid, n
        self.blocks, self.params = blocks, params          # [(lo, hi)], one oracle Params per block
        self.env_id0, self.seed, self.auto_reset = env_id0, seed, auto_reset
        self.st = [oracle.RolloutState(j1[lo:hi], j2[lo:hi]) for lo, hi in blocks]
        self.stats = np.zeros(oracle.ST_COUNT, dtype=np.int64)
        self.gid = env_id0 + np.arange(n, dtype=np.int64)
        self.g = grid.of_env(self.gid)

    def cat(self, k):
        return np.concatenate([getattr(s, k) for s in self.st])

    def targets(self):
        t = np.zeros((self.n, 2))
        for (lo, hi), p in zip(self.blocks, self.params):
            t[lo:hi] = (p.target_x, p.target_y)
        return t

    def step(self, a):
        """a: [n,2] float32 or float64.  -> dict(q1, q2 (post-step, pre-reset), reward, flags, rec_j1, rec_j2)"""
        q1, q2 = self.cat("j1") + a[:, 0].astype(np.float64), self.cat("j2") + a[:, 1].astype(np.float64)
        if a.dtype == np.float32 and self.auto_reset:
            out = self._step_rollout(a)
        else:
            out = self._step_batch(a.astype(np.float64))
        out.update(q1=q1, q2=q2)
        return out

    def _step_rollout(self, a):
        o = self.o
        rec = dict(j1=[], j2=[], reward=[], flags=[])
        for (lo, hi), p, s in zip(self.blocks, self.params, self.st):
            r, st = o.rollout(s, 1, self.grid.squares, envs_per_grid=self.grid.epg, env_id0=self.env_id0 + lo,
                              seed=self.seed, actions_f32=a[None, lo:hi], params=p)
            self.stats += st
            for k in rec:
                rec[k].append(r[k][0])
        rec = {k: np.concatenate(v) for k, v in rec.items()}
        return dict(reward=rec["reward"], flags=rec["flags"], rec_j1=rec["j1"], rec_j2=rec["j2"])

    def _step_batch(self, a):
        o, o_stats = self.o, self.stats
        j1, j2, rc, el = self.cat("j1"), self.cat("j2"), self.cat("reset_ctr"), self.cat("ep_len")
        rw, fl = self.cat("reward").astype(np.float64), self.cat("flags")
        for (lo, hi), p in zip(self.blocks, self.params):
            for g in np.unique(self.g[lo:hi]):
                idx = lo + np.flatnonzero(self.g[lo:hi] == g)
                b1, b2, brw, bfl = j1[idx], j2[idx], rw[idx], fl[idx]
                res = o.step_batch(b1, b2, a[idx], brw, bfl, self.grid.squares[g], params=p)
                j1[idx], j2[idx], rw[idx], fl[idx] = b1, b2, brw, bfl
                o_stats[o.ST_AXIS_ALIGNED] += res["axis_aligned"]
        out = dict(reward=rw.astype(np.float32), flags=fl.copy(), rec_j1=j1.astype(np.float32), rec_j2=j2.astype(np.float32))
        el = el + 1
        o_stats[o.ST_ENV_STEPS] += self.n
        if self.auto_reset:
            term = fl != 0
            o_stats[o.ST_EPISODES] += int(term.sum())
            o_stats[o.ST_COLLISIONS] += int((fl & 1).astype(bool).sum())
            o_stats[o.ST_SUCCESSES] += int((fl & 2).astype(bool).sum())
            o_stats[o.ST_EP_LEN_SUM] += int(el[term].sum())
            o_stats[o.ST_RETURN_MILLI] += int(np.round(rw[term] / 1000.0).sum())
            self._reset(j1, j2, rc, np.flatnonzero(fl & 1))
            rw[term], fl[term], el[term] = 0.0, 0, 0
        for (lo, hi), s in zip(self.blocks, self.st):
            s.j1[:], s.j2[:], s.reset_ctr[:], s.ep_len[:] = j1[lo:hi], j2[lo:hi], rc[lo:hi], el[lo:hi]
            s.reward[:], s.flags[:] = rw[lo:hi].astype(np.float32), fl[lo:hi]
        return out

    def _reset(self, j1, j2, rc, active):
        """Scene.reset() of the colliding terminated envs (scene_0.py:105-113,174-181): candidates (u*pi)*2.0 from
        Philox stream 1 keyed by (global id, reset_ctr) until one is collision-free, at most max_reset_tries.  (The
        oracle's collision_batch does not count axis-aligned evaluations of the candidates; none occur on these
        poses, and the float32 path checks that slot through the oracle's rollout.)"""
        o = self.o
        tries = 0
        while active.size:
            if tries >= self.params[0].max_reset_tries:
                self.stats[o.ST_STUCK_RESETS] += active.size
                break
            for e in active:
                u0, u1 = o.philox_uniform2(self.seed, int(self.gid[e]), int(rc[e]), 1)
                j1[e], j2[e] = (u0 * np.pi) * 2.0, (u1 * np.pi) * 2.0
            rc[active] += 1
            tries += 1
            hit = np.zeros(active.size, dtype=bool)
            for g in np.unique(self.g[active]):
                m = self.g[active] == g
                hit[m] = o.collision_batch(j1[active[m]], j2[active[m]], self.grid.squares[g], want_first_hit=False)[0] != 0
            active = active[hit]


def crop_ref(grid, gid_grid, ee, c):
    """c x c cells centred on the end effector's true (unclamped) cell: 2 outside [0, S), else the occupancy bit"""
    dg = grid.dg
    col = np.floor((ee[:, 0] + dg.environment_size / 2) / dg.side).astype(np.int64)
    row = (np.floor((dg.environment_size / 2 - ee[:, 1]) / dg.side) + 1).astype(np.int64)
    d = np.arange(c) - c // 2
    r = row[:, None, None] + d[None, :, None]
    cc = col[:, None, None] + d[None, None, :]
    r, cc = np.broadcast_arrays(r, cc)
    inside = (r >= 0) & (r < grid.S) & (cc >= 0) & (cc < grid.S)
    g = np.broadcast_to(gid_grid[:, None, None], r.shape)
    out = np.full(r.shape, 2, dtype=np.uint8)
    out[inside] = grid.occ[g[inside], r[inside], cc[inside]]
    return out


def geometry_close(got, want):
    err = np.abs(got - want)
    assert np.all(err <= TOL * np.maximum(np.abs(want), 1e-3)) and err.max(initial=0.0) < 1e-14, err.max(initial=0.0)


# ------------------------------------------------------------------ the two fronts

class OpFront:
    """K6 through torch.ops.abstract_gym_b200.step_obs on tensors this test owns"""

    def __init__(self, ag, torch, ops, grid, j1, j2, params, targets, engine, seed, auto_reset, env_id0, crop):
        n, dev = len(j1), "cuda"
        self.torch, self.ops = torch, ops
        self.P, self.GA = self._pack(ag, ops, params), ops.grid_args(grid.dg)
        self.j1, self.j2 = torch.as_tensor(j1, device=dev).clone(), torch.as_tensor(j2, device=dev).clone()
        self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flags = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.reset_ctr = torch.zeros(n, dtype=torch.int32, device=dev)
        self.ep_len = torch.zeros(n, dtype=torch.int32, device=dev)
        self.targets = None if targets is None else torch.as_tensor(targets, device=dev).contiguous()
        self.obs = torch.zeros(n, 6, dtype=torch.float64, device=dev)
        self.final_obs = torch.zeros(n, 6, dtype=torch.float64, device=dev)
        self.reward_out = torch.zeros(n, dtype=torch.float32, device=dev)
        self.terminated = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.collision = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.crop = torch.zeros(n, crop, crop, dtype=torch.uint8, device=dev) if crop else None
        self.stats = torch.zeros(len(ag.STAT_NAMES), dtype=torch.int64, device=dev)
        self.engine, self.seed, self.auto_reset, self.env_id0 = ENGINE_ID[engine], seed, auto_reset, env_id0

    @staticmethod
    def _pack(ag, ops, p):
        q = ag.default_params()
        for f, _ in type(p)._fields_:
            setattr(q, f, getattr(p, f))
        return ops.pack_params(q)

    def step(self, a):
        act = self.torch.as_tensor(a, device="cuda").contiguous()
        self.ops.step_obs(self.P, *self.GA, self.j1, self.j2, act, self.reward, self.flags, self.reset_ctr, self.ep_len,
                          self.targets, self.obs, self.reward_out, self.terminated, self.collision, self.final_obs, self.crop,
                          self.stats, self.seed, self.auto_reset, self.env_id0, self.engine)
        return self.read()

    def read(self):
        f = lambda t: None if t is None else t.cpu().numpy()
        return dict(obs=f(self.obs), final_obs=f(self.final_obs), reward_out=f(self.reward_out),
                    terminated=f(self.terminated), collision=f(self.collision), crop=f(self.crop),
                    j1=f(self.j1), j2=f(self.j2), reward=f(self.reward), flags=f(self.flags),
                    reset_ctr=f(self.reset_ctr).view(np.uint32), ep_len=f(self.ep_len).view(np.uint32), stats=f(self.stats))


class EnvFront:
    """K6 through VectorEnv.step (float64 actions), started from the given joints instead of reset()"""

    def __init__(self, ag, torch, grid, j1, j2, params, targets, engine, seed, auto_reset, env_id0, crop, graph=False):
        n = len(j1)
        self.torch = torch
        self.env = ag.VectorEnv(n, env=grid.obj, device="cuda", seed=seed, engine=engine, auto_reset=auto_reset,
                                target_c=ag.Point(params.target_x, params.target_y), choose_j_tar=bool(params.choose_j_tar),
                                env_id0=env_id0, targets=targets, crop_size=crop)
        sc = self.env.scene
        sc.target_j = np.array([params.target_j1, params.target_j2])
        sc.robot.joint_1.copy_(torch.as_tensor(j1, device="cuda"))
        sc.robot.joint_2.copy_(torch.as_tensor(j2, device="cuda"))
        if graph:
            self.env.capture()

    def step(self, a):
        obs, rw, term, trunc, info = self.env.step(self.torch.as_tensor(a, device="cuda"))
        assert not bool(trunc.any())
        sc = self.env.scene
        f = lambda t: None if t is None else t.cpu().numpy()
        return dict(obs=f(obs), final_obs=f(info["final_obs"]), reward_out=f(rw), terminated=f(term).astype(np.uint8),
                    collision=f(info["collision"]).astype(np.uint8), crop=f(info["crop"]),
                    j1=f(sc.robot.joint_1), j2=f(sc.robot.joint_2), reward=f(sc.step_reward), flags=f(sc.flags),
                    reset_ctr=f(sc.reset_ctr).view(np.uint32), ep_len=f(sc.ep_len).view(np.uint32), stats=f(sc.stats))


# ------------------------------------------------------------------ one case

def setup_case(oracle, n, T, target, huge, a_dtype, seed):
    """initial joints, per-step actions and the per-block targets.  Every target mode is reached by some env: the
    cartesian target (and each block's target) is the end effector of a block's first env after step 0; in joint mode a
    third of the envs start exactly one action short of target_j, and the odd envs roam the map from uniform poses."""
    rng = np.random.default_rng(seed)
    joint = target == "joint"
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    scale = np.full((n, 1), 0.3)
    if joint:
        near = np.arange(n) % 2 == 0
        j1[near], j2[near] = TJ[0] + rng.normal(0, 0.02, near.sum()), TJ[1] + rng.normal(0, 0.02, near.sum())
        scale[near] = 0.02
    if huge:
        j1[::5] += 2 * np.pi * np.round(rng.uniform(2e5, 3e6, len(j1[::5])))     # ~2^21 rad: float64 path of the filter
    acts = (rng.random((T, n, 2)) - 0.5) * scale
    if a_dtype == "f32":
        acts = acts.astype(np.float32)
    if joint:
        j1[::3], j2[::3] = TJ[0] - acts[0, ::3, 0].astype(np.float64), TJ[1] - acts[0, ::3, 1].astype(np.float64)
    nb = N_BLOCKS if target == "per_env" else 1
    edges = np.linspace(0, n, min(nb, n) + 1).astype(int)
    blocks = [(int(lo), int(hi)) for lo, hi in zip(edges[:-1], edges[1:])]
    ee0 = fk_ref(oracle, j1 + acts[0, :, 0].astype(np.float64), j2 + acts[0, :, 1].astype(np.float64))
    params = [make_params(oracle, ee0[lo] if target != "joint" else (-0.2, -0.3), joint) for lo, _ in blocks]
    return j1, j2, acts, blocks, params


def run_case(ag, torch, oracle, ops, monkeypatch, grid, engine, front, n, T, env_id0=0, target="cart",
             auto_reset=True, crop=3, huge=False, seed=None):
    seed = n + T + env_id0 + len(grid) if seed is None else seed
    g = Grid(ag, torch, oracle, grid, monkeypatch)
    a_dtype = "f32" if front == "op_f32" else "f64"
    j1, j2, acts, blocks, params = setup_case(oracle, n, T, target, huge, a_dtype, seed)
    ref = Reference(oracle, g, j1, j2, blocks, params, env_id0, seed, auto_reset)
    targets = ref.targets() if target == "per_env" else None
    args = (g, j1, j2, params[0], targets, engine, seed, auto_reset, env_id0, crop)
    dev = EnvFront(ag, torch, *args) if front == "env" else OpFront(ag, torch, ops, *args)
    tgt = ref.targets()
    seen = np.zeros(3, dtype=np.int64)          # terminal steps with collision, with done; steps of envs far out
    for t in range(T):
        a = acts[t]
        r = ref.step(a)
        d = dev.step(a)
        what = "%s step %d" % (grid, t)
        # the step itself: post-step joints, reward, flags
        assert np.array_equal(d["final_obs"][:, 0], r["q1"]) and np.array_equal(d["final_obs"][:, 1], r["q2"]), what
        assert np.array_equal(d["final_obs"][:, 0].astype(np.float32), r["rec_j1"]), what
        assert np.array_equal(d["final_obs"][:, 1].astype(np.float32), r["rec_j2"]), what
        assert np.array_equal(d["reward_out"], r["reward"]), what
        assert np.array_equal(d["terminated"], (r["flags"] != 0).astype(np.uint8)), what
        assert np.array_equal(d["collision"], (r["flags"] & 1).astype(np.uint8)), what
        # the state the env continues from, after the same-step reset
        assert np.array_equal(d["j1"], ref.cat("j1")) and np.array_equal(d["j2"], ref.cat("j2")), what
        assert np.array_equal(d["obs"][:, 0], d["j1"]) and np.array_equal(d["obs"][:, 1], d["j2"]), what
        assert np.array_equal(d["reset_ctr"], ref.cat("reset_ctr")) and np.array_equal(d["ep_len"], ref.cat("ep_len")), what
        assert np.array_equal(d["flags"], ref.cat("flags")) and np.array_equal(d["reward"], ref.cat("reward")), what
        assert np.array_equal(d["stats"], ref.stats), (what, d["stats"], ref.stats)
        # observation geometry: end effector and goal distance of the terminal and of the continuing pose
        for o, (q1, q2) in ((d["final_obs"], (r["q1"], r["q2"])), (d["obs"], (ref.cat("j1"), ref.cat("j2")))):
            ee = fk_ref(oracle, q1, q2)
            geometry_close(o[:, 2:4], ee)
            geometry_close(o[:, 4:6], np.abs(tgt - ee))
            assert np.array_equal(o[:, 4:6], np.abs(tgt - o[:, 2:4])), what
        # the crop around the continuing pose's end effector, every env
        if crop:
            want = crop_ref(g, ref.g, d["obs"][:, 2:4], crop)
            bad = np.flatnonzero((d["crop"] != want).any(axis=(1, 2)))
            assert bad.size == 0, "%s: crop differs for %d envs, first env %d at EE %s:\n%s\nwant\n%s" % (
                what, bad.size, bad[0], d["obs"][bad[0], 2:4], d["crop"][bad[0]], want[bad[0]])
        seen += [int((r["flags"] & 1).astype(bool).sum()), int((r["flags"] & 2).astype(bool).sum()),
                 int((np.abs(d["obs"][:, 2:4]) > g.E / 2).any(axis=1).sum())]
    st = dict(zip(ag.STAT_NAMES, ref.stats.tolist()))
    assert st["env_steps"] == n * T
    assert seen[0] > 0 and seen[1] > 0, (grid, seen)            # every case sees collisions and reached targets
    if auto_reset:
        assert st["episodes"] > 0 and st["collisions"] > 0 and st["successes"] > 0 and st["ep_len_sum"] > st["episodes"] - 1
    else:
        assert st["episodes"] == 0 and st["ep_len_sum"] == 0
        assert np.array_equal(d["ep_len"], np.full(n, T, dtype=np.uint32))                   # ep_len keeps counting
        assert np.array_equal(d["terminated"], (d["flags"] != 0).astype(np.uint8))           # terminated stays set
    return st, seen


# grid, engine, front (op_f32 / op_f64 / env = VectorEnv with float64), n, T, env_id0, target, auto_reset, crop, huge
CASES = [
    ("scene0", "fast", "env", 4096, 40, 0, "cart", True, 3, False),
    ("scene0", "exact", "op_f32", 4096, 30, 1000, "per_env", True, 1, True),
    ("scene0", "brute", "op_f64", 257, 30, 1000, "joint", True, 63, False),
    ("rand31", "exact", "env", 257, 30, 0, "joint", False, 31, False),
    ("rand31", "fast", "op_f32", 4096, 30, 1000, "cart", True, 3, False),
    ("dense31", "brute", "op_f32", 31, 20, 0, "cart", True, 1, False),
    ("dense31", "exact", "op_f64", 1, 40, 1000, "per_env", True, 3, False),
    ("dense31", "fast", "env", 257, 20, 0, "joint", True, 31, False),
    ("rand64", "fast", "op_f32", 4096, 30, 1000, "per_env", True, 31, False),
    ("rand256", "brute", "env", 257, 20, 0, "cart", False, 31, True),
    ("rand256_t", "fast", "op_f64", 4096, 30, 0, "joint", True, 63, False),
    ("rand256_t", "exact", "op_f32", 257, 20, 1000, "cart", True, 3, False),
    ("rand1024", "fast", "op_f32", 4096, 20, 0, "cart", False, 1, False),
    ("het256_epg256", "fast", "op_f32", 4096, 30, 0, "per_env", True, 3, True),
    ("het256_epg256", "exact", "op_f32", 4096, 30, 0, "cart", False, 63, False),
    ("het256_epg100", "exact", "env", 4096, 30, 1000, "cart", True, 31, False),
    ("het256_epg100", "brute", "op_f32", 257, 20, 1000, "joint", False, 1, False),
    ("het256_epg100", "fast", "op_f64", 257, 30, 1000, "per_env", False, 3, False),
    ("edge9_e1", "fast", "op_f32", 4096, 30, 0, "cart", True, 3, False),
    ("edge9_e1", "exact", "env", 257, 30, 1000, "per_env", True, 31, False),
    ("edge9_e1", "brute", "op_f32", 31, 30, 0, "per_env", False, 3, False),
]


@pytest.mark.parametrize("grid,engine,front,n,T,env_id0,target,auto_reset,crop,huge", CASES,
                         ids=["-".join(str(x) for x in c[:4]) + ("-%s" % c[6]) + ("-noreset" if not c[7] else "")
                              + "-c%d" % c[8] + ("-huge" if c[9] else "") + "-id%d" % c[5] for c in CASES])
def test_step_obs_vs_oracle(ag, torch_, oracle, ops, monkeypatch, grid, engine, front, n, T, env_id0, target, auto_reset,
                            crop, huge):
    st, seen = run_case(ag, torch_, oracle, ops, monkeypatch, grid, engine, front, n, T, env_id0, target, auto_reset, crop,
                        huge)
    if grid == "dense31":
        assert st["stuck_resets"] > 0                      # max_reset_tries exhausted
    if grid == "edge9_e1":
        assert seen[2] > 0                                 # end effectors beyond the grid's edge reach the crop


@pytest.mark.parametrize("engine", ["exact", "fast", "brute"])
def test_float32_exact_actions_as_float64(ag, torch_, oracle, ops, monkeypatch, engine):
    """float32 actions and the same values given as float64 take different K6 instantiations and must agree bit for bit"""
    n, T = 257 if engine == "brute" else 4096, 20
    g = Grid(ag, torch_, oracle, "het256_epg100", monkeypatch)
    j1, j2, acts, blocks, params = setup_case(oracle, n, T, "cart", True, "f32", 5)
    fronts = [OpFront(ag, torch_, ops, g, j1, j2, params[0], None, engine, 5, True, 1000, 3) for _ in range(2)]
    for t in range(T):
        a = fronts[0].step(acts[t])
        b = fronts[1].step(acts[t].astype(np.float64))
        for k in a:
            assert np.array_equal(a[k], b[k]), (engine, t, k)
    assert a["stats"][0] > 0


@pytest.mark.parametrize("engine", ["exact", "fast"])
def test_vector_env_graph_equals_eager_heterogeneous(ag, torch_, oracle, engine, monkeypatch):
    """VectorEnv.capture() replays the same K6 launch: identical outputs and state on heterogeneous grids"""
    n, T = 4096, 20
    g = Grid(ag, torch_, oracle, "het256_epg100", monkeypatch)
    j1, j2, acts, blocks, params = setup_case(oracle, n, T, "per_env", False, "f64", 9)
    tg = Reference(oracle, g, j1, j2, blocks, params, 0, 9, True).targets()
    eager, graph = (EnvFront(ag, torch_, g, j1, j2, params[0], tg, engine, 9, True, 1000, 31, graph=c) for c in (False, True))
    for t in range(T):
        a, b = eager.step(acts[t]), graph.step(acts[t])
        for k in a:
            assert np.array_equal(a[k], b[k]), (engine, t, k)
    assert a["stats"][0] > 0 and a["stats"][2] > 0


_DEMANGLED = re.compile(r"k_step_obs<\s*(\d+)\s*,\s*(true|false)\s*>")
_MANGLED = re.compile(r"k_step_obsILi(\d+)ELb([01])E")


def test_every_instantiation_launches(ag, torch_, oracle, ops, monkeypatch):
    """the dispatch of ag_step_obs reaches all six k_step_obs<engine, float32 actions> instantiations, each from the
    engine and action dtype it was asked for (kernel names from the profiler's CUDA activity)"""
    from torch.profiler import ProfilerActivity, profile
    g = Grid(ag, torch_, oracle, "scene0", monkeypatch)
    j1, j2, acts, blocks, params = setup_case(oracle, 64, 1, "cart", False, "f64", 3)
    want = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for engine, eid in ENGINE_ID.items():
            for f32 in (False, True):
                f = OpFront(ag, torch_, ops, g, j1, j2, params[0], None, engine, 3, True, 0, 3)
                f.step(acts[0].astype(np.float32) if f32 else acts[0])
                want.append((eid, f32))
        torch_.cuda.synchronize()
    got = []
    for e in prof.events():
        m = _DEMANGLED.search(e.name) or _MANGLED.search(e.name)
        if m:
            got.append((int(m.group(1)), m.group(2) in ("true", "1")))
    assert Counter(got) == Counter(want), got
    assert len(set(got)) == 6


def test_step_obs_op_checks_element_counts(ag, torch_, oracle, ops, monkeypatch):
    """every state and output tensor of the step_obs op is checked for its element count before anything launches"""
    n = 64
    g = Grid(ag, torch_, oracle, "scene0", monkeypatch)
    j1, j2, acts, blocks, params = setup_case(oracle, n, 1, "cart", False, "f64", 4)
    f = OpFront(ag, torch_, ops, g, j1, j2, params[0], np.zeros((n, 2)), "fast", 4, True, 0, 3)
    sizes = dict(j2=n, reward=n, flags=n, reset_ctr=n, ep_len=n, reward_out=n, terminated=n, collision=n,
                 stats=len(ag.STAT_NAMES), targets=2 * n, final_obs=6 * n)
    for name, count in sizes.items():
        good = getattr(f, name)
        assert good.numel() == count
        setattr(f, name, good.flatten()[:count - 1].clone())
        before = ag.launch_count()
        with pytest.raises(RuntimeError):
            f.step(acts[0])
        torch_.cuda.synchronize()
        assert ag.launch_count() == before, name
        setattr(f, name, good)
    before = ag.launch_count()
    f.step(acts[0])
    assert ag.launch_count() == before + 1
