"""Every instantiation of the rollout (k_rollout, k_rollout_async, k_rollout_lut), step (k_step), reset (k_reset) and
collision (k_collision) kernel families against the CPU oracle, each from the inputs that reach it.

Every rollout row of ROLLOUT_ROWS names one instantiation and the inputs that reach it under ag_rollout_impl
(csrc/ag_kernels.cu) and launch_rollout_lut (csrc/ag_rollout_lut.cu); the profiler's CUDA activity must show exactly
that kernel, so a dispatch change fails the row that depended on it.  A captured rollout is identified by the kernel
nodes of its graph (the graph's DOT dump).  test_rows_cover_every_instantiation reads the
instantiations of the six families from the release library: a new one without a row fails there.

Per-env targets are checked against the oracle, which has one scene-wide target, the way test_step_obs_gpu does it: the
envs are split into contiguous blocks that share a target, and the oracle runs once per block with env_id0 + lo and the
block's Params, which keeps the Philox keys and the env -> grid mapping ((gid // epg) % G) those of the device.  The first
env of most blocks gets a target reach_eps -+ 1e-12 from its step-0 end effector (in x or in y): far above the
CUDA / glibc sincos difference (~1e-16), far below the float32 filter's band, so those envs take the float64 decision.

The bar is test_gpu_parity's: record planes, final joints, reward, flags, step_ctr, reset_ctr, ep_len and the whole
statistics vector bit for bit; for k_step the geometry within 1e-5 relative and 1e-14 absolute.
"""
import gc
import html
import re
from collections import Counter

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-5                  # relative, the project's bar for float64 geometry
ENGINE_ID = {"exact": 0, "fast": 1, "brute": 2}
TJ = (2.3, 4.1)             # target_j of the joint-target rows
N_BLOCKS = 16               # per-env targets: contiguous blocks of envs share one target
FAMILIES = ("k_rollout", "k_rollout_async", "k_rollout_lut", "k_step", "k_reset", "k_collision")


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


# ------------------------------------------------------------------ kernel names

def _template_args(s):
    return tuple(1 if a == "true" else 0 if a == "false" else int(a) for a in (x.strip() for x in s.split(",")))


def kernel_of(name):
    """(family, template arguments) of a kernel name of one of FAMILIES, demangled or mangled; None otherwise"""
    for f in FAMILIES:
        m = re.search(r"(?<![A-Za-z0-9_])%s<([^<>]*)>" % f, name)
        if m:
            return f, _template_args(m.group(1))
        m = re.search(r"%d%sI((?:L[ib]-?\d+E)+)E" % (len(f), f), name)
        if m:
            return f, tuple(int(v) for v in re.findall(r"L[ib](-?\d+)E", m.group(1)))
    return None


def launched_kernels(torch, fn):
    """run fn() under the profiler; -> the (family, args) of every launch of FAMILIES, in order"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [k for k in (kernel_of(e.name) for e in prof.events()) if k is not None]


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


def cells_occ(S, cells, G=1):
    occ = np.zeros((G, S, S), dtype=np.uint8)
    for g, r, c in cells:
        occ[g, r, c] = 1
    return occ


def list4():
    """four 9x9 grids of at most 8 cells each: the obstacle list on staged per-batch grids"""
    rng = np.random.default_rng(11)
    occ = np.zeros((4, 9, 9), dtype=np.uint8)
    for g in range(4):
        free = np.flatnonzero(clear_base(np.ones((9, 9), dtype=np.uint8), 1.6).ravel())
        occ[g].ravel()[rng.choice(free, 4 + g, replace=False)] = 1
    return occ


SCENE0_CELLS = [(0, 5, 6), (0, 5, 7), (0, 2, 3)]                       # occupancy_grid.py:45-47, (row, col)
SIX9_CELLS = [(0, 1, 1), (0, 1, 7), (0, 7, 1), (0, 7, 7), (0, 2, 5), (0, 6, 6)]

# name -> (occ [G,S,S], environment size, envs_per_grid or None for one grid)
GRIDS = {
    "scene0": lambda: (cells_occ(9, SCENE0_CELLS), 1.6, None),            # 3 cells: the M3 table-arm form
    "six9": lambda: (cells_occ(9, SIX9_CELLS), 1.6, None),                # 6 cells: the general table-arm form
    "list4_epg256": lambda: (list4(), 1.6, 256),                          # staged per-batch obstacle lists
    "rand31": lambda: (random_occ(1, 1, 31, 0.03), 1.6, None),            # > 8 cells: traversal
    "dense31": lambda: (random_occ(2, 1, 31, 0.5), 1.6, None),            # stuck resets
    "het64_epg100": lambda: (random_occ(3, 4, 64, 0.01), 1.6, 100),       # unstaged, per-thread grid lookup
    "edge9_e1": lambda: (random_occ(4, 1, 9, 0.3), 1.0, None),            # the arm reaches past the grid; > 8 cells
}


class Grid:
    def __init__(self, ag, torch, oracle, occ, E, epg):
        self.occ, self.E, self.S, self.G = occ, E, occ.shape[1], occ.shape[0]
        self.epg = epg if epg is not None else 1 << 62
        self.dg = ag.DeviceGrid.from_device_matrices(torch.as_tensor(occ, device="cuda"), E, self.epg)
        assert np.array_equal(self.dg.unpack(), occ)
        sq = [oracle.grid_squares(o, E) for o in occ]
        self.squares, self.cells = [q for q, _ in sq], [c for _, c in sq]

    @classmethod
    def named(cls, ag, torch, oracle, name):
        return cls(ag, torch, oracle, *GRIDS[name]())

    def of_env(self, gid):
        return (gid // self.epg) % self.G


@pytest.fixture(autouse=True)
def _rows_grid_form(monkeypatch):
    monkeypatch.delenv("AG_GRID_FORM", raising=False)          # every grid in its default device form


# ------------------------------------------------------------------ parameters and targets

def make_params(oracle, target=(-0.2, -0.3), joint=False, links=None, tries=None):
    p = oracle.default_params()
    p.target_x, p.target_y = float(target[0]), float(target[1])
    if joint:
        p.choose_j_tar, p.target_j1, p.target_j2 = 1, TJ[0], TJ[1]
    if links:
        p.link_1, p.link_2 = links
    if tries is not None:
        p.max_reset_tries = tries
    return p


def pack(ag, ops, p):
    q = ag.default_params()
    for f, _ in type(p)._fields_:
        setattr(q, f, getattr(p, f))
    return ops.pack_params(q)


def fk_ref(oracle, j1, j2, p=None):
    """the oracle's forward kinematics (glibc sin / cos), batched: a zero-action step_batch on an empty map"""
    a, b = np.array(j1, dtype=np.float64), np.array(j2, dtype=np.float64)
    res = oracle.step_batch(a, b, np.zeros((len(a), 2)), np.zeros(len(a)), np.zeros(len(a), dtype=np.uint8),
                            np.zeros((0, 4)), params=p)
    assert np.array_equal(a, j1) and np.array_equal(b, j2)
    return res["ee"]


def philox_action(oracle, p, seed, gid, ctr):
    """the in-kernel action of step counter ctr (Philox stream 0): (u - 0.5) * action_scale, float64"""
    u0, u1 = oracle.philox_uniform2(seed, int(gid), int(ctr), 0)
    return (u0 - 0.5) * p.action_scale, (u1 - 0.5) * p.action_scale


def boundary_targets(oracle, ee0, blocks, p, E):
    """one target per block.  Block b's first env ends step 0 at ee0[lo]: its target sits reach_eps - 1e-12 (even b,
    reached) or reach_eps + 1e-12 (odd b, missed) from it, in x or in y, on either side.  With more than two blocks the
    last two are out of reach inside the grid and outside the grid.  -> ([(tx, ty)] per block, [(lo, reached)])"""
    tg, probes = [], []
    nb = len(blocks)
    for b, (lo, hi) in enumerate(blocks):
        if nb > 2 and b == nb - 2:
            tg.append((0.75, 0.0)); continue
        if nb > 2 and b == nb - 1:
            tg.append((E / 2 + 0.3, -(E / 2 + 0.2))); continue
        t = np.array(ee0[lo], dtype=np.float64)
        off = p.reach_eps + (1e-12 if b % 2 else -1e-12)
        t[(b // 2) % 2] += off if (b // 4) % 2 == 0 else -off
        tg.append((t[0], t[1]))
        probes.append((lo, b % 2 == 0))
    return tg, probes


# ------------------------------------------------------------------ rollout rows

def R(kernel, args, grid, engine, n, K, env_id0=0, opts=""):
    return (kernel, tuple(args), grid, engine, n, K, env_id0, opts)


# options: ha = actions given; hr<R> = reset_u with R candidates; rec = all four record planes; joints = joint planes
# only; misal = all four planes, the reward plane 4 bytes off 16-byte alignment (no warp-wide zero fill); per_env =
# per-env targets; joint = joint-target mode; long = links 0.6 / 0.6 (beyond the table arm's error budget); sticky =
# flags, reward and counters left by earlier calls; huge = joints near 2^20 and 2^21 rad; ev = event sink; evshort =
# event sink with less capacity than events; tries<k> = max_reset_tries
ROLLOUT_ROWS = [
    # EXACT: k_rollout<0, BP_ANY, HA, HR, REC, false, 256>
    R("k_rollout", (0, 0, 0, 0, 0, 0, 256), "dense31", "exact", 4096, 3, 1000, "huge"),
    R("k_rollout", (0, 0, 0, 0, 1, 0, 256), "scene0", "exact", 257, 5, 0, "rec per_env sticky"),
    R("k_rollout", (0, 0, 0, 1, 0, 0, 256), "dense31", "exact", 1, 40, 1000, "hr3"),
    R("k_rollout", (0, 0, 0, 1, 1, 0, 256), "rand31", "exact", 31, 4, 0, "hr2 joints evshort sticky"),
    R("k_rollout", (0, 0, 1, 0, 0, 0, 256), "edge9_e1", "exact", 4096, 2, 0, "ha joint"),
    R("k_rollout", (0, 0, 1, 0, 1, 0, 256), "het64_epg100", "exact", 257, 17, 1000, "ha rec per_env ev"),
    R("k_rollout", (0, 0, 1, 1, 0, 0, 256), "het64_epg100", "exact", 4096, 1, 0, "ha hr4 sticky"),
    R("k_rollout", (0, 0, 1, 1, 1, 0, 256), "dense31", "exact", 4096, 5, 0, "ha hr8 rec huge"),
    # BRUTE: k_rollout<2, BP_ANY, HA, HR, REC, false, 256>, small n
    R("k_rollout", (2, 0, 0, 0, 0, 0, 256), "scene0", "brute", 31, 4, 1000, "sticky"),
    R("k_rollout", (2, 0, 0, 0, 1, 0, 256), "rand31", "brute", 257, 3, 0, "rec per_env huge"),
    R("k_rollout", (2, 0, 0, 1, 0, 0, 256), "dense31", "brute", 1, 20, 0, "hr2"),
    R("k_rollout", (2, 0, 0, 1, 1, 0, 256), "edge9_e1", "brute", 257, 5, 1000, "hr6 joints ev"),
    R("k_rollout", (2, 0, 1, 0, 0, 0, 256), "het64_epg100", "brute", 257, 2, 1000, "ha tries3"),
    R("k_rollout", (2, 0, 1, 0, 1, 0, 256), "six9", "brute", 32, 1, 0, "ha rec joint"),
    R("k_rollout", (2, 0, 1, 1, 0, 0, 256), "rand31", "brute", 31, 5, 0, "ha hr3 sticky"),
    R("k_rollout", (2, 0, 1, 1, 1, 0, 256), "scene0", "brute", 257, 40, 0, "ha hr24 rec per_env evshort"),
    # FAST, obstacle list, one grid, complete warps: k_rollout<1, BP_LIST, HA, HR, REC, true, 32> (the LUT kept
    # out by joint-target mode, long links or records without the zero fill)
    R("k_rollout", (1, 1, 0, 0, 0, 1, 32), "scene0", "fast", 4096, 5, 0, "joint"),
    R("k_rollout", (1, 1, 0, 0, 1, 1, 32), "six9", "fast", 64, 3, 0, "misal per_env"),
    R("k_rollout", (1, 1, 0, 1, 0, 1, 32), "scene0", "fast", 32, 2, 0, "hr2 long"),
    R("k_rollout", (1, 1, 0, 1, 1, 1, 32), "six9", "fast", 4096, 4, 1000, "hr3 joints long ev"),
    R("k_rollout", (1, 1, 1, 0, 0, 1, 32), "six9", "fast", 4096, 1, 0, "ha long sticky huge"),
    R("k_rollout", (1, 1, 1, 0, 1, 1, 32), "scene0", "fast", 4096, 40, 0, "ha rec joint ev"),
    R("k_rollout", (1, 1, 1, 1, 0, 1, 32), "six9", "fast", 32, 3, 1000, "ha hr2 joint"),
    R("k_rollout", (1, 1, 1, 1, 1, 1, 32), "scene0", "fast", 4096, 17, 0, "ha hr24 misal per_env sticky"),
    # FAST, obstacle list, one grid, ragged n: k_rollout<1, BP_LIST, HA, HR, REC, false, 32>
    R("k_rollout", (1, 1, 0, 0, 0, 0, 32), "scene0", "fast", 257, 4, 0, "long"),
    R("k_rollout", (1, 1, 0, 0, 1, 0, 32), "six9", "fast", 31, 5, 1000, "rec per_env"),
    R("k_rollout", (1, 1, 0, 1, 0, 0, 32), "six9", "fast", 1, 40, 0, "hr2 joint"),
    R("k_rollout", (1, 1, 0, 1, 1, 0, 32), "scene0", "fast", 257, 3, 0, "hr3 joints evshort"),
    R("k_rollout", (1, 1, 1, 0, 0, 0, 32), "scene0", "fast", 31, 2, 0, "ha joint huge"),
    R("k_rollout", (1, 1, 1, 0, 1, 0, 32), "six9", "fast", 257, 17, 0, "ha rec sticky"),
    R("k_rollout", (1, 1, 1, 1, 0, 0, 32), "six9", "fast", 257, 5, 0, "ha hr4 long sticky"),
    R("k_rollout", (1, 1, 1, 1, 1, 0, 32), "scene0", "fast", 1, 1, 1000, "ha hr2 rec"),
    # FAST, obstacle list, staged per-batch grids: k_rollout<1, BP_LIST, HA, HR, REC, false, 256>
    R("k_rollout", (1, 1, 0, 0, 0, 0, 256), "list4_epg256", "fast", 4096, 3, 0, ""),
    R("k_rollout", (1, 1, 0, 0, 1, 0, 256), "list4_epg256", "fast", 1024, 5, 512, "rec per_env"),
    R("k_rollout", (1, 1, 0, 1, 0, 0, 256), "list4_epg256", "fast", 257, 4, 768, "hr2"),
    R("k_rollout", (1, 1, 0, 1, 1, 0, 256), "list4_epg256", "fast", 1024, 2, 0, "hr3 joints ev"),
    R("k_rollout", (1, 1, 1, 0, 0, 0, 256), "list4_epg256", "fast", 4096, 1, 256, "ha joint"),
    R("k_rollout", (1, 1, 1, 0, 1, 0, 256), "list4_epg256", "fast", 1000, 17, 0, "ha rec sticky huge"),
    R("k_rollout", (1, 1, 1, 1, 0, 0, 256), "list4_epg256", "fast", 1024, 5, 512, "ha hr4 long"),
    R("k_rollout", (1, 1, 1, 1, 1, 0, 256), "list4_epg256", "fast", 4096, 4, 0, "ha hr8 rec per_env evshort"),
    # FAST, traversal (more than 8 cells, or an unstaged grid): k_rollout_async<BP_TRAVERSAL, HA, HR, REC>
    R("k_rollout_async", (2, 0, 0, 0), "rand31", "fast", 4096, 3, 0, ""),
    R("k_rollout_async", (2, 0, 0, 1), "het64_epg100", "fast", 257, 5, 1000, "rec per_env"),
    R("k_rollout_async", (2, 0, 1, 0), "dense31", "fast", 257, 4, 0, "hr2"),
    R("k_rollout_async", (2, 0, 1, 1), "edge9_e1", "fast", 31, 2, 0, "hr3 joints evshort"),
    R("k_rollout_async", (2, 1, 0, 0), "het64_epg100", "fast", 1, 40, 1000, "ha joint"),
    R("k_rollout_async", (2, 1, 0, 1), "rand31", "fast", 4096, 17, 0, "ha rec huge sticky ev tries4"),
    R("k_rollout_async", (2, 1, 1, 0), "dense31", "fast", 4096, 5, 0, "ha hr6"),
    R("k_rollout_async", (2, 1, 1, 1), "rand31", "fast", 257, 1, 0, "ha hr2 rec per_env sticky"),
    # the persistent kernel k_rollout_lut<HA, REC, M3, CM>: the map form with the scene-wide target ...
    R("k_rollout_lut", (0, 0, 0, 1), "scene0", "fast", 257, 5, 1000, ""),
    R("k_rollout_lut", (0, 1, 0, 1), "six9", "fast", 4096, 17, 0, "rec ev"),
    R("k_rollout_lut", (1, 0, 0, 1), "six9", "fast", 1, 3, 0, "ha hr2 sticky"),
    R("k_rollout_lut", (1, 1, 0, 1), "scene0", "fast", 4096, 40, 0, "ha joints evshort huge"),
    # ... and the table-arm forms with per-env targets: M3 (at most 3 cells) and general (4 to 8)
    R("k_rollout_lut", (0, 0, 1, 0), "scene0", "fast", 31, 4, 0, "per_env hr3"),
    R("k_rollout_lut", (0, 1, 1, 0), "scene0", "fast", 4096, 5, 0, "per_env rec sticky"),
    R("k_rollout_lut", (1, 0, 1, 0), "scene0", "fast", 4096, 2, 1000, "per_env ha huge"),
    R("k_rollout_lut", (1, 1, 1, 0), "scene0", "fast", 64, 17, 0, "per_env ha hr4 joints ev"),
    R("k_rollout_lut", (0, 0, 0, 0), "six9", "fast", 4096, 1, 0, "per_env huge"),
    R("k_rollout_lut", (0, 1, 0, 0), "six9", "fast", 32, 40, 0, "per_env rec hr24"),
    R("k_rollout_lut", (1, 0, 0, 0), "six9", "fast", 257, 3, 1000, "per_env ha sticky"),
    R("k_rollout_lut", (1, 1, 0, 0), "six9", "fast", 4096, 4, 0, "per_env ha rec evshort"),
]


def parse_opts(s):
    o = dict(ha=False, R=0, rec=None, target="scene", sticky=False, huge=False, events=None, links=None, tries=None)
    for tok in s.split():
        if tok == "ha":
            o["ha"] = True
        elif tok.startswith("hr"):
            o["R"] = int(tok[2:])
        elif tok in ("rec", "joints", "misal"):
            o["rec"] = tok
        elif tok in ("per_env", "joint"):
            o["target"] = tok
        elif tok in ("sticky", "huge"):
            o[tok] = True
        elif tok in ("ev", "evshort"):
            o["events"] = tok
        elif tok == "long":
            o["links"] = (0.6, 0.6)
        elif tok.startswith("tries"):
            o["tries"] = int(tok[5:])
        else:
            raise ValueError(tok)
    return o


class RolloutCase:
    """the inputs of one rollout, its oracle reference (one oracle.rollout per target block) and its device run"""

    def __init__(self, oracle, grid, n, K, env_id0, seed, o):
        rng = np.random.default_rng(seed)
        self.grid, self.n, self.K, self.env_id0, self.seed, self.o = grid, n, K, env_id0, seed, o
        j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
        if o["huge"]:                                     # around the map's phase range and the float32 filter's
            i = np.arange(0, n, 5)
            j1[i] += np.where(i % 2 == 0, 1.0, -1.0) * 2.0 ** 20 + rng.uniform(-3, 3, len(i))
            j2[i[::2]] += 2.0 ** 21 + rng.uniform(-3, 3, len(i[::2]))
        self.acts = ((rng.random((K, n, 2)) - 0.5) * 0.3).astype(np.float32) if o["ha"] else None
        self.reset_u = rng.random((n, o["R"], 2)) if o["R"] else None
        # entry state
        self.flags0 = np.zeros(n, np.uint8)
        self.reward0 = np.zeros(n, np.float32)
        self.step_ctr0 = np.zeros(n, np.uint32)
        self.reset_ctr0 = np.zeros(n, np.uint32)
        self.ep_len0 = np.zeros(n, np.uint32)
        if o["sticky"]:
            s = rng.random(n) < 0.25
            self.flags0[s] = rng.integers(1, 4, int(s.sum()))
            self.reward0[s] = np.where(self.flags0[s] & 2, 10.0, -1000.0).astype(np.float32)
            self.ep_len0[:] = rng.integers(0, 50, n)
            self.step_ctr0[:] = rng.integers(0, 1 << 20, n)
            self.reset_ctr0[:] = rng.integers(0, max(o["R"], 3) + 1, n)      # some at R: no candidate left
        base = make_params(oracle, joint=o["target"] == "joint", links=o["links"], tries=o["tries"])
        self.base = base
        # step-0 actions (float64), for targets placed relative to the step-0 end effector
        if self.acts is not None:
            a0 = self.acts[0].astype(np.float64)
        else:
            a0 = np.array([philox_action(oracle, base, seed, env_id0 + e, self.step_ctr0[e]) for e in range(n)])
        if o["target"] == "joint":                      # every third env ends step 0 on target_j
            j1[::3], j2[::3] = TJ[0] - a0[::3, 0], TJ[1] - a0[::3, 1]
        self.j1, self.j2 = j1, j2
        nb = min(N_BLOCKS, n) if o["target"] == "per_env" else 1
        edges = np.linspace(0, n, nb + 1).astype(int)
        self.blocks = [(int(lo), int(hi)) for lo, hi in zip(edges[:-1], edges[1:])]
        self.probes = []
        if o["target"] == "joint":
            self.params = [base]
        else:
            ee0 = fk_ref(oracle, j1 + a0[:, 0], j2 + a0[:, 1], base)
            tg, self.probes = boundary_targets(oracle, ee0, self.blocks, base, grid.E)
            self.params = []
            for t in tg:
                p = make_params(oracle, t, links=o["links"], tries=o["tries"])
                self.params.append(p)
        self.targets = None
        if o["target"] == "per_env":
            self.targets = np.zeros((n, 2))
            for (lo, hi), p in zip(self.blocks, self.params):
                self.targets[lo:hi] = (p.target_x, p.target_y)

    def reference(self, oracle):
        rec = dict(j1=[], j2=[], reward=[], flags=[])
        fin = dict(j1=[], j2=[], reward=[], flags=[], step_ctr=[], reset_ctr=[], ep_len=[])
        stats = np.zeros(oracle.ST_COUNT, dtype=np.int64)
        epg = self.grid.epg if self.grid.G > 1 else None
        for (lo, hi), p in zip(self.blocks, self.params):
            st = oracle.RolloutState(self.j1[lo:hi], self.j2[lo:hi])
            st.flags[:], st.reward[:] = self.flags0[lo:hi], self.reward0[lo:hi]
            st.step_ctr[:], st.reset_ctr[:], st.ep_len[:] = self.step_ctr0[lo:hi], self.reset_ctr0[lo:hi], self.ep_len0[lo:hi]
            r, s = oracle.rollout(st, self.K, self.grid.squares, envs_per_grid=epg, env_id0=self.env_id0 + lo,
                                  seed=self.seed, actions_f32=None if self.acts is None else self.acts[:, lo:hi],
                                  reset_u=None if self.reset_u is None else self.reset_u[lo:hi], params=p)
            stats += s
            for k in rec:
                rec[k].append(r[k])
            for k in fin:
                fin[k].append(getattr(st, k))
        rec = {k: np.concatenate(v, axis=1) for k, v in rec.items()}
        fin = {k: np.concatenate(v) for k, v in fin.items()}
        return rec, fin, stats

    def device(self, ag, torch, ops, event_cap=0):
        n, K, dev = self.n, self.K, "cuda"
        T = lambda a: torch.as_tensor(a, device=dev).clone()
        self.t = t = dict(j1=T(self.j1), j2=T(self.j2), reward=T(self.reward0), flags=T(self.flags0),
                          step_ctr=T(self.step_ctr0.view(np.int32)), reset_ctr=T(self.reset_ctr0.view(np.int32)),
                          ep_len=T(self.ep_len0.view(np.int32)),
                          stats=torch.zeros(len(ag.STAT_NAMES), dtype=torch.int64, device=dev),
                          diag=torch.zeros(3, dtype=torch.int64, device=dev))
        t["actions"] = None if self.acts is None else T(self.acts)
        t["reset_u"] = None if self.reset_u is None else T(self.reset_u)
        t["targets"] = None if self.targets is None else T(self.targets)
        rec = self.o["rec"]
        z = lambda dt: torch.zeros(K, n, dtype=dt, device=dev)
        t["rec_j1"], t["rec_j2"] = (z(torch.float32), z(torch.float32)) if rec else (None, None)
        t["rec_reward"], t["rec_flags"] = (z(torch.float32), z(torch.uint8)) if rec in ("rec", "misal") else (None, None)
        if rec == "misal":                               # 4 bytes past a 16-byte boundary: no warp-wide zero fill
            t["rec_reward"] = torch.zeros(K * n + 1, dtype=torch.float32, device=dev)[1:].view(K, n)
            assert t["rec_reward"].data_ptr() % 16 == 4 and t["rec_reward"].is_contiguous()
        t["events"] = t["event_count"] = None
        if self.o["events"]:
            t["events"] = torch.zeros(3 * max(event_cap, 0), dtype=torch.int32, device=dev)
            t["event_count"] = torch.zeros(1, dtype=torch.int64, device=dev)
        self.P, self.GA = pack(ag, ops, self.params[0]), ops.grid_args(self.grid.dg)

    def launch(self, ops):
        t = self.t
        ops.rollout(self.P, *self.GA, t["j1"], t["j2"], t["reward"], t["flags"], t["step_ctr"], t["reset_ctr"], t["ep_len"],
                    t["actions"], t["reset_u"], t["targets"], t["rec_j1"], t["rec_j2"], t["rec_reward"], t["rec_flags"],
                    t["stats"], t["diag"], t["events"], t["event_count"], self.K, self.seed, self.env_id0,
                    ENGINE_ID[self.engine])

    def compare(self, oracle, ref, what):
        rec, fin, stats = ref
        t = self.t
        f = lambda x: x.cpu().numpy()
        planes = {"rec": ("j1", "j2", "reward", "flags"), "misal": ("j1", "j2", "reward", "flags"),
                  "joints": ("j1", "j2"), None: ()}[self.o["rec"]]
        for k in planes:
            got = f(t["rec_" + k])
            bad = np.argwhere(got != rec[k])
            assert bad.size == 0, "%s: record plane %s differs at %d (step, env), first %s: %s vs %s" % (
                what, k, len(bad), bad[0], got[tuple(bad[0])], rec[k][tuple(bad[0])])
        assert np.array_equal(f(t["j1"]), fin["j1"]) and np.array_equal(f(t["j2"]), fin["j2"]), what
        assert np.array_equal(f(t["reward"]), fin["reward"]) and np.array_equal(f(t["flags"]), fin["flags"]), what
        for k in ("step_ctr", "reset_ctr", "ep_len"):
            assert np.array_equal(f(t[k]).view(np.uint32), fin[k]), (what, k)
        assert np.array_equal(f(t["stats"]), stats), (what, f(t["stats"]), stats)
        if self.o["events"]:
            want = [(e, (s << 8) | int(rec["flags"][s, e]), int(rec["reward"][s, e:e + 1].view(np.uint32)[0]))
                    for s, e in zip(*np.nonzero((rec["flags"] != 0) | (rec["reward"] != 0)))]
            count = int(f(t["event_count"])[0])
            cap = t["events"].numel() // 3
            got = [tuple(int(x) for x in r) for r in f(t["events"]).view(np.uint32).reshape(-1, 3)[:min(count, cap)]]
            assert count == len(want), (what, count, len(want))
            if count <= cap:
                assert Counter(got) == Counter(want), what
            else:                                           # the first `cap` events stored, in no particular order
                assert len(got) == cap and not (Counter(got) - Counter(want)), what


def run_rollout_row(ag, torch, oracle, ops, row, idx, grid=None):
    kernel, args, grid_name, engine, n, K, env_id0, opts = row
    o = parse_opts(opts)
    g = grid or Grid.named(ag, torch, oracle, grid_name)
    case = RolloutCase(oracle, g, n, K, env_id0, 7919 * idx + 17, o)
    case.engine = engine
    ref = case.reference(oracle)
    rec, fin, stats = ref
    # the reach-boundary envs: reached at step 0 by the oracle exactly when placed inside
    for lo, inside in case.probes:
        if case.flags0[lo] == 0:
            assert bool(rec["flags"][0, lo] & 2) == inside, (lo, inside)
    n_events = int(((rec["flags"] != 0) | (rec["reward"] != 0)).sum())
    cap = {None: 0, "ev": n_events + 5, "evshort": n_events // 2}[o["events"]]
    if o["events"] == "evshort":
        assert n_events >= 2, n_events
    case.device(ag, torch, ops, cap)
    got = launched_kernels(torch, lambda: case.launch(ops))
    assert got == [(kernel, args)], got
    case.compare(oracle, ref, "%s%s on %s" % (kernel, args, grid_name))
    assert stats[oracle.ST_ENV_STEPS] == n * K
    return case, stats


def _row_id(r):
    kernel, args, grid, engine, n, K, env_id0, opts = r
    return "%s<%s>-%s-n%d-K%d-id%d%s" % (kernel, ",".join(map(str, args)), grid, n, K, env_id0,
                                        ("-" + "-".join(opts.split())) if opts else "")


@pytest.mark.parametrize("idx", range(len(ROLLOUT_ROWS)), ids=[_row_id(r) for r in ROLLOUT_ROWS])
def test_rollout_form_vs_oracle(ag, torch_, oracle, ops, idx):
    row = ROLLOUT_ROWS[idx]
    case, stats = run_rollout_row(ag, torch_, oracle, ops, row, idx)
    o = case.o
    if row[2] == "dense31" and not o["R"]:
        assert stats[oracle.ST_STUCK_RESETS] > 0                       # max_reset_tries exhausted
    if o["R"] and o["R"] <= 3 and row[2] == "dense31":
        assert stats[oracle.ST_STUCK_RESETS] > 0                       # the candidate list ran out


def test_rollout_rows_reach_every_edge(oracle):
    """the table's rows together take every edge case: sizes, step counts around the action ring (AG_RING = 4), entry
    ids, sticky entry, huge joints, short candidate lists, both event sinks, and every flag combination per engine"""
    ns = {r[4] for r in ROLLOUT_ROWS}
    assert {1, 31, 257, 4096} <= ns and any(n % 32 == 0 and n < 4096 for n in ns)
    assert set(range(1, 6)) <= {r[5] for r in ROLLOUT_ROWS} and max(r[5] for r in ROLLOUT_ROWS) >= 17
    assert {0, 1000, 256, 512, 768} <= {r[6] for r in ROLLOUT_ROWS}
    toks = Counter(t for r in ROLLOUT_ROWS for t in r[7].split())
    for t in ("sticky", "huge", "ev", "evshort", "hr2", "per_env", "joint", "long", "misal", "joints", "rec"):
        assert toks[t] > 0, t
    for e in (0, 2):
        assert {r[1][2:5] for r in ROLLOUT_ROWS if r[0] == "k_rollout" and r[1][0] == e} == \
               {(a, b, c) for a in (0, 1) for b in (0, 1) for c in (0, 1)}


# ------------------------------------------------------------------ k_step, k_reset, k_collision

def first_hit_engine(e):
    return 0 if e == 1 else e            # first_hit: the FAST engine runs the EXACT kernel


STEP_CASES = [(e, f32, wf) for e in ENGINE_ID for f32 in (False, True) for wf in (False, True)]


@pytest.mark.parametrize("engine,f32,wf", STEP_CASES,
                         ids=["%s-%s-%s" % (e, "f32" if f else "f64", "fh" if w else "nofh") for e, f, w in STEP_CASES])
def test_step_kernel_vs_oracle(ag, torch_, oracle, ops, engine, f32, wf):
    """k_step<engine, float32 actions, first_hit> with ee / dist and per-env targets against oracle.step_batch per
    (target block, grid), three steps from sticky entry state"""
    torch = torch_
    grid = Grid.named(ag, torch, oracle, "het64_epg100" if engine != "brute" else "rand31")
    n, T, env_id0 = (4096 if engine != "brute" else 257), 3, 1000
    rng = np.random.default_rng(100 + 4 * ENGINE_ID[engine] + 2 * f32 + wf)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    j1[::7] += 2.0 ** 20 * np.where(np.arange(0, n, 7) % 2 == 0, 1.0, 2.0)
    acts = (rng.random((T, n, 2)) - 0.5) * 0.3
    if f32:
        acts = acts.astype(np.float32)
    fl = np.where(rng.random(n) < 0.2, rng.integers(1, 4, n), 0).astype(np.uint8)
    rw = np.where(fl != 0, -1000.0, 0.0)
    fl0 = fl.copy()
    base = make_params(oracle)
    edges = np.linspace(0, n, N_BLOCKS + 1).astype(int)
    blocks = list(zip(edges[:-1].tolist(), edges[1:].tolist()))
    ee0 = fk_ref(oracle, j1 + acts[0, :, 0].astype(np.float64), j2 + acts[0, :, 1].astype(np.float64))
    tg, probes = boundary_targets(oracle, ee0, blocks, base, grid.E)
    params = [make_params(oracle, t) for t in tg]
    targets = np.zeros((n, 2))
    for (lo, hi), t in zip(blocks, tg):
        targets[lo:hi] = t
    gi = grid.of_env(env_id0 + np.arange(n))
    dv = dict(j1=torch.as_tensor(j1, device="cuda").clone(), j2=torch.as_tensor(j2, device="cuda").clone(),
              reward=torch.as_tensor(rw.astype(np.float32), device="cuda").clone(),
              flags=torch.as_tensor(fl, device="cuda").clone())
    ee, dist = (torch.zeros(n, 2, dtype=torch.float64, device="cuda") for _ in range(2))
    fh = torch.zeros(n, dtype=torch.int32, device="cuda") if wf else None
    stats = torch.zeros(len(ag.STAT_NAMES), dtype=torch.int64, device="cuda")
    tgt = torch.as_tensor(targets, device="cuda")
    P, GA = pack(ag, ops, base), ops.grid_args(grid.dg)
    want_stats = np.zeros(oracle.ST_COUNT, dtype=np.int64)
    for t in range(T):
        a = torch.as_tensor(acts[t], device="cuda")
        got = launched_kernels(torch, lambda: ops.step(P, *GA, dv["j1"], dv["j2"], a, dv["reward"], dv["flags"], ee, dist,
                                                       fh, stats, tgt, env_id0, ENGINE_ID[engine]))
        assert got == [("k_step", (first_hit_engine(ENGINE_ID[engine]) if wf else ENGINE_ID[engine], int(f32), int(wf)))], got
        w_ee, w_dist, w_fh = np.zeros((n, 2)), np.zeros((n, 2)), np.full(n, -1, np.int32)
        for (lo, hi), p in zip(blocks, params):
            for g in np.unique(gi[lo:hi]):
                idx = lo + np.flatnonzero(gi[lo:hi] == g)
                b1, b2, brw, bfl = j1[idx], j2[idx], rw[idx], fl[idx]
                res = oracle.step_batch(b1, b2, acts[t][idx].astype(np.float64), brw, bfl, grid.squares[g], grid.cells[g],
                                        params=p)
                j1[idx], j2[idx], rw[idx], fl[idx] = b1, b2, brw, bfl
                w_ee[idx], w_dist[idx], w_fh[idx] = res["ee"], res["dist"], res["first_hit"]
                want_stats[oracle.ST_AXIS_ALIGNED] += res["axis_aligned"]
        want_stats[oracle.ST_ENV_STEPS] += n
        if t == 0:
            for lo, inside in probes:
                if fl0[lo] == 0:
                    assert bool(fl[lo] & 2) == inside, (lo, inside)
        f = lambda x: x.cpu().numpy()
        what = (engine, f32, wf, t)
        assert np.array_equal(f(dv["j1"]), j1) and np.array_equal(f(dv["j2"]), j2), what
        assert np.array_equal(f(dv["flags"]), fl) and np.array_equal(f(dv["reward"]), rw.astype(np.float32)), what
        if wf:
            assert np.array_equal(f(fh), w_fh), what
        for got_g, want_g in ((f(ee), w_ee), (f(dist), w_dist)):
            err = np.abs(got_g - want_g)
            assert np.all(err <= TOL * np.maximum(np.abs(want_g), 1e-3)) and err.max() < 1e-14, (what, err.max())
        assert np.array_equal(f(stats), want_stats), (what, f(stats), want_stats)
    assert (fl & 1).any() and (fl & 2).any()


RESET_CASES = [(e, hr, m, c) for e in ENGINE_ID for hr in (False, True) for m in (False, True) for c in (False, True)]


def reset_reference(oracle, grid, j1, j2, rc, active, seed, env_id0, p, reset_u):
    """Scene.reset() / random_valid_pose() (scene_0.py:105-113,174-181) with the library's bound: candidates
    (u*pi)*2.0 from reset_u[e, rc] or Philox stream 1 keyed by (seed, global id, rc) while the pose collides, at most
    max_reset_tries of them and none past the end of reset_u; the last candidate stays when the draw gives up.
    -> number of envs that gave up"""
    gi = grid.of_env(env_id0 + np.arange(len(j1)))

    def colliding(idx):
        hit = np.zeros(idx.size, dtype=bool)
        for g in np.unique(gi[idx]):
            m = gi[idx] == g
            hit[m] = oracle.collision_batch(j1[idx[m]], j2[idx[m]], grid.squares[g], want_first_hit=False)[0] != 0
        return hit

    active = active[colliding(active)]
    stuck, tries = 0, 0
    while active.size:
        out = (rc[active] >= reset_u.shape[1]) if reset_u is not None else np.zeros(active.size, dtype=bool)
        if tries >= p.max_reset_tries:
            out[:] = True
        stuck += int(out.sum())
        active = active[~out]
        for e in active:
            u0, u1 = (reset_u[e, rc[e]] if reset_u is not None else oracle.philox_uniform2(seed, env_id0 + int(e), int(rc[e]), 1))
            j1[e], j2[e] = (u0 * np.pi) * 2.0, (u1 * np.pi) * 2.0
        rc[active] += 1
        tries += 1
        active = active[colliding(active)]
    return stuck


@pytest.mark.parametrize("engine,hr,masked,clear", RESET_CASES,
                         ids=["%s-%s-%s-%s" % (e, "reset_u" if h else "philox", "mask" if m else "all",
                                               "clear" if c else "keep") for e, h, m, c in RESET_CASES])
def test_reset_kernel_vs_reference(ag, torch_, oracle, ops, engine, hr, masked, clear):
    """k_reset<engine, reset_u> against the reset rule, with candidate lists that run out (entry reset_ctr up to R) and
    draws that exhaust max_reset_tries on a dense grid"""
    torch = torch_
    grid = Grid.named(ag, torch, oracle, "dense31" if engine == "brute" else "het64_epg100")
    n, R, env_id0, seed = (4096 if engine != "brute" else 257), 5, 1000, 31
    rng = np.random.default_rng(200 + 8 * ENGINE_ID[engine] + 4 * hr + 2 * masked + clear)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    rc = rng.integers(0, R + 1, n).astype(np.uint32)
    reset_u = rng.random((n, R, 2)) if hr else None
    mask = (rng.random(n) < 0.7).astype(np.uint8) if masked else None
    fl = rng.integers(0, 4, n).astype(np.uint8)
    rw = np.where(fl != 0, -1000.0, 0.0).astype(np.float32)
    p = make_params(oracle, tries=3)
    dv = [torch.as_tensor(x, device="cuda").clone() for x in (j1, j2, rw, fl, rc.view(np.int32))]
    stats = torch.zeros(len(ag.STAT_NAMES), dtype=torch.int64, device="cuda")
    m_t = None if mask is None else torch.as_tensor(mask, device="cuda")
    ru_t = None if reset_u is None else torch.as_tensor(reset_u, device="cuda")
    got = launched_kernels(torch, lambda: ops.reset(pack(ag, ops, p), *ops.grid_args(grid.dg), *dv, m_t, ru_t, stats, seed,
                                                    clear, env_id0, ENGINE_ID[engine]))
    assert got == [("k_reset", (ENGINE_ID[engine], int(hr)))], got
    active = np.flatnonzero(mask != 0) if masked else np.arange(n)
    stuck = reset_reference(oracle, grid, j1, j2, rc, active, seed, env_id0, p, reset_u)
    if clear:
        rw[active], fl[active] = 0.0, 0
    f = lambda x: x.cpu().numpy()
    assert np.array_equal(f(dv[0]), j1) and np.array_equal(f(dv[1]), j2)
    assert np.array_equal(f(dv[2]), rw) and np.array_equal(f(dv[3]), fl)
    assert np.array_equal(f(dv[4]).view(np.uint32), rc)
    want = np.zeros(oracle.ST_COUNT, dtype=np.int64)
    want[oracle.ST_STUCK_RESETS] = stuck
    assert np.array_equal(f(stats), want), (f(stats), want)
    assert stuck > 0 and int((rc != 0).sum()) > 0


COLLISION_CASES = [(e, wf) for e in ENGINE_ID for wf in (False, True)]


@pytest.mark.parametrize("engine,wf", COLLISION_CASES, ids=["%s-%s" % (e, "fh" if w else "nofh") for e, w in COLLISION_CASES])
@pytest.mark.parametrize("grid_name", ["scene0", "het64_epg100", "edge9_e1"])
def test_collision_kernel_vs_oracle(ag, torch_, oracle, ops, engine, wf, grid_name):
    """k_collision<engine, first_hit> against oracle.collision_batch per grid"""
    torch = torch_
    grid = Grid.named(ag, torch, oracle, grid_name)
    n, env_id0 = (4096 if engine != "brute" else 257), 1000
    rng = np.random.default_rng(300 + 2 * ENGINE_ID[engine] + wf)
    j1, j2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n)
    j1[::9] += 2.0 ** 21
    hit = torch.zeros(n, dtype=torch.uint8, device="cuda")
    fh = torch.zeros(n, dtype=torch.int32, device="cuda") if wf else None
    a, b = torch.as_tensor(j1, device="cuda"), torch.as_tensor(j2, device="cuda")
    got = launched_kernels(torch, lambda: ops.collision_check(pack(ag, ops, make_params(oracle)), *ops.grid_args(grid.dg),
                                                              a, b, hit, fh, env_id0, ENGINE_ID[engine]))
    assert got == [("k_collision", (first_hit_engine(ENGINE_ID[engine]) if wf else ENGINE_ID[engine], int(wf)))], got
    gi = grid.of_env(env_id0 + np.arange(n))
    w_hit, w_fh = np.zeros(n, np.uint8), np.full(n, -1, np.int32)
    for g in np.unique(gi):
        idx = np.flatnonzero(gi == g)
        h, f_, _ = oracle.collision_batch(j1[idx], j2[idx], grid.squares[g], grid.cells[g])
        w_hit[idx], w_fh[idx] = h, f_
    assert np.array_equal(hit.cpu().numpy(), w_hit)
    if wf:
        assert np.array_equal(fh.cpu().numpy(), w_fh)
    assert 0 < int(w_hit.sum()) < n


# ------------------------------------------------------------------ coverage of the library

def library_instantiations(ag):
    import os
    import subprocess
    from abstract_gym_b200 import build as ag_build
    cuobjdump = os.path.join(os.path.dirname(ag_build.find_nvcc()), "cuobjdump")
    out = subprocess.run([cuobjdump, "-sass", ag_build.LIB], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                         check=True).stdout
    return [k for k in (kernel_of(m) for m in re.findall(r"Function : (\S+)", out)) if k is not None]


def named_instantiations():
    named = {(r[0], r[1]) for r in ROLLOUT_ROWS}
    named |= {("k_step", (first_hit_engine(ENGINE_ID[e]) if w else ENGINE_ID[e], int(f), int(w))) for e, f, w in STEP_CASES}
    named |= {("k_reset", (ENGINE_ID[e], int(h))) for e, h, _, _ in RESET_CASES}
    named |= {("k_collision", (first_hit_engine(ENGINE_ID[e]) if w else ENGINE_ID[e], int(w))) for e, w in COLLISION_CASES}
    return named


def test_rows_cover_every_instantiation(ag):
    """the instantiations of the six families in the release library are exactly those the rows name"""
    lib = library_instantiations(ag)
    assert len(lib) == len(set(lib))
    assert Counter(f for f, _ in lib) == {"k_rollout": 40, "k_rollout_async": 8, "k_rollout_lut": 12, "k_step": 10,
                                          "k_reset": 6, "k_collision": 5}
    named = named_instantiations()
    assert set(lib) == named, (sorted(set(lib) - named), sorted(named - set(lib)))
    print("%d instantiations, each named by a row" % len(lib))


# ------------------------------------------------------------------ capture and the map cache

LUT_CM = ("k_rollout_lut", (1, 1, 0, 1))             # actions, records, general squares, the map
LUT_TABLE = ("k_rollout_lut", (1, 1, 0, 0))          # the same without the map: the table-arm form


def prepared_case(ag, torch, oracle, ops, grid, seed, n=4096, K=6, opts="ha rec"):
    case = RolloutCase(oracle, grid, n, K, 0, seed, parse_opts(opts))
    case.engine = "fast"
    ref = case.reference(oracle)
    case.device(ag, torch, ops)
    return case, ref


def captured(torch, ops, case, dot):
    """case's rollout captured in a CUDA graph -> (graph, launches counted while capturing, the (family, args) of the
    graph's kernel nodes of FAMILIES, read from its DOT dump at path `dot`)"""
    import abstract_gym_b200 as ag
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(keep_graph=True)          # the captured cudaGraph_t stays for debug_dump
    before = ag.launch_count()
    with torch.cuda.graph(g):
        case.launch(ops)
    counted = ag.launch_count() - before
    g.debug_dump(str(dot))
    g.instantiate()
    torch.cuda.synchronize()
    with open(dot) as f:
        text = html.unescape(f.read()).replace("\\<", "<").replace("\\>", ">")
    nodes = {k for k in (kernel_of(line) for line in text.splitlines()) if k is not None}
    return g, counted, nodes


def six_cells(seed):
    rng = np.random.default_rng(seed)
    free = np.flatnonzero(clear_base(np.ones((9, 9), dtype=np.uint8), 1.6).ravel())
    occ = np.zeros((1, 9, 9), dtype=np.uint8)
    occ[0].ravel()[rng.choice(free, 6, replace=False)] = 1
    return occ


def test_capture_takes_table_arm_form_until_the_map_is_cached(ag, torch_, oracle, ops, tmp_path):
    """a rollout captured on a grid that never ran uncaptured has no map entry: it takes the table-arm form (no map
    build in the graph) and equals the oracle; once an uncaptured launch has cached the map, a capture takes the map form"""
    torch = torch_
    warm, _ = prepared_case(ag, torch, oracle, ops, Grid(ag, torch, oracle, six_cells(50), 1.6, None), 1)
    warm.launch(ops)                                   # the kernels are loaded and their shared memory opted in
    torch.cuda.synchronize()
    grid = Grid(ag, torch, oracle, six_cells(51), 1.6, None)
    case, ref = prepared_case(ag, torch, oracle, ops, grid, 2)
    g, counted, nodes = captured(torch, ops, case, tmp_path / "uncached.dot")
    assert counted == 1 and nodes == {LUT_TABLE}, (counted, nodes)      # the rollout alone: no k_cspace_build
    g.replay()
    torch.cuda.synchronize()
    case.compare(oracle, ref, "captured, uncached")
    # an uncaptured launch caches the map; a capture from now on takes the map form
    case2, ref2 = prepared_case(ag, torch, oracle, ops, grid, 2)
    assert launched_kernels(torch, lambda: case2.launch(ops)) == [LUT_CM]
    case2.compare(oracle, ref2, "uncached, eager")
    case3, ref3 = prepared_case(ag, torch, oracle, ops, grid, 2)
    g3, counted, nodes = captured(torch, ops, case3, tmp_path / "cached.dot")
    assert counted == 2 and nodes == {LUT_CM}, (counted, nodes)         # k_cspace_build + the rollout
    g3.replay()
    torch.cuda.synchronize()
    case3.compare(oracle, ref3, "captured, cached")


def test_graph_replay_after_its_map_entry_passed_to_other_grids(ag, torch_, oracle, ops, tmp_path):
    """cycle more than 32 (grid, parameter) pairs twice, so that every entry is evicted and handed on, then replay a graph
    captured with the map form: its map build finds another grid's map in the buffer, rebuilds, and the replay equals
    the oracle.  That the graph's entry did change hands is checked first: a capture on the graph's grid and parameters
    finds no entry (a capture never creates one) and takes the table-arm form"""
    torch = torch_
    grid = Grid(ag, torch, oracle, six_cells(60), 1.6, None)
    eager, _ = prepared_case(ag, torch, oracle, ops, grid, 3)
    eager.launch(ops)
    case, ref = prepared_case(ag, torch, oracle, ops, grid, 3)
    g, counted, nodes = captured(torch, ops, case, tmp_path / "graph.dot")
    assert counted == 2 and nodes == {LUT_CM}, (counted, nodes)
    grids = [Grid(ag, torch, oracle, six_cells(61 + i), 1.6, None) for i in range(5)]
    for rnd in range(2):
        for i in range(40):                            # 5 grids x 8 targets: 40 distinct entries
            c, r = prepared_case(ag, torch, oracle, ops, grids[i % 5], 100 + i, n=64, K=3, opts="ha rec")
            c.launch(ops)
            c.compare(oracle, r, "cycle %d pair %d" % (rnd, i))
    probe, _ = prepared_case(ag, torch, oracle, ops, grid, 3)
    _, counted, nodes = captured(torch, ops, probe, tmp_path / "probe.dot")
    assert counted == 1 and nodes == {LUT_TABLE}, (counted, nodes)      # the entry is gone: no map build, no map
    g.replay()
    torch.cuda.synchronize()
    case.compare(oracle, ref, "replay after eviction")


def test_map_follows_a_grid_rewritten_in_place(ag, torch_, oracle, ops):
    """a DeviceGrid whose bits are rewritten in place (same pointers, same parameters, no more cells than promised):
    the next rollout follows the new content"""
    torch = torch_
    grid = Grid(ag, torch, oracle, six_cells(70), 1.6, None)
    ptrs = (grid.dg.bits.data_ptr(), grid.dg.min_x.data_ptr())
    case, ref = prepared_case(ag, torch, oracle, ops, grid, 4, K=10)
    assert launched_kernels(torch, lambda: case.launch(ops)) == [LUT_CM]
    case.compare(oracle, ref, "before the rewrite")
    new = six_cells(71)
    packed = ag.DeviceGrid.from_device_matrices(torch.as_tensor(new, device="cuda"), 1.6)
    grid.dg.bits.copy_(packed.bits)
    grid.occ, grid.squares = new, [oracle.grid_squares(new[0], 1.6)[0]]
    assert np.array_equal(grid.dg.unpack(), new) and (grid.dg.bits.data_ptr(), grid.dg.min_x.data_ptr()) == ptrs
    case, ref = prepared_case(ag, torch, oracle, ops, grid, 4, K=10)       # the same joints, actions and target
    assert launched_kernels(torch, lambda: case.launch(ops)) == [LUT_CM]
    case.compare(oracle, ref, "after the rewrite")
    assert ref[2][oracle.ST_COLLISIONS] > 0


def test_map_of_a_new_grid_at_a_recycled_address(ag, torch_, oracle, ops):
    """a grid freed and a new one of the same size whose device arrays sit at the freed addresses (what the caching
    allocator hands out after a free; forced here by building the new DeviceGrid on the freed grid's storage): the same
    pointers and parameters as the stale cache entry, new content, and more cells (6) than the old grid promised (3).
    The rollout on the new grid equals the oracle for the new grid"""
    torch = torch_
    grid = Grid(ag, torch, oracle, cells_occ(9, SCENE0_CELLS), 1.6, None)
    case, ref = prepared_case(ag, torch, oracle, ops, grid, 5, K=10)
    assert launched_kernels(torch, lambda: case.launch(ops)) == [LUT_CM]
    case.compare(oracle, ref, "old grid")
    storage = (grid.dg.bits, grid.dg.min_x, grid.dg.min_y)
    ptrs = tuple(t.data_ptr() for t in storage)
    del case, grid
    gc.collect()
    grid = Grid(ag, torch, oracle, six_cells(80), 1.6, None)
    dg = grid.dg
    for old, new in zip(storage, (dg.bits, dg.min_x, dg.min_y)):
        old.copy_(new)
    dg.bits, dg.min_x, dg.min_y = storage
    del storage
    assert tuple(t.data_ptr() for t in (dg.bits, dg.min_x, dg.min_y)) == ptrs and dg.max_occupied == 6
    assert np.array_equal(dg.unpack(), grid.occ)
    case, ref = prepared_case(ag, torch, oracle, ops, grid, 5, K=10)
    assert launched_kernels(torch, lambda: case.launch(ops)) == [LUT_CM]
    case.compare(oracle, ref, "new grid at the old addresses")
    assert ref[2][oracle.ST_COLLISIONS] > 0


# ------------------------------------------------------------------ element counts of the ops

def test_ops_check_element_counts(ag, torch_, oracle, ops):
    """every state and output tensor of the rollout, step, reset and collision_check ops is checked for its element
    count before anything launches"""
    torch = torch_
    grid = Grid.named(ag, torch, oracle, "scene0")
    n, K = 64, 2
    case = RolloutCase(oracle, grid, n, K, 0, 6, parse_opts("ha hr3 rec per_env ev"))
    case.engine = "exact"
    case.device(ag, torch, ops, 16)
    P, GA, t = case.P, case.GA, case.t
    Z = lambda m, dt: torch.zeros(m, dtype=dt, device="cuda")
    st = dict(j1=t["j1"], j2=t["j2"], reward=t["reward"], flags=t["flags"], reset_ctr=t["reset_ctr"],
              actions=torch.zeros(n, 2, dtype=torch.float64, device="cuda"), ee=Z(2 * n, torch.float64),
              dist=Z(2 * n, torch.float64), first_hit=Z(n, torch.int32), stats=t["stats"], targets=t["targets"],
              mask=Z(n, torch.uint8) + 1, hit=Z(n, torch.uint8))
    calls = {
        "rollout": (case.t, lambda d: case.launch(ops),
                    dict(j2=n, reward=n, flags=n, step_ctr=n, reset_ctr=n, ep_len=n, stats=len(ag.STAT_NAMES), diag=3,
                         targets=2 * n, event_count=1)),
        "step": (st, lambda d: ops.step(P, *GA, d["j1"], d["j2"], d["actions"], d["reward"], d["flags"], d["ee"], d["dist"],
                                        d["first_hit"], d["stats"], d["targets"], 0, 0),
                 dict(j2=n, reward=n, flags=n, ee=2 * n, dist=2 * n, first_hit=n, stats=len(ag.STAT_NAMES), targets=2 * n)),
        "reset": (st, lambda d: ops.reset(P, *GA, d["j1"], d["j2"], d["reward"], d["flags"], d["reset_ctr"], d["mask"], None,
                                          d["stats"], 3, True, 0, 0),
                  dict(j2=n, reward=n, flags=n, reset_ctr=n, mask=n, stats=len(ag.STAT_NAMES))),
        "collision_check": (st, lambda d: ops.collision_check(P, *GA, d["j1"], d["j2"], d["hit"], d["first_hit"], 0, 0),
                            dict(j2=n, hit=n, first_hit=n)),
    }
    for op, (d, call, sizes) in calls.items():
        for name, count in sizes.items():
            good = d[name]
            assert good.numel() == count, (op, name)
            d[name] = good.flatten()[:count - 1].clone()
            before = ag.launch_count()
            with pytest.raises(RuntimeError):
                call(d)
            torch.cuda.synchronize()
            assert ag.launch_count() == before, (op, name)
            d[name] = good
        before = ag.launch_count()
        call(d)
        torch.cuda.synchronize()
        assert ag.launch_count() == before + 1, op
