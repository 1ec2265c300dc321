"""scene_0: the reference's `Scene` (scenario/scene_0.py:13-181) and `BatchedScene`, the same
step / reset / collision_check / rollout semantics for N independent environments in HBM.

Everything that computes (FK, segment-vs-grid collision, reach test, reward/flag logic, reset
rejection sampling, the fused K-step rollout) is CUDA in libabstract_gym_b200.so; this module is
argument plumbing.  Visualisation (render / occ_to_patch, scene_0.py:41-58,135-172) is out of
scope and raises.
"""
import ctypes as C
import math

import numpy as np
import torch

from .. import _lib
from .._device import as_f64, ptr, require_cuda, stream_ptr
from ..environment.occupancy_grid import BatchedOccupancyGrid, DeviceGrid, OccupancyGrid
from ..robot.two_joint_robot import BatchedTwoJointRobot, TwoJointRobot
from ..utils.geometry import Point
from ..sharding import StatsReducer


def _engine(e):
    if isinstance(e, str):
        return _lib.ENGINES[e]
    return int(e)


def _pack_words(img):
    """bool [n, b1, b2] -> int32 words [n, b1, ceil(b2/32)] in the layout of cspace_occupancy(packed=True): pose (i, j)
    is bit j % 32 of word j // 32, padding bits 0"""
    n, b1, b2 = img.shape
    w = (b2 + 31) // 32
    pad = torch.zeros(n, b1, w * 32, dtype=torch.uint8, device=img.device)
    pad[..., :b2] = img
    # one byte per 8 poses (distinct bits: the sum is an OR), then 4 little-endian bytes per word: 2 bytes of
    # temporaries per pose
    shifts = torch.arange(8, dtype=torch.uint8, device=img.device)
    octets = (pad.view(n, b1, w * 4, 8) << shifts).sum(dim=-1, dtype=torch.uint8)
    return octets.view(torch.int32)


class BatchedScene:
    """N environments sharing one grid (or one grid per block of `envs_per_grid` envs).

    State (structure of arrays, all CUDA tensors of length N):
        robot.joint_1, robot.joint_2  float64   joint angles
        step_reward                   float32   sticky reward (0, -1000, 10000)
        flags                         uint8     bit0 collision_status, bit1 done (sticky)
        step_ctr, reset_ctr, ep_len   int32     Philox draw counters / current episode length
    `env_id0` is the global id of env 0: Philox streams and grid selection use global ids, so a
    rollout sharded over ranks equals the unsharded one (tests/test_sharding.py).
    """

    def __init__(self, robot, env, target_c=None, engine="fast", seed=0, env_id0=0, max_reset_tries=64):
        self.robot = robot
        self.device = robot.device
        self.n = len(robot)
        self.env = env
        self.grid = env if isinstance(env, DeviceGrid) else env.device_grid(self.device)
        self.target_c = target_c if target_c is not None else Point(-0.2, -0.3)   # scene_0.py:17
        self.target_j = np.array([1.1, -0.2])                                      # scene_0.py:30
        self.choose_j_tar = False                                                  # scene_0.py:31
        self.engine = _engine(engine)
        self.seed = int(seed)
        self.env_id0 = int(env_id0)
        self.max_reset_tries = int(max_reset_tries)
        dev, n = self.device, self.n
        self.step_reward = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flags = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.step_ctr = torch.zeros(n, dtype=torch.int32, device=dev)
        self.reset_ctr = torch.zeros(n, dtype=torch.int32, device=dev)
        self.ep_len = torch.zeros(n, dtype=torch.int32, device=dev)
        self.stats = torch.zeros(_lib.ST_COUNT, dtype=torch.int64, device=dev)
        self.diag = torch.zeros(len(_lib.DIAG_NAMES), dtype=torch.int64, device=dev)   # FAST-filter diagnostics
        self._pipelines = {}
        self._reducer = StatsReducer()
        self._lib = _lib.load()

    # ---- views with the reference's attribute names ---------------------------------------------
    @property
    def collision_status(self):
        return (self.flags & _lib.FLAG_COLLISION) != 0

    @property
    def done(self):
        return (self.flags & _lib.FLAG_DONE) != 0

    def params(self) -> _lib.Params:
        p = _lib.default_params()
        p.link_1, p.link_2 = float(self.robot.link_1), float(self.robot.link_2)
        p.target_x, p.target_y = float(self.target_c.x), float(self.target_c.y)
        p.target_j1, p.target_j2 = float(self.target_j[0]), float(self.target_j[1])
        p.choose_j_tar = 1 if self.choose_j_tar else 0
        p.max_reset_tries = self.max_reset_tries
        return p

    def stats_dict(self):
        return dict(zip(_lib.STAT_NAMES, self.stats.tolist()))

    def diag_dict(self):
        """FAST-engine diagnostics accumulated by rollout(): float64 re-evaluations, cold-section visits, warp exits."""
        return dict(zip(_lib.DIAG_NAMES, self.diag.tolist()))

    def all_reduce_stats(self, wait=True):
        """Sum the episode counters over ranks (the only collective on this path, SURVEY 8e): one
        int64[8] all-reduce of a snapshot of this rank's cumulative counters, started asynchronously
        so that it overlaps the next rollout launch.  Returns the global totals (wait=True) or
        None (wait=False; fetch them later with global_stats())."""
        self._reducer.submit(self.stats)
        return self._reducer.result() if wait else None

    def global_stats(self):
        """Global cumulative counters of the newest all_reduce_stats() call."""
        return self._reducer.result()

    # ---- checkpoint / resume (SURVEY 8f.4) --------------------------------------------------------
    _STATE = ("step_reward", "flags", "step_ctr", "reset_ctr", "ep_len", "stats", "diag")

    def state_dict(self):
        """Everything a resumed run needs to continue bit for bit: joint angles, sticky reward / flags, the
        Philox draw counters, episode lengths and counters, seed and global env offset (host copies)."""
        d = {k: getattr(self, k).detach().cpu().clone() for k in self._STATE}
        d["joint_1"], d["joint_2"] = self.robot.joint_1.detach().cpu().clone(), self.robot.joint_2.detach().cpu().clone()
        d["meta"] = dict(seed=self.seed, env_id0=self.env_id0, n=self.n, max_reset_tries=self.max_reset_tries,
                         link_1=float(self.robot.link_1), link_2=float(self.robot.link_2),
                         target_c=(float(self.target_c.x), float(self.target_c.y)),
                         target_j=[float(self.target_j[0]), float(self.target_j[1])], choose_j_tar=bool(self.choose_j_tar))
        return d

    def load_state_dict(self, d):
        m = d["meta"]
        if int(m["n"]) != self.n:
            raise ValueError("checkpoint holds %d envs, this scene %d" % (m["n"], self.n))
        for k in self._STATE:
            getattr(self, k).copy_(d[k])
        self.robot.joint_1.copy_(d["joint_1"]); self.robot.joint_2.copy_(d["joint_2"])
        self.seed, self.env_id0, self.max_reset_tries = int(m["seed"]), int(m["env_id0"]), int(m["max_reset_tries"])
        self.robot.link_1, self.robot.link_2 = m["link_1"], m["link_2"]
        self.target_c = Point(*m["target_c"])
        self.target_j = np.array(m["target_j"])
        self.choose_j_tar = bool(m["choose_j_tar"])

    # ---- K2 ------------------------------------------------------------------------------------
    def collision_check(self, first_hit=False, engine=None):
        """scene_0.py:60-76 for every env -> bool [N] (and int32 [N] min hit cell index, -1 if none)."""
        hit = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        fh = torch.empty(self.n, dtype=torch.int32, device=self.device) if first_hit else None
        g = self.grid.c_struct()
        _lib.check(self._lib.ag_collision_check(self.params(), g, ptr(self.robot.joint_1), ptr(self.robot.joint_2),
                                                ptr(hit), ptr(fh), self.n, self.env_id0,
                                                self.engine if engine is None else _engine(engine),
                                                stream_ptr(self.device)), "ag_collision_check")
        return (hit != 0, fh) if first_hit else hit != 0

    def check_motion(self, goal, start=None, steps=100, first_hit=False, last_free=False, engine=None):
        """robot/two_joint_robot.py:49-62 move_to_joint_pose() with collision_check() (scene_0.py:60-76) at every
        intermediate pose, for M motions; nothing is moved.  Motion i goes from start[i] (default: the current joints,
        M = N) to goal[i] in steps[i] increments, pose_k = pose_{k-1} + (1/steps)*(goal - start), and stops at its
        first colliding pose; the start pose is not checked.  Motion i uses the grid of env i.
        goal, start: [M,2] float64; steps: int or int32 [M].
        Returns first_collision int32 [M]: the smallest colliding k, -1 if the motion is free, -2 if steps < 1; with
        first_hit / last_free also a dict: first_hit int32 [M] (min hit cell index at that pose, -1 if none) and
        last_free float64 [M,2] (the last pose before the first collision: RRT's "steer until blocked")."""
        if start is None:
            j1, j2 = self.robot.joint_1, self.robot.joint_2
        else:
            st = as_f64(start, self.device).reshape(-1, 2)
            j1, j2 = st[:, 0].contiguous(), st[:, 1].contiguous()
        m = j1.numel()
        goal = as_f64(goal, self.device).reshape(m, 2).contiguous()
        if isinstance(steps, torch.Tensor):
            if steps.dtype != torch.int32 or steps.numel() != m:
                raise ValueError("steps must be an int or an int32 tensor with one entry per motion")
            steps = steps.to(self.device).reshape(m).contiguous()
        else:
            steps = torch.full((m,), int(steps), dtype=torch.int32, device=self.device)
        fc = torch.empty(m, dtype=torch.int32, device=self.device)
        fh = torch.empty(m, dtype=torch.int32, device=self.device) if first_hit else None
        lf = torch.empty(m, 2, dtype=torch.float64, device=self.device) if last_free else None
        g = self.grid.c_struct()
        _lib.check(self._lib.ag_check_motion(self.params(), g, ptr(j1), ptr(j2), ptr(goal), ptr(steps), ptr(fc), ptr(fh),
                                             ptr(lf), m, self.env_id0, self.engine if engine is None else _engine(engine),
                                             stream_ptr(self.device)), "ag_check_motion")
        if first_hit or last_free:
            return fc, dict(first_hit=fh, last_free=lf)
        return fc

    def cspace_occupancy(self, b1, b2=None, lo=(0.0, 0.0), step=None, packed=False, free_count=False, engine=None):
        """collision_check() (scene_0.py:60-76) at every pose of a b1 x b2 lattice of joint angles, for every grid of the
        scene: the exact obstacle image of the configuration-space torus.  Nothing is moved.
        Pose (i, j) = (lo[0] + i * step[0], lo[1] + j * step[1]) in float64; its entry is True exactly when
        collision_check with the same engine says that pose collides on that grid.  Defaults: b2 = b1, step = 2 pi / b
        per axis, so the lattice covers the whole torus from 0.
        Returns bool [n_grids, b1, b2], or with packed=True the int32 words [n_grids, b1, ceil(b2/32)] (pose (i, j) is bit
        j % 32 of word j // 32, padding bits 0); with free_count=True also int64 [n_grids], the collision-free poses."""
        b1 = int(b1)
        b2 = b1 if b2 is None else int(b2)
        if b1 < 1 or b2 < 1:
            raise ValueError("the lattice needs b1, b2 >= 1, got %d x %d" % (b1, b2))
        lo1, lo2 = (float(v) for v in lo)
        st1, st2 = (2.0 * math.pi / b1, 2.0 * math.pi / b2) if step is None else (float(v) for v in step)
        n_grids = int(self.grid.n_grids)
        words = torch.empty(n_grids, b1, (b2 + 31) // 32, dtype=torch.int32, device=self.device)
        fc = torch.empty(n_grids, dtype=torch.int64, device=self.device) if free_count else None
        g = self.grid.c_struct()
        _lib.check(self._lib.ag_cspace_occupancy(self.params(), g, lo1, st1, b1, lo2, st2, b2, ptr(words), ptr(fc),
                                                 self.engine if engine is None else _engine(engine), stream_ptr(self.device)),
                   "ag_cspace_occupancy")
        if not packed:
            shifts = torch.arange(32, dtype=torch.int32, device=self.device)
            words = ((words.unsqueeze(-1) >> shifts) & 1).reshape(n_grids, b1, -1)[:, :, :b2] != 0
        return (words, fc) if free_count else words

    @staticmethod
    def _lattice(b1, b2, lo, step, wrap):
        """(lo1, lo2), (step1, step2), wrap bits of cspace_components' lattice (the defaults of cspace_occupancy; wrap=None:
        both axes when the default steps cover the torus, neither otherwise)"""
        lo1, lo2 = (float(v) for v in lo)
        st = (2.0 * math.pi / b1, 2.0 * math.pi / b2) if step is None else tuple(float(v) for v in step)
        w = (step is None, step is None) if wrap is None else tuple(bool(v) for v in wrap)
        if len(w) != 2:
            raise ValueError("wrap must be a pair of bools (joint_1, joint_2)")
        return (lo1, lo2), st, int(w[0]) | int(w[1]) << 1

    def cspace_components(self, b1, b2=None, lo=(0.0, 0.0), step=None, wrap=None, count=False, engine=None):
        """Connected components of the free poses of cspace_occupancy(b1, b2, lo, step, engine=engine), per grid: which
        lattice poses reach which through 4-neighbour steps between free poses.  wrap = (joint_1, joint_2) says which
        axes wrap (row b1-1 next to row 0, column b2-1 next to column 0); None: both when step is None (the default
        lattice covers the torus), neither otherwise.  Grids never connect to each other.
        Returns labels int32 [n_grids, b1, b2]: -1 for a colliding pose, else the smallest row-major index i * b2 + j of
        its component on that grid; with count=True also int64 [n_grids], the components of each grid.
        This is connectivity of the lattice image, not of continuous joint space: two adjacent free poses can have a
        colliding pose between them when the lattice is coarse for the grid's cells (check_motion checks such a step)."""
        b1 = int(b1)
        b2 = b1 if b2 is None else int(b2)
        if b1 < 1 or b2 < 1:
            raise ValueError("the lattice needs b1, b2 >= 1, got %d x %d" % (b1, b2))
        lo, st, w = self._lattice(b1, b2, lo, step, wrap)
        words = self.cspace_occupancy(b1, b2, lo=lo, step=st, packed=True, engine=engine)
        n_grids = words.shape[0]
        labels = torch.empty(n_grids, b1, b2, dtype=torch.int32, device=self.device)
        nc = torch.empty(n_grids, dtype=torch.int64, device=self.device) if count else None
        _lib.check(self._lib.ag_cspace_components(ptr(words), n_grids, b1, b2, w, ptr(labels), ptr(nc),
                                                  stream_ptr(self.device)), "ag_cspace_components")
        return (labels, nc) if count else labels

    @staticmethod
    def _nearest(q, b1, b2, lo, st, w):
        """the nearest lattice pose of each pose q [M, 2] float64: (k1, k2) int64 [M] and ok bool [M].  Per axis, in
        float64: k = floor((q - lo) / step + 0.5); on a wrapping axis k mod b; on any other, k outside [0, b) is not ok,
        and neither is a NaN or infinite q (k is 0 where not ok)"""
        ok = torch.ones(q.shape[0], dtype=torch.bool, device=q.device)
        idx = []
        for a, b in enumerate((b1, b2)):
            k = torch.floor((q[:, a] - lo[a]) / st[a] + 0.5)
            ok &= torch.isfinite(k)
            if w >> a & 1:
                k = torch.fmod(k, b)                          # exact for every integer-valued double
                k = torch.where(k < 0, k + b, k)
            else:
                ok &= (k >= 0) & (k < b)
            idx.append(torch.where(ok, k, 0.0).to(torch.int64))
        return idx[0], idx[1], ok

    def _snap(self, shape, joints, lo, step, wrap):
        """grid (the env rule of check_motion), nearest lattice pose (k1, k2) and ok of each of M poses, for a per-grid
        field of `shape` [n_grids, b1, b2] made with lo, step, wrap; joints None: the current joints (M = N)"""
        n_grids, b1, b2 = shape
        if n_grids != int(self.grid.n_grids):
            raise ValueError("the field holds %d grids, the scene %d" % (n_grids, int(self.grid.n_grids)))
        lo, st, w = self._lattice(b1, b2, lo, step, wrap)
        if joints is None:
            q = torch.stack([self.robot.joint_1, self.robot.joint_2], dim=1)
        else:
            q = as_f64(joints, self.device).reshape(-1, 2)
        env = self.env_id0 + torch.arange(q.shape[0], dtype=torch.int64, device=self.device)
        g = torch.div(env, int(self.grid.envs_per_grid), rounding_mode="floor") % n_grids
        return (g,) + self._nearest(q, b1, b2, lo, st, w)

    def _lookup(self, field, joints, lo, step, wrap):
        """the entry of a per-grid lattice field at the nearest lattice pose of each of M poses, -1 off the lattice"""
        g, k1, k2, ok = self._snap(field.shape, joints, lo, step, wrap)
        out = field.to(self.device)[g, k1, k2]
        return torch.where(ok, out, -1).to(torch.int32)

    def cspace_component_of(self, labels, joints=None, lo=(0.0, 0.0), step=None, wrap=None):
        """The label (cspace_components) at the nearest lattice pose of each of M poses, on the grid of env m
        (((env_id0 + m) // envs_per_grid) % n_grids, as check_motion).  joints: [M, 2] float64 (default: the current
        joints, M = N); lo, step, wrap: those of the call that made `labels`.
        Per axis, in float64: k = floor((q - lo) / step + 0.5); on a wrapping axis k mod b, on any other k outside [0, b)
        gives -1, and so does a NaN or infinite q.  Returns int32 [M].
        Whether env i can reach pose t_i on the lattice: component_of(labels)[i] == component_of(labels, t)[i] >= 0."""
        return self._lookup(labels, joints, lo, step, wrap)

    def cspace_distance(self, b1, b2=None, goals=None, lo=(0.0, 0.0), step=None, wrap=None, max_dist=False, engine=None):
        """Steps to the goal from every lattice pose, per grid: the fewest 4-neighbour steps through free poses of
        cspace_occupancy(b1, b2, lo, step, engine=engine) to a free goal pose (a multi-source BFS on the lattice).  The
        lattice and wrap are those of cspace_components.
        goals: a bool [n_grids, b1, b2] goal image; or float64 joint poses [G, 2] (goals of every grid) or
        [n_grids, G, 2], each snapped to its nearest lattice pose by the rule of cspace_component_of (a NaN or
        off-lattice pose seeds nothing); or None: the scene's own task -- target_j when choose_j_tar is set, else the
        valid solutions (both elbows) of robot.inverse_kinematic(target_c, corrected=True).  A goal is the lattice pose
        nearest each such pose, not the box that check_target_reached accepts.  Goals on colliding poses seed nothing.
        Returns dist int32 [n_grids, b1, b2]: -1 colliding, -2 free but no goal in its component, else the steps to the
        nearest goal (0 at a goal); with max_dist=True also int32 [n_grids], the largest distance of each grid (-1 if
        none).  Like cspace_components this is the lattice image, not continuous joint space.  The call synchronises
        with the current stream (it reads convergence back), so it cannot be captured in a CUDA graph."""
        b1 = int(b1)
        b2 = b1 if b2 is None else int(b2)
        if b1 < 1 or b2 < 1:
            raise ValueError("the lattice needs b1, b2 >= 1, got %d x %d" % (b1, b2))
        lo, st, w = self._lattice(b1, b2, lo, step, wrap)
        words = self.cspace_occupancy(b1, b2, lo=lo, step=st, packed=True, engine=engine)
        n_grids = words.shape[0]
        goal_words = _pack_words(self._goal_image(goals, n_grids, b1, b2, lo, st, w))
        dist = torch.empty(n_grids, b1, b2, dtype=torch.int32, device=self.device)
        md = torch.empty(n_grids, dtype=torch.int32, device=self.device) if max_dist else None
        _lib.check(self._lib.ag_cspace_distance(ptr(words), ptr(goal_words), n_grids, b1, b2, w, ptr(dist), ptr(md),
                                                stream_ptr(self.device)), "ag_cspace_distance")
        return (dist, md) if max_dist else dist

    def _goal_image(self, goals, n_grids, b1, b2, lo, st, w):
        """bool [n_grids, b1, b2] goal image of cspace_distance's `goals` argument"""
        if isinstance(goals, torch.Tensor) and goals.dtype == torch.bool:
            if tuple(goals.shape) != (n_grids, b1, b2):
                raise ValueError("a goal image must be [n_grids, b1, b2] = %s, got %s" % ((n_grids, b1, b2), tuple(goals.shape)))
            return goals.to(self.device)
        if goals is None:
            if self.choose_j_tar:
                goals = torch.tensor([[float(self.target_j[0]), float(self.target_j[1])]], dtype=torch.float64)
            else:
                valid, s1, s2 = self.robot.inverse_kinematic([[float(self.target_c.x), float(self.target_c.y)]], corrected=True)
                goals = torch.cat([s1[valid], s2[valid]])
        q = as_f64(goals, self.device)
        if q.dim() == 2 and q.shape[1] == 2:
            q = q.unsqueeze(0).expand(n_grids, -1, -1)
        if q.dim() != 3 or q.shape[0] != n_grids or q.shape[2] != 2:
            raise ValueError("goal poses must be [G, 2] or [n_grids, G, 2], got %s" % (tuple(q.shape),))
        k1, k2, ok = self._nearest(q.reshape(-1, 2), b1, b2, lo, st, w)
        g = torch.arange(n_grids, dtype=torch.int64, device=self.device).repeat_interleave(q.shape[1])
        img = torch.zeros(n_grids * b1 * b2, dtype=torch.bool, device=self.device)
        img[((g * b1 + k1) * b2 + k2)[ok]] = True
        return img.view(n_grids, b1, b2)

    def cspace_distance_of(self, dist, joints=None, lo=(0.0, 0.0), step=None, wrap=None):
        """The distance (cspace_distance) at the nearest lattice pose of each of M poses, on the grid of env m: the rule
        of cspace_component_of.  -1 for a colliding pose and for a pose off the lattice (or NaN), -2 where no goal is
        reachable.  Returns int32 [M]."""
        return self._lookup(dist, joints, lo, step, wrap)

    def cspace_path(self, dist, max_len, joints=None, lo=(0.0, 0.0), step=None, wrap=None):
        """Lattice paths down a cspace_distance field: from the nearest lattice pose of each of M poses (the snapping
        rule of cspace_component_of, on the grid of env m), each step goes to the first neighbour, in the order
        (i+1, j), (i-1, j), (i, j+1), (i, j-1) (across a seam only where the axis wraps), whose distance is one less,
        until a goal or max_len poses.  joints: [M, 2] float64 (default: the current joints); lo, step, wrap: those of
        the call that made `dist`.
        Returns (path int32 [M, max_len], length int32 [M]).  path[m, :length[m]] are grid-local indices k = i * b2 + j,
        then -1; index k is the joint pose lo + (k // b2, k % b2) * step.  length = min(dist + 1, max_len), 0 for a
        start that is colliding, unreachable, off the lattice or NaN.  The walk is on the lattice image only."""
        max_len = int(max_len)
        if max_len < 1:
            raise ValueError("max_len must be >= 1, got %d" % max_len)
        n_grids, b1, b2 = dist.shape
        g, k1, k2, ok = self._snap(dist.shape, joints, lo, step, wrap)
        _, _, w = self._lattice(b1, b2, lo, step, wrap)
        start = torch.where(ok, k1 * b2 + k2, -1).to(torch.int32)
        m = start.numel()
        path = torch.empty(m, max_len, dtype=torch.int32, device=self.device)
        length = torch.empty(m, dtype=torch.int32, device=self.device)
        d = dist.to(self.device, torch.int32).contiguous()
        _lib.check(self._lib.ag_cspace_descend(ptr(d), n_grids, b1, b2, w, ptr(start), ptr(g), m, max_len, ptr(path),
                                               ptr(length), stream_ptr(self.device)), "ag_cspace_descend")
        return path, length

    def check_target_reached(self):
        """scene_0.py:115-133 -> bool [N]"""
        eps = 2e-3
        if self.choose_j_tar:
            return ((self.robot.joint_1 - float(self.target_j[0])).abs() < eps) & \
                   ((self.robot.joint_2 - float(self.target_j[1])).abs() < eps)
        ee = self.robot.end_effector()
        return ((float(self.target_c.x) - ee[:, 0]).abs() < eps) & ((float(self.target_c.y) - ee[:, 1]).abs() < eps)

    def sample_action(self, scale_factor=0.1, generator=None):
        """scene_0.py:78-86 for every env: (u - 0.5) * scale_factor, float64 [N,2] on the device."""
        u = torch.rand(self.n, 2, dtype=torch.float64, device=self.device, generator=generator)
        return (u - 0.5) * scale_factor

    # ---- K1 ------------------------------------------------------------------------------------
    def step(self, action, want_ee=False, want_first_hit=False, engine=None, targets=None):
        """scene_0.py:88-103 for every env.  action: [N,2] float64 (or float32) CUDA tensor.
        Returns (joint_1, joint_2, step_reward, done, collision_status) tensors, plus a dict with
        ee / dist / first_hit when requested.  targets: optional [N,2] float64 per-env cartesian targets
        replacing target_c (gym-style callers)."""
        action = torch.as_tensor(action, device=self.device)
        if action.dtype not in (torch.float32, torch.float64):
            action = action.to(torch.float64)
        action = action.reshape(self.n, 2).contiguous()
        if targets is not None:
            targets = as_f64(targets, self.device).reshape(self.n, 2).contiguous()
        ee = torch.empty(self.n, 2, dtype=torch.float64, device=self.device) if want_ee else None
        dist = torch.empty(self.n, 2, dtype=torch.float64, device=self.device) if want_ee else None
        fh = torch.empty(self.n, dtype=torch.int32, device=self.device) if want_first_hit else None
        g = self.grid.c_struct()
        _lib.check(self._lib.ag_step(self.params(), g, ptr(self.robot.joint_1), ptr(self.robot.joint_2), ptr(action),
                                     1 if action.dtype == torch.float32 else 0, ptr(self.step_reward),
                                     ptr(self.flags), ptr(ee), ptr(dist), ptr(fh), ptr(self.stats), ptr(targets), self.n,
                                     self.env_id0, self.engine if engine is None else _engine(engine),
                                     stream_ptr(self.device)), "ag_step")
        out = (self.robot.joint_1, self.robot.joint_2, self.step_reward, self.done, self.collision_status)
        if want_ee or want_first_hit:
            return out + (dict(ee=ee, dist=dist, first_hit=fh),)
        return out

    # ---- K3 ------------------------------------------------------------------------------------
    def _reset(self, mask, reset_u, clear_flags, engine=None):
        if mask is not None:
            mask = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        R = 0
        if reset_u is not None:
            reset_u = as_f64(reset_u, self.device).reshape(self.n, -1, 2).contiguous()
            R = reset_u.shape[1]
        g = self.grid.c_struct()
        _lib.check(self._lib.ag_reset(self.params(), g, ptr(self.robot.joint_1), ptr(self.robot.joint_2),
                                      ptr(self.step_reward), ptr(self.flags), ptr(self.reset_ctr), ptr(mask),
                                      ptr(reset_u), R, self.seed, 1 if clear_flags else 0, ptr(self.stats), self.n,
                                      self.env_id0, self.engine if engine is None else _engine(engine),
                                      stream_ptr(self.device)), "ag_reset")

    def reset(self, mask=None, reset_u=None):
        """scene_0.py:105-113 for envs with mask != 0 (all if None): resample the pose only while it
        collides, then clear reward / done / collision_status.  Candidates: reset_u [N,R,2]
        uniforms consumed from reset_ctr, or Philox stream 1."""
        self._reset(mask, reset_u, True)

    def random_valid_pose(self, mask=None, reset_u=None):
        """scene_0.py:174-181 (bounded by max_reset_tries; exhausted envs are counted in stats)."""
        self._reset(mask, reset_u, False)

    # ---- K4 ------------------------------------------------------------------------------------
    def _rollout_args(self, K, actions, reset_u, rec, engine, targets=None, diag=True, events=None):
        a = _lib.RolloutArgs()
        a.n, a.env_id0, a.K = self.n, self.env_id0, int(K)
        a.engine = self.engine if engine is None else _engine(engine)
        a.seed = self.seed
        a.actions = None if actions is None else actions.data_ptr()
        a.R = 0
        if reset_u is not None:
            a.reset_u, a.R = reset_u.data_ptr(), reset_u.shape[1]
        a.j1, a.j2 = self.robot.joint_1.data_ptr(), self.robot.joint_2.data_ptr()
        a.reward, a.flags = self.step_reward.data_ptr(), self.flags.data_ptr()
        a.step_ctr, a.reset_ctr, a.ep_len = self.step_ctr.data_ptr(), self.reset_ctr.data_ptr(), self.ep_len.data_ptr()
        if rec is not None:
            a.rec_j1, a.rec_j2 = rec["j1"].data_ptr(), rec["j2"].data_ptr()
            a.rec_reward = rec["reward"].data_ptr() if rec.get("reward") is not None else None
            a.rec_flags = rec["flags"].data_ptr() if rec.get("flags") is not None else None
        if events is not None:
            a.events, a.event_count = events["events"].data_ptr(), events["count_buf"].data_ptr()
            a.event_capacity = events["events"].shape[0]
        a.stats = self.stats.data_ptr()
        a.diag = self.diag.data_ptr() if diag else None
        a.targets = None if targets is None else targets.data_ptr()
        return a

    def alloc_records(self, K, pinned_host=False, reward=True):
        """Record buffers of a K-step rollout.  reward=False (host buffers only) leaves the reward plane out: in a
        rollout record the reward is a function of the flags (`reward_from_flags`), so it need not cross PCIe."""
        kw = dict(device="cpu", pin_memory=True) if pinned_host else dict(device=self.device)
        rec = dict(j1=torch.empty(K, self.n, dtype=torch.float32, **kw),
                   j2=torch.empty(K, self.n, dtype=torch.float32, **kw),
                   flags=torch.empty(K, self.n, dtype=torch.uint8, **kw))
        if reward or not pinned_host:
            rec["reward"] = torch.empty(K, self.n, dtype=torch.float32, **kw)
        return rec

    def reward_from_flags(self, flags):
        """step_reward of rollout records from their flags (scene_0.py:95-100; the rollout loop resets after every
        terminal step, so nothing is sticky): 1e4 if done, else -1e3 if collision, else 0."""
        p = self.params()
        f = torch.as_tensor(flags)
        out = torch.zeros(f.shape, dtype=torch.float32, device=f.device)
        out[(f & _lib.FLAG_COLLISION) != 0] = float(p.reward_collision)
        out[(f & _lib.FLAG_DONE) != 0] = float(p.reward_reach)
        return out

    def rollout(self, K, actions=None, reset_u=None, record=True, out=None, engine=None, targets=None, diag=True,
                events=None):
        """The loop body of experiment/experiment_0.py:20-34, K times, in ONE kernel:
        action -> step -> record -> reset when done or collision.

        actions: [K,N,2] float32 CUDA tensor, or None for in-kernel Philox actions
                 ((u-0.5)*0.1 in float64, stream 0, keyed by (seed, global env id, step counter)).
        reset_u: [N,R,2] float64 uniforms for reset candidates, or None for Philox stream 1.
        record : write (joint_1, joint_2, step_reward, flags) per step into `out`
                 (dict of [K,N] tensors from alloc_records) -- post-step, pre-reset, like the reference's
                 record.append.  Episode statistics always accumulate into self.stats.
        targets: optional [N,2] float64 per-env cartesian targets replacing target_c in the reach test
                 (scene_0.py:129-130); ignored in joint-target mode.
        diag   : accumulate the FAST-filter diagnostics into self.diag (a few shared-memory atomics per warp exit).
        events : optional event sink from alloc_event_sink(device tensors): every eventful step appends
                 (env, step << 8 | flags, reward bits); with it `out` may hold the joint planes only.
        """
        if actions is not None:
            actions = torch.as_tensor(actions, device=self.device)
            if actions.dtype != torch.float32 or tuple(actions.shape) != (K, self.n, 2):
                raise ValueError("actions must be float32 [K,N,2]")
            actions = actions.contiguous()
        if reset_u is not None:
            reset_u = as_f64(reset_u, self.device).reshape(self.n, -1, 2).contiguous()
        rec = None
        if record:
            rec = out if out is not None else self.alloc_records(K)
        if targets is not None:
            targets = as_f64(targets, self.device).reshape(self.n, 2).contiguous()
        a = self._rollout_args(K, actions, reset_u, rec, engine, targets, diag, events)
        g = self.grid.c_struct()
        _lib.check(self._lib.ag_rollout(self.params(), g, C.byref(a), stream_ptr(self.device)), "ag_rollout")
        return rec

    # ---- event-compacted sink (SURVEY 8f.1): joints per step, reward / flags only where something happened ----
    def alloc_event_sink(self, K, capacity=None, pinned_host=False):
        """Buffers of the compact trajectory form: the two joint planes [K,N] float32 and an event list
        [capacity,3] uint32 = (env, step << 8 | flags, float32 bits of step_reward) for the eventful env-steps (terminal
        steps: ~0.1 % on scene_0).  `count_buf` is the int64 event counter the kernels advance (reset it between device
        rollouts); `count` holds the number of events of the last rollout_events_host call."""
        kw = dict(device="cpu", pin_memory=True) if pinned_host else dict(device=self.device)
        cap = int(capacity) if capacity is not None else max(1024, (K * self.n) // 16)
        return dict(j1=torch.empty(K, self.n, dtype=torch.float32, **kw), j2=torch.empty(K, self.n, dtype=torch.float32, **kw),
                    events=torch.zeros(cap, 3, dtype=torch.int32, **kw), count_buf=torch.zeros(1, dtype=torch.int64, **kw), count=0)

    @staticmethod
    def decode_events(sink, count=None):
        """(env [M], step [M], flags [M], reward [M]) numpy arrays of the first `count` events of a sink (host side)."""
        c = int(sink["count"] if count is None else count)
        c = min(c, sink["events"].shape[0])
        ev = sink["events"][:c].cpu().numpy().view(np.uint32)
        return (ev[:, 0].astype(np.int64), (ev[:, 1] >> 8).astype(np.int64), (ev[:, 1] & 0xFF).astype(np.uint8),
                ev[:, 2].copy().view(np.float32))

    def events_to_planes(self, sink, K, count=None):
        """Rebuild the dense reward / flags planes [K,N] of a rollout from its event list (numpy)."""
        env, step, fl, rw = self.decode_events(sink, count)
        reward = np.zeros((K, self.n), dtype=np.float32)
        flags = np.zeros((K, self.n), dtype=np.uint8)
        reward[step, env] = rw
        flags[step, env] = fl
        return reward, flags

    def rollout_events_host(self, K, sink, chunk_steps=4, engine=None):
        """End-to-end form with the least bytes on the bus: the actions are drawn in the kernel (Philox stream 0 keyed by
        (seed, global env id, step counter) -- `philox_actions` reproduces any env's actions on the host), nothing goes
        host -> device; the joint planes stream out (8 B per env-step) and reward / flags only as events (12 B each).
        `sink` = alloc_event_sink(K, pinned_host=True).  Returns the episode statistics of this call."""
        cap = sink["events"].shape[0]
        key = ("events", K, int(chunk_steps), cap)
        if key not in self._pipelines:
            h = C.c_void_p()
            _lib.check(self._lib.ag_pipeline_create(C.byref(h), self.device.index, self.n, K, 1 << 17, max(1, int(chunk_steps)),
                                                    1, cap), "ag_pipeline_create")
            self._pipelines[key] = h
        a = self._rollout_args(K, None, None, dict(j1=sink["j1"], j2=sink["j2"]), engine, None, False, sink)
        a.stats = None
        g = self.grid.c_struct()
        st = np.zeros(_lib.ST_COUNT, dtype=np.int64)
        torch.cuda.current_stream(self.device).synchronize()   # env state must be settled
        _lib.check(self._lib.ag_rollout_host(self._pipelines[key], self.params(), g, C.byref(a),
                                             st.ctypes.data_as(C.c_void_p)), "ag_rollout_host")
        sink["count"] = int(sink["count_buf"][0].item())
        self.stats += torch.from_numpy(st).to(self.device)
        return dict(zip(_lib.STAT_NAMES, st.tolist()))

    def philox_actions(self, env_ids, step_ctr0, K):
        """The float64 actions the kernels draw for local envs `env_ids` at draw indices step_ctr0 .. step_ctr0+K-1
        (scene_0.py:84-85 with Philox4x32-10 stream 0 keyed by (seed, global env id)): [K, len(env_ids), 2]."""
        from ..utils.philox import uniform2
        env_ids = np.asarray(env_ids, dtype=np.uint64)
        gid = env_ids + np.uint64(self.env_id0)
        draws = (np.asarray(step_ctr0, dtype=np.uint64).reshape(1, -1) + np.arange(K, dtype=np.uint64).reshape(-1, 1))
        u0, u1 = uniform2(self.seed, np.broadcast_to(gid, draws.shape), draws, 0)
        scale = float(self.params().action_scale)
        return np.stack([(u0 - 0.5) * scale, (u1 - 0.5) * scale], axis=-1)

    def rollout_host(self, K, actions_host=None, out_host=None, chunk_envs=1 << 17, engine=None, chunk_steps=0):
        """End-to-end form of `rollout` for host-resident data: actions_host [K,N,2] float32 and
        the record arrays of `out_host` (alloc_records(K, pinned_host=True)) live in (pinned) host
        memory; H2D copy, kernel and D2H copy are pipelined on three streams, over slices of `chunk_steps` steps
        (all envs; contiguous copies, the faster form) or, with chunk_steps=0, over slices of `chunk_envs` envs.
        Returns the episode statistics of this call as a dict (also added to self.stats)."""
        record = out_host is not None
        key = (K, int(chunk_envs), int(chunk_steps), record)
        if key not in self._pipelines:
            h = C.c_void_p()
            _lib.check(self._lib.ag_pipeline_create(C.byref(h), self.device.index, self.n, K, int(chunk_envs),
                                                    int(chunk_steps), 1 if record else 0, 0), "ag_pipeline_create")
            self._pipelines[key] = h
        if actions_host is not None:
            if actions_host.dtype != torch.float32 or tuple(actions_host.shape) != (K, self.n, 2) \
                    or actions_host.device.type != "cpu":
                raise ValueError("actions_host must be a float32 [K,N,2] host tensor")
        a = self._rollout_args(K, actions_host, None, out_host, engine)
        a.stats = None
        g = self.grid.c_struct()
        st = np.zeros(_lib.ST_COUNT, dtype=np.int64)
        torch.cuda.current_stream(self.device).synchronize()   # env state must be settled
        _lib.check(self._lib.ag_rollout_host(self._pipelines[key], self.params(), g, C.byref(a),
                                             st.ctypes.data_as(C.c_void_p)), "ag_rollout_host")
        self.stats += torch.from_numpy(st).to(self.device)
        return dict(zip(_lib.STAT_NAMES, st.tolist()))

    def __del__(self):
        try:
            for h in self._pipelines.values():
                self._lib.ag_pipeline_destroy(h)
        except Exception:
            pass


class Scene:
    """The reference's single-environment `Scene`, same constructor, attributes and return
    values; each call is one N=1 launch of the batched kernels.  Random draws come from the
    global numpy stream in the reference's order (sample_action: d1 then d2; random_valid_pose:
    joint_1 then joint_2 per attempt), so a seeded run reproduces the reference's trajectory."""

    def __init__(self, robot=None, env=None, target_c=None, visualize=False):
        if visualize:
            raise NotImplementedError("visualisation (scene_0.py:41-58,135-172) is outside the hot path")
        self.robot = robot if robot is not None else TwoJointRobot()
        env = env if env is not None else OccupancyGrid()
        self._env = env
        self.occ_matrix, self.occ_coord, self.obstacle_list, self.obstacle_side_length = env.get_occupancy_grid()
        self.vis = False
        self.target_c = target_c if target_c is not None else Point(-0.2, -0.3)
        self.target_j = np.array([1.1, -0.2])
        self.choose_j_tar = False
        self.step_reward = 0
        self.collision_status = False
        self.done = False
        self._b = None

    def _batched(self) -> BatchedScene:
        r = self.robot
        if self._b is None:
            br = BatchedTwoJointRobot([r.joint_1], [r.joint_2], r.link_1, r.link_2)
            self._b = BatchedScene(br, self._env, self.target_c, engine="exact")
        b = self._b
        b.robot.link_1, b.robot.link_2 = r.link_1, r.link_2
        b.target_c, b.target_j, b.choose_j_tar = self.target_c, self.target_j, self.choose_j_tar
        b.robot.joint_1.fill_(float(r.joint_1))
        b.robot.joint_2.fill_(float(r.joint_2))
        b.step_reward.fill_(float(self.step_reward))
        b.flags.fill_((1 if self.collision_status else 0) | (2 if self.done else 0))
        return b

    def collision_check(self):
        return bool(self._batched().collision_check()[0].item())

    def sample_action(self, scale_factor=0.1):
        d1 = (np.random.rand() - 0.5) * scale_factor
        d2 = (np.random.rand() - 0.5) * scale_factor
        return np.array([d1, d2])

    def step(self, action):
        b = self._batched()
        act = torch.tensor([[float(action[0]), float(action[1])]], dtype=torch.float64, device=b.device)
        j1, j2, rw, done, coll = b.step(act)
        self.robot.joint_1 = np.float64(j1.item())
        self.robot.joint_2 = np.float64(j2.item())
        r = float(rw.item())
        self.step_reward = r if r != 0.0 else 0   # the reference keeps the int 0 until a terminal step
        self.done = bool(done.item())
        self.collision_status = bool(coll.item())
        return self.robot.joint_1, self.robot.joint_2, self.step_reward, self.done, self.collision_status

    def reset(self):
        self.random_valid_pose()
        self.collision_status = False
        self.done = False
        self.step_reward = 0

    def check_target_reached(self):
        return bool(self._batched().check_target_reached()[0].item())

    def random_valid_pose(self):
        while self.collision_check():
            self.robot.joint_1 = np.random.rand() * np.pi * 2.0
            self.robot.joint_2 = np.random.rand() * np.pi * 2.0

    def render(self):
        raise NotImplementedError("visualisation is outside the hot path")

    def occ_to_patch(self):
        raise NotImplementedError("visualisation is outside the hot path")
