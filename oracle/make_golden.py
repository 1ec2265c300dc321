"""Generate tests/golden/* by running the UNMODIFIED reference (via oracle/ref_boot.py).

Run here (the container that has /root/reference):  python oracle/make_golden.py
The fixtures are committed; the GPU box and the CPU test suite only read them.
TEST INFRASTRUCTURE ONLY.
"""
import hashlib
import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_boot  # noqa: E402

OUT = os.path.join(HERE, "..", "tests", "golden")


def experiment0(R, seed, steps=20000):
    """experiment/experiment_0.py:13-34 with a seeded global numpy stream."""
    np.random.seed(seed)
    rob = R.TwoJointRobot(joint_1=1.0, joint_2=2.5)
    occ = R.OccupancyGrid(size=9, random_obstacle=False)
    s = R.Scene(rob, occ)
    s.random_valid_pose()
    h = hashlib.sha256()
    resets, first, dones = [], None, 0
    for i in range(steps):
        a = s.sample_action(scale_factor=0.1)
        j1, j2, r, d, c = s.step(a)
        h.update(struct.pack("<5d2B", j1, j2, a[0], a[1], r, d, c))
        if i == 0:
            first = [float(j1), float(j2), float(a[0]), float(a[1]), float(r), bool(d), bool(c)]
        dones += int(d)
        if d or c:
            resets.append(i)
            s.reset()
    return dict(seed=seed, steps=steps, sha256=h.hexdigest(), resets=resets, dones=dones,
                first_record=first, final_joints=[float(rob.joint_1), float(rob.joint_2)],
                start_joints=[1.0, 2.5])


def predicate_cases(R, rng, n):
    """Random + adversarial (segment, square) pairs through Line/CollisionChecker."""
    seg = np.zeros((n, 4)); sq = np.zeros((n, 4))
    abc = np.zeros((n, 3)); signs = np.zeros((n, 4)); out = np.zeros(n, dtype=np.int8)
    for i in range(n):
        kind = i % 8
        side = rng.choice([0.2, 1.6 / 30, 0.4, 0.008])
        bx, by = rng.uniform(-0.9, 0.7, 2)
        if kind == 0:      # arm-like: link 1 from the origin
            th = rng.uniform(0, 2 * np.pi)
            p0 = (0, 0); p1 = (np.cos(th) * 0.4, np.sin(th) * 0.4)
            bx, by = rng.uniform(-0.6, 0.4, 2)
        elif kind == 1:    # arm-like: link 2
            t1, t2 = rng.uniform(0, 2 * np.pi, 2)
            p0 = (np.cos(t1) * 0.4, np.sin(t1) * 0.4)
            p1 = (p0[0] + np.cos(t2) * 0.3, p0[1] + np.sin(t2) * 0.3)
            bx, by = p0[0] + rng.uniform(-0.3, 0.2), p0[1] + rng.uniform(-0.3, 0.2)
        elif kind == 2:    # endpoint exactly on a corner / edge of the square
            p0 = tuple(rng.uniform(-0.7, 0.7, 2))
            p1 = (bx + side * rng.integers(0, 2), by + side * rng.choice([0.0, 0.5, 1.0]))
        elif kind == 3:    # segment wholly inside the square
            p0 = (bx + side * rng.uniform(0.05, 0.95), by + side * rng.uniform(0.05, 0.95))
            p1 = (bx + side * rng.uniform(0.05, 0.95), by + side * rng.uniform(0.05, 0.95))
        elif kind == 4:    # starts inside, leaves
            p0 = (bx + side * rng.uniform(0.05, 0.95), by + side * rng.uniform(0.05, 0.95))
            p1 = tuple(rng.uniform(-0.9, 0.9, 2))
        elif kind == 5:    # line through the square, segment stops short / beyond
            cx, cy = bx + side / 2, by + side / 2
            th = rng.uniform(0, 2 * np.pi); d0 = rng.uniform(0.05, 0.6); ln = rng.uniform(0.01, 0.7)
            p0 = (cx - np.cos(th) * d0, cy - np.sin(th) * d0)
            p1 = (p0[0] + np.cos(th) * ln, p0[1] + np.sin(th) * ln)
        elif kind == 6:    # axis-aligned segments (crash in the reference when the line crosses)
            p0 = tuple(rng.uniform(-0.7, 0.7, 2))
            p1 = (p0[0], rng.uniform(-0.7, 0.7)) if rng.random() < 0.5 else (rng.uniform(-0.7, 0.7), p0[1])
        else:              # generic
            p0 = tuple(rng.uniform(-0.9, 0.9, 2)); p1 = tuple(rng.uniform(-0.9, 0.9, 2))
        square = R.Square(R.Point(bx, by), R.Point(bx + side, by + side))
        line = R.Line(R.Point(p0[0], p0[1]), R.Point(p1[0], p1[1]))
        cc = R.CollisionChecker(line, square)
        seg[i] = (p0[0], p0[1], p1[0], p1[1])
        sq[i] = (square.min_x, square.min_y, square.max_x, square.max_y)
        abc[i] = (cc.a, cc.b, cc.c)
        signs[i] = cc.compute_corner_line_value()
        try:
            out[i] = 1 if cc.collision_check() else 0
        except AttributeError:   # utils/collision_checker.py:60,65 (Line has no max_x/min_x)
            out[i] = 2
    return dict(seg=seg, sq=sq, abc=abc, signs=signs, out=out)


def grid_from_ref(g):
    occ = np.asarray(g.occ)
    sq = np.array([[o.min_x, o.min_y, o.max_x, o.max_y] for o in g.obstacle_list], dtype=np.float64)
    return occ, sq


def ref_collision_all(R, scene):
    """flag (Scene.collision_check) and min row-major cell index over ALL hit obstacles."""
    rb = scene.robot
    l1 = R.Line(R.Point(0, 0), R.Point(rb.elbow_point().x, rb.elbow_point().y))
    l2 = R.Line(R.Point(rb.elbow_point().x, rb.elbow_point().y), R.Point(rb.end_effector().x, rb.end_effector().y))
    hits = []
    for i, ob in enumerate(scene.obstacle_list):
        if R.CollisionChecker(l1, ob).collision_check() or R.CollisionChecker(l2, ob).collision_check():
            hits.append(i)
    return hits


def scene_cases(R, rng, grid, cell_index, n_env, n_steps):
    """n_env envs x n_steps sticky steps (no reset) through Scene.step."""
    j0 = rng.uniform(0, 2 * np.pi, (n_env, 2))
    acts = (rng.random((n_env, n_steps, 2)) - 0.5) * 0.1
    # a few envs aimed at the target so that `done` and collide+reach orderings are exercised
    out = np.zeros((n_env, n_steps, 5)); fh = np.full((n_env, n_steps), -1, dtype=np.int32)
    ee = np.zeros((n_env, n_steps, 2))
    for e in range(n_env):
        rob = R.TwoJointRobot(joint_1=j0[e, 0], joint_2=j0[e, 1])
        sc = R.Scene(rob, grid)
        for t in range(n_steps):
            j1, j2, r, d, c = sc.step(acts[e, t])
            out[e, t] = (j1, j2, r, d, c)
            hits = ref_collision_all(R, sc)
            assert bool(hits) == bool(sc.collision_check())
            fh[e, t] = min(cell_index[h] for h in hits) if hits else -1
            p = rob.end_effector()
            ee[e, t] = (p.x, p.y)
    return dict(j0=j0, actions=acts, out=out, first_hit=fh, ee=ee)


def main():
    R = ref_boot.boot()
    os.makedirs(OUT, exist_ok=True)
    meta = {"numpy": np.__version__}

    # --- known answers of the reference's __main__ blocks (SURVEY.md section 4)
    c = R.CollisionChecker(R.Line(R.Point(0, 0), R.Point(1, 2)), R.Square(R.Point(0, 0.8), R.Point(0.9, 1.4)))
    s1, s2 = R.TwoJointRobot().inverse_kinematic(R.Point(0.5, 0.0))
    np.random.seed(0)
    g201 = R.OccupancyGrid(201)
    rb = R.TwoJointRobot(0.3, 1.2)
    meta["known"] = dict(collision_main=bool(c.collision_check()), ik_s1=[float(x) for x in s1],
                         ik_s2=[float(x) for x in s2], grid201_seed0_count=len(g201.occ_coordinate),
                         grid201_side=float(g201.obstacle_side_length),
                         fk_0p3_1p2=dict(ee=[float(rb.end_effector().x), float(rb.end_effector().y)],
                                         elbow=[float(rb.elbow_point().x), float(rb.elbow_point().y)]))
    np.savez_compressed(os.path.join(OUT, "grid201_seed0.npz"), occ=np.packbits(np.asarray(g201.occ, dtype=np.uint8)),
                        first_squares=grid_from_ref(g201)[1][:64], last_squares=grid_from_ref(g201)[1][-64:])

    # --- experiment_0 loops
    meta["experiment0"] = [experiment0(R, s) for s in (0, 1, 2)]

    # --- predicate / FK fixtures
    rng = np.random.default_rng(1234)
    # 16000 cases are drawn (the later fixtures depend on the generator's state); the first 12000 (1500 of each kind)
    # are stored, which keeps the file under 1 MB
    pred = predicate_cases(R, rng, 16000)
    np.savez_compressed(os.path.join(OUT, "predicate_cases.npz"), **{k: v[:12000] for k, v in pred.items()})
    j = rng.uniform(-20, 20, (4000, 2))
    fk = np.zeros((4000, 4))
    for i in range(4000):
        rb = R.TwoJointRobot(j[i, 0], j[i, 1])
        fk[i] = (rb.elbow_point().x, rb.elbow_point().y, rb.end_effector().x, rb.end_effector().y)
    np.savez_compressed(os.path.join(OUT, "fk_cases.npz"), j=j, fk=fk)

    # --- grids (G1) and scene steps (C1,R1,ST)
    grids = {}
    g = R.OccupancyGrid(size=9, random_obstacle=False)
    grids["manual9"] = (g, [5 * 9 + 6, 5 * 9 + 7, 2 * 9 + 3])
    for name, S, p, seed in (("rand9", 9, 0.1, 11), ("rand31", 31, 0.01, 12), ("rand64", 64, 0.02, 13),
                             ("rand6", 6, 0.2, 14)):
        np.random.seed(seed)
        g = R.OccupancyGrid(size=S, random_obstacle=True, obstacle_probability=p)
        ys, xs = np.where(np.asarray(g.occ) != 0)
        grids[name] = (g, [int(r * S + c) for r, c in zip(ys, xs)])
    mat = np.array([[0, 0, 1, 0, 0], [0, 1, 1, 0, 0], [0, 1, 1, 0, 0], [0, 0, 0, 0, 0], [0, 1, 0, 0, 1]])
    g = R.OccupancyGrid(size=9, random_obstacle=False)
    g.load_from_matrix(mat)          # environment/occupancy_grid.py:73-93 (the commented example :97-99)
    ys, xs = np.where(mat != 0)
    grids["matrix5"] = (g, [int(r * 5 + c) for r, c in zip(ys, xs)])
    save = {}
    for name, (g, ci) in grids.items():
        occ, sq = grid_from_ref(g)
        n_env, n_steps = (96, 12) if name != "rand64" else (48, 8)
        sc = scene_cases(R, rng, g, ci, n_env, n_steps)
        save[name + "/occ"] = np.asarray(occ != 0, dtype=np.uint8)
        save[name + "/squares"] = sq
        save[name + "/cell_index"] = np.asarray(ci, dtype=np.int32)
        save[name + "/env_size"] = np.float64(g.environment_size)
        for k, v in sc.items():
            save[name + "/" + k] = v
    # target-reaching sequence: walk the arm onto the default target (collide+reach / done paths)
    g = grids["manual9"][0]
    rob = R.TwoJointRobot(joint_1=0.0, joint_2=0.0)
    s1, s2 = rob.inverse_kinematic(R.Point(-0.2, 0.3))  # IK drops the sign of y (SURVEY 2.1 #3)
    reach = []
    for sol in (s1, s2):
        for flip in (1.0, -1.0):
            jt = np.array([flip * sol[0], flip * sol[1]])
            rob = R.TwoJointRobot(joint_1=jt[0] - 0.03, joint_2=jt[1] + 0.02)
            sc = R.Scene(rob, g)
            seq = []
            for t in range(8):
                a = np.array([0.01, -0.00666]) if t < 3 else np.array([0.0004, 0.0003])
                j1, j2, r, d, c = sc.step(a)
                seq.append((a[0], a[1], j1, j2, r, d, c))
            reach.append([(jt[0] - 0.03, jt[1] + 0.02)] + seq)
    save["reach/start"] = np.array([r[0] for r in reach])
    save["reach/seq"] = np.array([r[1:] for r in reach], dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "scene_cases.npz"), **save)

    with open(os.path.join(OUT, "reference_goldens.json"), "w") as f:
        json.dump(meta, f, indent=1)
    print(json.dumps({k: (v if k != "experiment0" else [dict(seed=x["seed"], sha=x["sha256"][:16],
                                                          resets=len(x["resets"])) for x in v])
                      for k, v in meta.items()}, indent=1))


if __name__ == "__main__":
    main()
