#!/usr/bin/env python
"""bench.py -- env-steps/s of the scene_0 step/reset hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU arithmetic (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the outputs of the last timed launch to DIR

One bench "step" = ONE fused rollout launch (K4) over this rank's environments:
2^20 envs x 64 env-steps, RECORD mode (reads float32 actions [64,N,2], writes the trajectory
records the reference appends per step: joint_1, joint_2, reward, flags) -- BASELINE.json
configs[2] ("scene_0 with 1M envs per GPU, fused 64-step rollout kernel, at 1/2/4/8 B200").
N>1: one process per GPU (torchrun), contiguous env slices with global env ids, replicated grid,
no data-path collective; the int64[8] episode statistics are all-reduced (NCCL) inside the timed
region -- every `--reduce-every` launches and once more at the end (the counters are cumulative,
so this equals a reduction after every launch).  `value` = env-steps of all ranks / max-over-ranks time.

After the headline the same run times BASELINE.json configs[3] and configs[4] (`configs.c4`, `configs.c5`
in the JSON line; `--grid c4|c5` makes one of them the headline instead):
  c4  one 1024x1024 bit-packed Bernoulli(0.002) map, 2^20 envs/GPU;
  c5  a distinct 256x256 Bernoulli(0.008) map per batch of 256 envs (cells around the arm's base kept free),
      auto-reset, episode statistics all-reduced across the ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic bytes per env-step, RECORD mode (SURVEY.md 8d / DESIGN.md): 8 read + 13 written + ~1 amortised state;
# config 5 adds its 8 KiB map per 256 envs x 64 steps = 0.5 B
B_ALG = {"scene0": 22.0, "c4": 22.0, "c5": 22.5}
METRIC = {"scene0": "env-steps/sec (FK+collision+reward), scene_0 fused 64-step rollout",
          "c4": "env-steps/sec (FK+collision+reward), 1024x1024 dense map, fused 64-step rollout",
          "c5": "env-steps/sec (FK+collision+reward), per-batch 256x256 maps, fused 64-step rollout"}
GRID_NAMES = {"scene0": "scene_0 manual 9x9 grid (3 obstacles)",
              "c4": "one 1024x1024 bit-packed grid, Bernoulli(0.002) obstacles (128 KiB, L2-resident)",
              "c5": "a distinct 256x256 Bernoulli(0.008) grid per batch of 256 envs (8 KiB each, staged by bulk async "
                    "copy; the 4x4 cells around the arm's base kept free so that every map has a free pose)"}
KERNELS = {"scene0": "k_rollout_lut", "c4": "k_rollout_async", "c5": "k_rollout_async"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="environments per GPU")
    ap.add_argument("--rollout-steps", type=int, default=64, help="env-steps fused per launch (K)")
    ap.add_argument("--engine", default="fast", choices=["fast", "exact"])
    ap.add_argument("--mode", default="record", choices=["record", "stats"])
    ap.add_argument("--grid", default="scene0", choices=["scene0", "c4", "c5"],
                    help="the headline workload: scene0 = manual 9x9 map (BASELINE configs[2]); c4 / c5 = configs[3] / [4]")
    ap.add_argument("--sub-configs", default="c4,c5", help="configs timed after the headline (comma list, '' = none)")
    ap.add_argument("--sub-steps", type=int, default=5)
    ap.add_argument("--reduce-every", type=int, default=8, help="statistics all-reduce every M launches (and at the end)")
    ap.add_argument("--chunk-envs", type=int, default=1 << 17, help="envs per pipeline stage of the host-buffer (e2e) path")
    ap.add_argument("--chunk-steps", type=int, default=4, help="steps per pipeline stage of the e2e path (0: slice over envs)")
    ap.add_argument("--e2e-mode", default="events", choices=["events", "records"],
                    help="headline e2e form: events = in-kernel actions, joints + event-compacted reward/flags; "
                         "records = host actions in, full records out")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample-envs", type=int, default=1 << 17)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed launches, write what the last one returned to DIR/<name>.npy (rank 0): the "
                         "record planes and final joints of a fixed, seeded sample of envs, and the episode statistics")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(grid):
    """per-launch DRAM bytes of this workload's kernel from the committed ncu --set full capture (profiles/)"""
    path = os.path.join(ROOT, "profiles", "rollout_traffic.json")
    try:
        d = json.load(open(path))
        return d.get(grid)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], 0.0, set(), 0.0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for r in self.rows if t0 <= r[0] <= t1 + 0.1] or self.rows[-3:]
        for _, line in rows:
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1])); power = max(power, float(f[2]))
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "power_w_max": power, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def workload_config(args, world, grid=None):
    grid = grid or args.grid
    return {"workload": "%s, %d envs/GPU, fused %d-step rollout (K4), %s mode, "
                        "random actions (u-0.5)*0.1, auto-reset" % (GRID_NAMES[grid], args.envs, args.rollout_steps,
                                                                    args.mode.upper()),
            "envs_per_gpu": args.envs, "rollout_steps": args.rollout_steps, "mode": args.mode, "engine": args.engine,
            "arithmetic": ("float64 decisions: float32 interval filter, float64 filter, then the reference's float64 "
                           "operation order for what they cannot settle") if args.engine == "fast" else "float64",
            "grid": grid, "parallelism": "env-sharded x%d, replicated grid, stats all-reduce every %d launches"
                                         % (world, args.reduce_every),
            "l2_policy": "inputs_exceed_l2 (%.0f MB streamed per launch)" %
                         (args.envs * args.rollout_steps * (21 if args.mode == "record" else 0) / 1e6)}


# ------------------------------------------------------------------------------------------ CPU arms
def oracle_workload(args, orc, np, grid=None):
    """(squares per grid, envs_per_grid, sample envs) of the CPU arms.  The oracle tests every obstacle
    (the reference's O(#obstacles) loop), so the high-resolution maps get a smaller sample."""
    grid = grid or args.grid
    if grid == "scene0":
        return [orc.manual_grid()[0]], None, args.cpu_sample_envs
    if grid == "c4":
        occ = (np.random.default_rng(4).random((1024, 1024)) < 0.002).astype(np.uint8)
        return [orc.grid_squares(occ)[0]], None, min(args.cpu_sample_envs, 1 << 11)
    rng = np.random.default_rng(5)
    occs = []
    for _ in range(8):
        o = (rng.random((256, 256)) < 0.008).astype(np.uint8)
        o[126:131, 125:130] = 0
        occs.append(o)
    return [orc.grid_squares(o)[0] for o in occs], 256, min(args.cpu_sample_envs, 1 << 11)


def run_reference(args, rank, world):
    """The reference's own CPU arithmetic for the path, on the host cores.  The reference is pure
    Python; this arm runs its bit-exact C restatement (oracle/, pinned to the reference's goldens) with
    all host threads -- a faster CPU baseline than the reference's interpreter loop, whose own speed is
    reported next to it (cpu_baseline.reference_python) when the vendored copy is present."""
    if rank != 0:
        return
    import numpy as np
    from oracle import oracle as orc
    K = args.rollout_steps
    rng = np.random.default_rng(0)
    sqs, epg, n = oracle_workload(args, orc, np)
    st = orc.RolloutState(rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n))
    actions = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32) if args.mode == "record" else None
    cores = host_cores()                             # torchrun exports OMP_NUM_THREADS=1: ask for every core explicitly
    for _ in range(args.warmup):
        orc.rollout(st, K, sqs, envs_per_grid=epg, seed=0, actions_f32=actions, record=args.mode == "record", threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.rollout(st, K, sqs, envs_per_grid=epg, seed=0, actions_f32=actions, record=args.mode == "record", threads=cores)
    dt = time.perf_counter() - t0
    value = n * K * args.steps / dt
    sample = "%d envs x %d env-steps per step (1/%d of one GPU's batch), OpenMP over envs" % (n, K, max(1, args.envs // n))
    cb = {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample}
    rp = reference_python(cores)
    if rp:
        cb["reference_python"] = rp
    line = {
        "impl": "reference", "metric": METRIC[args.grid], "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_python(cores, steps=20000):
    """The UNMODIFIED reference's loop body (experiment/experiment_0.py:20-34: sample_action -> step -> reset on
    done/collision; manual 9x9 grid), one process and one process per host core (its own threads share the GIL), from
    the vendored copy baseline/_ref/abstract_gym (oracle/vendor_reference.py).  None when the copy is absent."""
    try:
        from oracle import vendor_reference
        if vendor_reference.vendored_root() is None:
            return None
    except Exception:
        return None
    script = os.path.join(ROOT, "oracle", "ref_loop.py")

    def run(nproc):
        ps = [subprocess.Popen([sys.executable, script, "--steps", str(steps), "--seed", str(i)],
                               stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True) for i in range(nproc)]
        outs = [p.communicate(timeout=300)[0] for p in ps]
        secs = [json.loads(o.strip().splitlines()[-1])["seconds"] for o in outs if o.strip()]
        if len(secs) != nproc:
            return None
        return sum(steps / s for s in secs)          # aggregate rate over the loops' own timed sections

    try:
        one, all_ = run(1), run(cores)
    except Exception:
        return None
    if one is None or all_ is None:
        return None
    return {"env_steps_per_s_1_process": one, "env_steps_per_s_all_cores": all_, "cores": cores,
            "steps_per_process": steps,
            "what": "unmodified reference, experiment_0.py:20-34 loop, manual 9x9 grid, one process per core"}


def cpu_baseline(args):
    import numpy as np
    from oracle import oracle as orc
    K = args.rollout_steps
    rng = np.random.default_rng(0)
    sqs, epg, n = oracle_workload(args, orc, np)
    n *= 2
    st = orc.RolloutState(rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 2 * np.pi, n))
    actions = ((rng.random((K, n, 2)) - 0.5) * 0.1).astype(np.float32) if args.mode == "record" else None
    cores = host_cores()
    orc.rollout(st, K, sqs, envs_per_grid=epg, seed=0, actions_f32=actions, record=args.mode == "record", threads=cores)
    reps, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < 8.0:
        orc.rollout(st, K, sqs, envs_per_grid=epg, seed=0, actions_f32=actions, record=args.mode == "record", threads=cores)
        reps += 1
    dt = time.perf_counter() - t0
    out = {"value": n * K * reps / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
           "sample": "%d x (%d envs x %d env-steps), %.1f s, OpenMP over envs" % (reps, n, K, dt)}
    rp = reference_python(cores)
    if rp:
        out["reference_python"] = rp
    return out


# ------------------------------------------------------------------------------------------ GPU arm
def make_grid(ag, np, torch, name, n, world, dev):
    if name == "scene0":
        return ag.OccupancyGrid(size=9, random_obstacle=False)
    if name == "c4":
        grid = ag.OccupancyGrid(size=9, random_obstacle=False)
        grid.load_from_matrix((np.random.default_rng(4).random((1024, 1024)) < 0.002).astype(np.uint8))
        return grid
    ggen = torch.Generator(device=dev).manual_seed(5)     # same maps on every rank; envs pick them by global id
    return ag.BatchedOccupancyGrid.random(max(1, world * n // 256), 256, 0.008, 256, device=dev, generator=ggen,
                                          clear_base_cells=2)


def time_config(args, ag, torch, dist, name, rank, world, dev, actions, rec, steps, warmup):
    """W warm-up + `steps` timed rollout launches of workload `name` on this rank's env slice; the statistics
    all-reduce runs inside the timed region.  Returns (result dict on every rank, scene)."""
    import numpy as np
    n, K = args.envs, args.rollout_steps
    record = args.mode == "record"
    lo = rank * n                                    # weak scaling: every rank owns n envs, global ids [lo, lo+n)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    grid = make_grid(ag, np, torch, name, n, world, dev)
    robot = ag.BatchedTwoJointRobot.random(n, device=dev, generator=gen)
    scene = ag.BatchedScene(robot, grid, engine=args.engine, seed=0, env_id0=lo)
    scene.random_valid_pose()                        # experiment_0.py:16
    M = max(1, args.reduce_every)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(warmup):
        scene.rollout(K, actions=actions, record=record, out=rec, diag=False)
        if (i + 1) % M == 0:
            scene.all_reduce_stats(wait=False)
    scene.all_reduce_stats(wait=True)
    barrier()
    launches0 = ag.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i, (a, b) in enumerate(evs):
        a.record()                                   # same stream the kernel is launched on (torch current stream)
        scene.rollout(K, actions=actions, record=record, out=rec, diag=False)
        b.record()
        if (i + 1) % M == 0:
            scene.all_reduce_stats(wait=False)       # async: overlaps the next launch
    loop_end = torch.cuda.Event(enable_timing=True)
    loop_end.record()
    scene.all_reduce_stats(wait=False)
    g_stats = scene.global_stats()                   # the last reduction is inside the timed region
    stop.record()
    barrier()
    total_ms = start.elapsed_time(stop)
    kern_ms = sum(a.elapsed_time(b) for a, b in evs) / steps
    tail_ms = loop_end.elapsed_time(stop)            # waiting for the last statistics reduction
    launches = ag.launch_count() - launches0
    t = torch.tensor([total_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = t.tolist()
    # the reduced totals must equal the sum of the per-rank counters (integer sums: exact)
    local = scene.stats.clone()
    if world > 1:
        parts = [torch.zeros_like(local) for _ in range(world)]
        dist.all_gather(parts, local)
        summed = torch.stack(parts).sum(dim=0)
    else:
        summed = local
    if not torch.equal(summed.cpu(), g_stats.cpu()):
        raise RuntimeError("all-reduced episode statistics differ from the sum of the per-rank counters: %s vs %s"
                           % (g_stats.tolist(), summed.tolist()))
    peak, peak_src = peaks()
    b_alg = B_ALG[name] if record else 64.0 / K
    achieved = n * K * b_alg / (kern_ms * 1e-3) / 1e9
    traffic = measured_traffic(name)
    res = {
        "metric": METRIC[name], "workload": workload_config(args, world, name)["workload"],
        "value": world * n * K * steps / (total_ms * 1e-3), "unit": "env-steps/s", "steps": steps, "warmup": warmup,
        "ms_per_step": total_ms / steps, "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None if not traffic else traffic.get("dram_bytes_per_launch"),
                     "traffic_source": None if not traffic else traffic.get("source"),
                     "peak_source": peak_src, "bytes_per_env_step": b_alg, "kernel_ms": kern_ms,
                     "kernel": KERNELS[name] if args.engine == "fast" else "k_rollout",
                     "note": "instruction-issue-bound path: see DESIGN.md roofline section"},
        "episode_stats": dict(zip(ag.STAT_NAMES, g_stats.tolist())),
        "stats_check": "all-reduce == sum of per-rank counters (%d ranks)" % world,
        "stats_reduce_tail_ms_rank0": tail_ms,
    }
    return res, scene


DUMP_BYTES = 48 << 20


def dump_outputs(path, scene, rec, K):
    """Write what the last rollout launch handed its caller, as float32 / float64 .npy files: the [K, m] record planes
    and the final joint angles of m envs drawn once with a fixed seed (m fits all of it in DUMP_BYTES), and the
    cumulative episode statistics.  Two builds run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    n = scene.n
    m = min(n, 1 << 15, DUMP_BYTES // (16 * K + 16))
    envs = torch.as_tensor(np.sort(np.random.default_rng(0).choice(n, m, replace=False)), device=scene.device)
    out = {"joint_1": scene.robot.joint_1[envs].double(), "joint_2": scene.robot.joint_2[envs].double(),
           "episode_stats": scene.stats.double()}
    if rec is not None:
        for k in ("j1", "j2", "reward", "flags"):
            out["rec_" + k] = rec[k][:, envs].float()
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def e2e_leg(args, ag, torch, dist, scene, rank, world, dev, actions):
    """The same metric end to end through the public API with HOST buffers, copies inside the timed region."""
    n, K = args.envs, args.rollout_steps
    record = args.mode == "record"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, reps):
        fn()                                         # warm-up (allocates the staging pipeline)
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        scene.all_reduce_stats(wait=True)
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    reps = args.steps
    out = {}
    # (a) full records: host actions in (8 B / env-step), all four record planes out (13 B / env-step)
    if record:
        hact = torch.empty(K, n, 2, dtype=torch.float32, pin_memory=True)
        hact.copy_(actions)
        hout = scene.alloc_records(K, pinned_host=True)
        dt = timed(lambda: scene.rollout_host(K, hact, hout, chunk_envs=args.chunk_envs, chunk_steps=args.chunk_steps), reps)
        out["records"] = {"value": world * n * K * reps / dt, "unit": "env-steps/s",
                          "h2d_bytes_per_step": K * n * 8, "d2h_bytes_per_step": K * n * 13 + 8 * 8 * 3,
                          "reps": reps, "ms_per_step": 1e3 * dt / reps,
                          "api": "BatchedScene.rollout_host(actions_host, records_host): pinned host buffers, 3-stream "
                                 "pipeline over slices of %d steps" % args.chunk_steps}
        del hout, hact
    # (b) event-compacted sink: actions drawn in the kernel (Philox stream 0; any env's actions can be reproduced on
    # the host), joints out (8 B / env-step), reward / flags only for the eventful env-steps
    if hasattr(scene, "rollout_events_host"):
        sink = scene.alloc_event_sink(K, pinned_host=True)
        dt = timed(lambda: scene.rollout_events_host(K, sink, chunk_steps=args.chunk_steps), reps)
        nev = int(sink["count"])
        out["events"] = {"value": world * n * K * reps / dt, "unit": "env-steps/s",
                         "h2d_bytes_per_step": 0, "d2h_bytes_per_step": K * n * 8 + nev * 12 + 8 * 8 * 3,
                         "events_last_call": nev, "reps": reps, "ms_per_step": 1e3 * dt / reps,
                         "api": "BatchedScene.rollout_events_host(sink): in-kernel Philox actions (reproducible on the "
                                "host per env), joints streamed out, (env, step, reward, flags) only for eventful steps"}
    if not out:
        return None
    key = args.e2e_mode if args.e2e_mode in out else next(iter(out))
    e2e = dict(out[key])
    e2e["form"] = key
    for k, v in out.items():
        if k != key:
            e2e[k] = v
    return e2e


def run_ours(args, rank, world, local):
    import torch
    import torch.distributed as dist
    import abstract_gym_b200 as ag

    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from abstract_gym_b200.sharding import bind_to_gpu_numa
    numa_bound = bind_to_gpu_numa(local) if (world > 1 and not os.environ.get("AG_NO_NUMA_BIND")) else False
    n, K = args.envs, args.rollout_steps
    record = args.mode == "record"
    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    actions = rec = None
    if record:   # actions and record buffers are shared by all configs (same shapes)
        actions = ((torch.rand(K, n, 2, device=dev, generator=gen) - 0.5) * 0.1).to(torch.float32)
        rec = {"j1": torch.empty(K, n, dtype=torch.float32, device=dev), "j2": torch.empty(K, n, dtype=torch.float32, device=dev),
               "reward": torch.empty(K, n, dtype=torch.float32, device=dev), "flags": torch.empty(K, n, dtype=torch.uint8, device=dev)}

    sampler = ClockSampler(local) if rank == 0 else None     # covers warm-up, the timed launches, e2e and the sub-configs
    wall_load0 = time.time()
    # ---- headline
    head, scene = time_config(args, ag, torch, dist, args.grid, rank, world, dev, actions, rec, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, scene, rec, K)
    # one more launch with the filter diagnostics on (outside every timed region)
    scene.diag.zero_()
    scene.rollout(K, actions=actions, record=record, out=rec, diag=True)
    torch.cuda.synchronize(dev)
    diag = scene.diag_dict()
    # ---- end to end: host buffers through the public API
    e2e = None
    if not args.no_e2e:
        e2e = e2e_leg(args, ag, torch, dist, scene, rank, world, dev, actions)
    del scene
    # ---- the other BASELINE configs
    subs = {}
    for name in [s for s in args.sub_configs.split(",") if s and s != args.grid]:
        r, sc = time_config(args, ag, torch, dist, name, rank, world, dev, actions, rec, args.sub_steps, 3)
        subs[name] = r
        del sc
        torch.cuda.empty_cache()
    clocks = sampler.stop(wall_load0, time.time()) if sampler else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed launches + e2e loop + sub-configs (the headline's timed launches last %.1f ms)" \
                           % (head["ms_per_step"] * args.steps)
    if rank != 0:
        return
    line = {
        "metric": head["metric"], "value": head["value"], "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": e2e, "gpu_launches": head["gpu_launches"],
        "roofline": head["roofline"],
        "clocks": clocks, "episode_stats": head["episode_stats"], "stats_check": head["stats_check"],
        "filter_diag_rank0": diag, "numa_bound": numa_bound,
        "stats_reduce_tail_ms_rank0": head["stats_reduce_tail_ms_rank0"],
        "configs": subs,
    }
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        from abstract_gym_b200.sharding import nccl_options
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local), pg_options=nccl_options())
    run_ours(args, rank, world, local)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
