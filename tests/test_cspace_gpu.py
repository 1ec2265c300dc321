"""Configuration-space occupancy on the device (ag_cspace_occupancy / BatchedScene.cspace_occupancy /
torch.ops.abstract_gym_b200.cspace_occupancy) against the compositions of tests/cspace_reference.py: K2 on the same poses
(default lattices, axis rows included: bit for bit, every engine) and the CPU oracle (half-step-offset lattices, which
keep every angle pi/b away from the axes)."""
import os

import numpy as np
import pytest

from cspace_reference import composed_occupancy, default_step, oracle_image, pack

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


def scene(ag, torch, grid, engine="fast"):
    z = torch.zeros(1, dtype=torch.float64, device="cuda")
    return ag.BatchedScene(ag.BatchedTwoJointRobot(z, z.clone()), grid, engine=engine)


def steps(b1, b2):
    return (default_step(b1), default_step(b2))


def offset(b1, b2):
    st = steps(b1, b2)
    return (0.5 * st[0], 0.5 * st[1]), st


def assert_words(got, want, what):
    got = got.cpu().numpy().view(np.uint32) if hasattr(got, "cpu") else np.asarray(got, np.uint32)
    want = want.cpu().numpy().view(np.uint32) if hasattr(want, "cpu") else np.asarray(want, np.uint32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    diff = got != want
    assert not diff.any(), "%s: %d of %d words differ, first at %s: %08x vs %08x" % (
        what, diff.sum(), diff.size, np.argwhere(diff)[0], got[diff][0], want[diff][0])


def check_k2(sc, b1, b2, engine, lo=(0.0, 0.0), step=None, what=""):
    """the kernel's words equal K2's composition; returns them"""
    from abstract_gym_b200 import _lib
    step = steps(b1, b2) if step is None else step
    got = sc.cspace_occupancy(b1, b2, lo=lo, step=step, packed=True, engine=engine)
    assert_words(got, composed_occupancy(sc, lo, step, b1, b2, _lib.ENGINES[engine]), "%s %s K2" % (what, engine))
    return got


def check_oracle(orc, sc, grids, b1, b2, engine, what=""):
    """on a half-step-offset lattice the kernel's words equal the oracle's image, grid by grid"""
    lo, st = offset(b1, b2)
    got = sc.cspace_occupancy(b1, b2, lo=lo, step=st, packed=True, engine=engine)
    want = np.stack([pack(oracle_image(orc, g, lo, st, b1, b2)) for g in grids])
    assert_words(got, want, "%s %s oracle" % (what, engine))


@pytest.mark.parametrize("engine", ENGINES)
def test_scene0_offset_lattice_equals_oracle(ag, torch_, oracle, engine):
    sc = scene(ag, torch_, grid_of(ag, None))
    check_oracle(oracle, sc, [oracle.manual_grid()], 512, 512, engine, "scene_0 512^2")


@pytest.mark.parametrize("b", [1024, 4096])
def test_scene0_default_lattice_equals_k2(ag, torch_, b):
    """the whole torus from 0, axis rows q1 = 0, ~pi/2, ~pi, ~3pi/2 included: every engine equals K2 (the map form for
    FAST), and EXACT equals BRUTE"""
    sc = scene(ag, torch_, grid_of(ag, None))
    got = {e: check_k2(sc, b, b, e, what="scene_0 %d^2" % b) for e in ENGINES}
    assert_words(got["exact"], got["brute"], "exact vs brute")
    img = sc.cspace_occupancy(b)[0]
    print("scene_0 %d^2: colliding poses in the axis rows %s; words where fast differs from exact: %d" % (
        b, [int(img[i].sum()) for i in (0, b // 4, b // 2, 3 * b // 4)], int((got["fast"] != got["exact"]).sum())))


GRIDS = {
    "rand31": lambda rng: (rng.random((31, 31)) < 0.006).astype(np.uint8),         # obstacle list: the map form
    "rand31_dense": lambda rng: (rng.random((31, 31)) < 0.05).astype(np.uint8),    # row traversal
    "rand48": lambda rng: (rng.random((48, 48)) < 0.02).astype(np.uint8),          # transposed copy
    "rand64": lambda rng: (rng.random((64, 64)) < 0.02).astype(np.uint8),          # two-level form
    "rand256": lambda rng: (rng.random((256, 256)) < 0.004).astype(np.uint8),      # two-level form, staged
}


@pytest.mark.parametrize("name", sorted(GRIDS))
def test_random_grids(ag, torch_, oracle, name):
    rng = np.random.default_rng(len(name) + 17)
    occ = GRIDS[name](rng)
    sc = scene(ag, torch_, grid_of(ag, occ))
    for engine in ENGINES:
        check_k2(sc, 256, 256, engine, what=name)
        check_oracle(oracle, sc, [oracle.grid_squares(occ)], 128, 96, engine, name)


def test_256_transposed_form(ag, torch_, oracle, monkeypatch):
    monkeypatch.setenv("AG_GRID_FORM", "transposed")
    rng = np.random.default_rng(23)
    occ = (rng.random((256, 256)) < 0.004).astype(np.uint8)
    sc = scene(ag, torch_, grid_of(ag, occ))
    assert sc.grid.bits_t is not None and sc.grid.hier is None
    for engine in ("fast", "exact"):
        check_k2(sc, 256, 256, engine, what="256 transposed")
        check_oracle(oracle, sc, [oracle.grid_squares(occ)], 96, 128, engine, "256 transposed")


def test_1024_map(ag, torch_, oracle):
    rng = np.random.default_rng(8)
    occ = (rng.random((1024, 1024)) < 0.002).astype(np.uint8)
    sc = scene(ag, torch_, grid_of(ag, occ))
    for engine in ENGINES:
        b = 32 if engine == "brute" else 256
        check_k2(sc, b, b, engine, what="1024")
        check_oracle(oracle, sc, [oracle.grid_squares(occ)], b // 2, b // 2, engine, "1024")


@pytest.mark.parametrize("kind", ["random", "clustered"])
def test_many_grids(ag, torch_, oracle, kind):
    """grid g's image equals K2 run on env ids of grid g, and the oracle on grid g"""
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(31)
    if kind == "random":
        grid = ag.BatchedOccupancyGrid.random(9, 64, 0.02, envs_per_grid=256, device="cuda", generator=gen, clear_base_cells=2)
    else:
        grid = ag.BatchedOccupancyGrid.clustered(8, 256, 6, 10, envs_per_grid=256, device="cuda", generator=gen)
    sc = scene(ag, torch, grid)
    occs = grid.device_grid().unpack()
    grids = [oracle.grid_squares(o) for o in occs]
    for engine in ENGINES:
        check_k2(sc, 96, 80, engine, what=kind)
        check_oracle(oracle, sc, grids, 48, 40, engine, kind)


def test_many_grids_unaligned_envs_per_grid(ag, torch_):
    """envs_per_grid not a multiple of 256 (K2 stages no grid), and the default 2^62 with three grids (no int64 env id
    selects grid 2): every grid still gets its image"""
    torch = torch_
    rng = np.random.default_rng(5)
    occs = np.stack([(rng.random((40, 40)) < 0.03).astype(np.uint8) for _ in range(3)])
    small = ag.BatchedOccupancyGrid(torch.as_tensor(occs, device="cuda"), 100)
    sc = scene(ag, torch, small)
    for engine in ENGINES:
        check_k2(sc, 64, 64, engine, what="envs_per_grid 100")
    huge = ag.DeviceGrid.from_device_matrices(torch.as_tensor(occs, device="cuda"))
    img = scene(ag, torch, huge).cspace_occupancy(64, packed=True)
    assert_words(img, sc.cspace_occupancy(64, packed=True), "envs_per_grid 2^62")


@pytest.mark.parametrize("b1", [1, 3])
@pytest.mark.parametrize("b2", [1, 31, 33, 100])
def test_ragged_shapes(ag, torch_, b1, b2):
    rng = np.random.default_rng(b1 * 1000 + b2)
    for occ in (None, (rng.random((64, 64)) < 0.03).astype(np.uint8)):
        sc = scene(ag, torch_, grid_of(ag, occ))
        for engine in ENGINES:
            got = check_k2(sc, b1, b2, engine, what="%d x %d" % (b1, b2))
            if b2 % 32:
                assert not (got[..., -1].cpu().numpy().view(np.uint32) >> np.uint32(b2 % 32)).any()   # padding bits 0


def test_free_count_and_packed_agree_with_bool(ag, torch_):
    torch = torch_
    gen = torch.Generator(device="cuda").manual_seed(3)
    grid = ag.BatchedOccupancyGrid.random(5, 31, 0.05, envs_per_grid=512, device="cuda", generator=gen)
    sc = scene(ag, torch, grid)
    for engine in ENGINES:
        for b1, b2 in ((200, 200), (7, 45)):
            img, fc = sc.cspace_occupancy(b1, b2, free_count=True, engine=engine)
            words, fc2 = sc.cspace_occupancy(b1, b2, packed=True, free_count=True, engine=engine)
            assert img.dtype == torch.bool and img.shape == (5, b1, b2) and fc.dtype == torch.int64 and fc.shape == (5,)
            assert torch.equal(fc, (~img).sum(dim=(1, 2))) and torch.equal(fc, fc2)
            assert_words(words, pack(img.cpu().numpy()), "packed vs bool")
            assert 0 < int(fc.sum()) < 5 * b1 * b2
    # written, not accumulated: a second call gives the same counts
    _, fa = sc.cspace_occupancy(64, free_count=True)
    _, fb = sc.cspace_occupancy(64, free_count=True)
    assert torch.equal(fa, fb)


@pytest.mark.parametrize("lo,step", [((2.0 ** 21, 2.0 ** 21 + 1.0), (0.01, 0.013)), ((6.0, 3.0), (-0.05, -0.021)),
                                     ((1.5e6, 0.1), (-0.3, 0.02))])
def test_lattices_outside_the_phase_range(ag, torch_, lo, step):
    """|q| >= 2^20 (outside the map's phase range) and negative steps: equal to K2"""
    for occ in (None, (np.random.default_rng(1).random((31, 31)) < 0.006).astype(np.uint8)):
        sc = scene(ag, torch_, grid_of(ag, occ))
        for engine in ENGINES:
            check_k2(sc, 130, 70, engine, lo=lo, step=step, what="lo %r step %r" % (lo, step))


@pytest.mark.parametrize("cached", [True, False])
def test_graph_capture(ag, torch_, cached):
    """a captured call equals the uncaptured one: on a grid whose map is cached, and with parameters no earlier call used
    (no cache entry can be made inside a capture: the general form runs)"""
    torch = torch_
    sc = scene(ag, torch, grid_of(ag, None))
    if not cached:
        sc.target_c = ag.Point(0.0321, -0.0654)             # the target is part of the map's key
    want = composed_occupancy(sc, (0.0, 0.0), steps(1024, 1024), 1024, 1024, ag.ENGINES["fast"]) if not cached else \
        sc.cspace_occupancy(1024, packed=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            words, fc = sc.cspace_occupancy(1024, packed=True, free_count=True)
    for _ in range(2):                                       # replays rewrite the counts
        g.replay()
        torch.cuda.synchronize()
        assert_words(words, want, "captured")
        popc = int(np.unpackbits(want.cpu().numpy().view(np.uint8)).sum())
        assert int(fc.item()) == 1024 * 1024 - popc


def test_torch_op_equals_object_api(ag, torch_):
    torch = torch_
    from abstract_gym_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(9)
    grid = ag.BatchedOccupancyGrid.random(3, 48, 0.02, envs_per_grid=256, device="cuda", generator=gen)
    sc = scene(ag, torch, grid)
    b1, b2 = 70, 90
    st = steps(b1, b2)
    for engine in ENGINES:
        want, want_fc = sc.cspace_occupancy(b1, b2, packed=True, free_count=True, engine=engine)
        words = torch.empty(3, b1, 3, dtype=torch.int32, device="cuda")
        fc = torch.empty(3, dtype=torch.int64, device="cuda")
        ops.cspace_occupancy(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), 0.0, st[0], b1, 0.0, st[1], b2, words, fc,
                             ag.ENGINES[engine])
        assert_words(words, want, "torch op")
        assert torch.equal(fc, want_fc)
    words2 = torch.empty_like(words)
    ops.cspace_occupancy(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), 0.0, st[0], b1, 0.0, st[1], b2, words2, None, 1)
    assert_words(words2, sc.cspace_occupancy(b1, b2, packed=True), "torch op, no counts")
    short = torch.empty(3 * b1 * 3 - 1, dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError):
        ops.cspace_occupancy(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), 0.0, st[0], b1, 0.0, st[1], b2, short, None, 1)
    with pytest.raises(RuntimeError):
        ops.cspace_occupancy(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), 0.0, st[0], b1, 0.0, st[1], b2, words,
                             fc[:2], 1)
    with pytest.raises((NotImplementedError, RuntimeError)):
        ops.cspace_occupancy(ops.pack_params(sc.params()), *ops.grid_args(sc.grid), 0.0, st[0], b1, 0.0, st[1], b2, words.cpu(),
                             None, 1)


_DEBUG_CHILD = r'''
import sys
import numpy as np, torch
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import abstract_gym_b200 as ag
from abstract_gym_b200 import _lib
from oracle import oracle as orc
from cspace_reference import oracle_image, pack, default_step
assert _lib.lib_path().endswith("_debug.so"), _lib.lib_path()
rng = np.random.default_rng(12)
z = torch.zeros(1, dtype=torch.float64, device="cuda")
for name, occs in (("scene0", None), ("rand64", [(rng.random((64, 64)) < 0.02).astype(np.uint8)]),
                   ("rand300", [(rng.random((300, 300)) < 0.004).astype(np.uint8) for _ in range(2)])):
    if occs is None:
        grid, grids = ag.OccupancyGrid(size=9, random_obstacle=False), [orc.manual_grid()]
    else:
        grid = ag.BatchedOccupancyGrid(torch.as_tensor(np.stack(occs), device="cuda"), 256)
        grids = [orc.grid_squares(o) for o in occs]
    sc = ag.BatchedScene(ag.BatchedTwoJointRobot(z, z.clone()), grid)
    b1, b2 = 40, 50
    st = (default_step(b1), default_step(b2))
    lo = (0.5 * st[0], 0.5 * st[1])
    want = np.stack([pack(oracle_image(orc, g, lo, st, b1, b2)) for g in grids])
    for engine in ("fast", "exact", "brute"):
        if engine == "brute" and name == "rand300":
            continue
        w, fc = sc.cspace_occupancy(b1, b2, lo=lo, step=st, packed=True, free_count=True, engine=engine)
        assert np.array_equal(w.cpu().numpy().view(np.uint32), want), (name, engine)
        assert int(fc.sum()) == len(grids) * b1 * b2 - int(np.unpackbits(want.view(np.uint8)).sum()), (name, engine)
print("debug cspace ok")
'''


def test_debug_bounds_build_cspace(ag, torch_):
    """the -DAG_DEBUG_BOUNDS library gives the oracle's images (child process); every occupancy kernel of it carries the
    index traps and the release library none (read from the machine code: no test sets a trap off)"""
    import subprocess
    import sys
    from abstract_gym_b200 import build as ag_build
    from test_gpu_parity import _traps_per_kernel
    lib = ag_build.build_debug()
    code = _DEBUG_CHILD % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, AG_LIB_PATH=lib), stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0 and "debug cspace ok" in r.stdout, r.stdout[-3000:]
    debug, release = _traps_per_kernel(lib), _traps_per_kernel(ag_build.LIB)
    kernels = [k for k in debug if "k_cspace" in k and "build" not in k]
    assert len(kernels) == 4 and all(debug[k] > 0 for k in kernels), {k: debug[k] for k in kernels}
    assert all(release[k] == 0 for k in kernels)
