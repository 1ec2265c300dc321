"""Reference compositions of a configuration-space occupancy image (BatchedScene.cspace_occupancy):
- on the CPU oracle: the lattice's poses built with numpy and Scene.collision_check (scenario/scene_0.py:60-76) at each;
- on the device: the same poses in torch, ag_collision_check (K2) on env ids of each grid, packing in torch.
tests/test_cspace_cpu.py checks the lattice and the oracle composition; tests/test_cspace_gpu.py and tools/cspace_bench.py
hold the kernel to them."""
import math

import numpy as np


def default_step(b):
    return 2.0 * math.pi / b


def lattice(lo, step, b):
    """lo + i * step for i = 0 .. b-1, float64: one rounding for the product, one for the sum (numpy never fuses)"""
    return np.float64(lo) + np.arange(b, dtype=np.float64) * np.float64(step)


def pack(img):
    """bool [..., b1, b2] -> uint32 words [..., b1, ceil(b2/32)]: pose j is bit j % 32 of word j // 32, padding 0"""
    img = np.asarray(img, dtype=bool)
    b2 = img.shape[-1]
    w = (b2 + 31) // 32
    pad = np.zeros(img.shape[:-1] + (w * 32,), dtype=np.uint64)
    pad[..., :b2] = img
    bits = pad.reshape(img.shape[:-1] + (w, 32)) << np.arange(32, dtype=np.uint64)
    return bits.sum(axis=-1).astype(np.uint32)


def oracle_image(orc, grid, lo, step, b1, b2):
    """bool [b1, b2] of one grid ((squares, cell_index) from the oracle)"""
    q1, q2 = lattice(lo[0], step[0], b1), lattice(lo[1], step[1], b2)
    hit, _, _ = orc.collision_batch(np.repeat(q1, b2), np.tile(q2, b1), grid[0], want_first_hit=False)
    return hit.reshape(b1, b2) != 0


def composed_occupancy(sc, lo, step, b1, b2, engine, chunk=1 << 24):
    """The image as a user composes it from K2: int32 words [n_grids, b1, W] on the device, the layout of
    cspace_occupancy(packed=True).  Envs of grid g are the env ids
    e with (e // envs_per_grid) % n_grids == g; one 'round' of n_grids * envs_per_grid consecutive ids holds
    envs_per_grid of each grid, so each K2 launch covers whole rounds (env_id0 a multiple of the round) and every pose
    is checked on an env id of its own grid.  Single-grid scenes use rounds of `chunk` poses."""
    import torch
    from abstract_gym_b200 import _lib
    from abstract_gym_b200._device import ptr, stream_ptr
    dev, grid = sc.device, sc.grid
    n = int(grid.n_grids)
    per = min(int(grid.envs_per_grid), chunk) if n == 1 else int(grid.envs_per_grid)
    P = b1 * b2
    rounds = (P + per - 1) // per
    step_rounds = max(1, chunk // (n * per))
    q1 = lo[0] + torch.arange(b1, dtype=torch.float64, device=dev) * step[0]
    q2 = lo[1] + torch.arange(b2, dtype=torch.float64, device=dev) * step[1]
    hit = torch.empty(n, rounds * per, dtype=torch.uint8, device=dev)
    lib, g, p = sc._lib, grid.c_struct(), sc.params()
    for r0 in range(0, rounds, step_rounds):
        r1 = min(rounds, r0 + step_rounds)
        k = torch.arange(r0 * per, r1 * per, device=dev).clamp_(max=P - 1)   # lattice pose of each env (past P: pose P-1)
        j1 = q1[k // b2].view(r1 - r0, 1, per).expand(r1 - r0, n, per).contiguous()
        j2 = q2[k % b2].view(r1 - r0, 1, per).expand(r1 - r0, n, per).contiguous()
        h = torch.empty(j1.numel(), dtype=torch.uint8, device=dev)
        _lib.check(lib.ag_collision_check(p, g, ptr(j1), ptr(j2), ptr(h), None, j1.numel(), r0 * n * per, engine,
                                          stream_ptr(dev)), "ag_collision_check")
        hit[:, r0 * per:r1 * per] = h.view(r1 - r0, n, per).transpose(0, 1).reshape(n, -1)
    img = hit[:, :P].view(n, b1, b2)
    w = (b2 + 31) // 32
    padded = torch.zeros(n, b1, w * 32, dtype=torch.int64, device=dev)
    padded[:, :, :b2] = img
    words = (padded.view(n, b1, w, 32) << torch.arange(32, device=dev)).sum(dim=-1)
    return torch.where(words >= 1 << 31, words - (1 << 32), words).to(torch.int32)
