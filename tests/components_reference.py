"""Reference forms of the free-space components of an occupancy image (ag_cspace_components /
BatchedScene.cspace_components / BatchedScene.cspace_component_of):
- label_numpy: a hook-and-jump union-find in numpy giving the canonical labels (-1 colliding, else the smallest grid-local
  row-major index of the component), 4-neighbour, with the requested seams;
- component_of_numpy: the lookup rule of cspace_component_of;
- composed_components: the form a user would write in torch: min-label propagation over the 4 neighbours (torch.roll,
  the seams masked where an axis does not wrap), then pointer jumping L = L[L] until fixpoint, until nothing changes.
tests/test_components_cpu.py holds label_numpy to a plain BFS; tests/test_components_gpu.py and tools/components_bench.py
hold the kernels to these."""
import numpy as np


def _edges(idx, free, wrap):
    """index pairs of the 4-neighbour edges between free poses, per grid, seams included where requested"""
    b1, b2 = free.shape[-2:]
    pairs = [(idx[..., :-1, :], idx[..., 1:, :], free[..., :-1, :] & free[..., 1:, :]),
             (idx[..., :, :-1], idx[..., :, 1:], free[..., :, :-1] & free[..., :, 1:])]
    if wrap & 1 and b1 > 1:
        pairs.append((idx[..., -1, :], idx[..., 0, :], free[..., -1, :] & free[..., 0, :]))
    if wrap & 2 and b2 > 1:
        pairs.append((idx[..., :, -1], idx[..., :, 0], free[..., :, -1] & free[..., :, 0]))
    a = np.concatenate([p[m] for p, _, m in pairs])
    b = np.concatenate([q[m] for _, q, m in pairs])
    return a, b


def label_numpy(free, wrap):
    """free: bool [..., b1, b2] (True = free pose) -> int32 labels of the same shape.  Every root only ever hooks under a
    smaller root, so each node's parent is <= the node and the final root of a component is its smallest index."""
    free = np.asarray(free, dtype=bool)
    b1, b2 = free.shape[-2:]
    n = free.size
    idx = np.arange(n, dtype=np.int64).reshape(free.shape)
    a, b = _edges(idx, free, wrap)
    L = np.where(free.ravel(), np.arange(n, dtype=np.int64), -1)
    nodes = np.flatnonzero(free.ravel())
    while True:
        ra, rb = L[a], L[b]
        live = ra != rb                                  # edges inside one tree stay there
        if not live.any():
            break
        a, b, ra, rb = a[live], b[live], ra[live], rb[live]
        np.minimum.at(L, np.maximum(ra, rb), np.minimum(ra, rb))       # hook: the larger root under the smaller
        while True:                                      # jump until every node points at its root
            up = L[L[nodes]]
            if np.array_equal(up, L[nodes]):
                break
            L[nodes] = up
    per = b1 * b2
    local = L - (idx.ravel() // per) * per
    return np.where(free.ravel(), local, -1).astype(np.int32).reshape(free.shape)


def spiral(b1, b2):
    """bool [b1, b2]: a width-1 corridor spiralling clockwise in from pose (0, 0) (its minimum index, at one end), with a
    wall of width 1 between turns: a single path of about b1 * b2 / 2 poses"""
    free = np.zeros((b1, b2), dtype=bool)
    i, j, d = 0, 0, 0
    steps = ((0, 1), (1, 0), (0, -1), (-1, 0))
    free[0, 0] = True

    def ok(u, v, fu, fv):                               # inside, and touching nothing but the pose it comes from
        if not (0 <= u < b1 and 0 <= v < b2) or free[u, v]:
            return False
        return all(not (0 <= x < b1 and 0 <= y < b2 and free[x, y]) or (x, y) == (fu, fv)
                   for x, y in ((u + 1, v), (u - 1, v), (u, v + 1), (u, v - 1)))
    turns = 0
    while turns < 2:
        u, v = i + steps[d][0], j + steps[d][1]
        if ok(u, v, i, j):
            free[u, v], i, j, turns = True, u, v, 0
        else:
            d, turns = (d + 1) % 4, turns + 1
    return free


def special_images(b1, b2):
    """{name: bool [b1, b2] free image} of adversarial cases (b1, b2 >= 6)"""
    out = {"spiral": spiral(b1, b2)}
    comb = np.zeros((b1, b2), dtype=bool)               # a serpentine: free rows joined at alternate ends
    comb[::2] = True
    comb[1::4, -1] = True
    comb[3::4, 0] = True
    out["comb"] = comb
    out["checkerboard"] = (np.add.outer(np.arange(b1), np.arange(b2)) % 2) == 0
    out["all_free"] = np.ones((b1, b2), dtype=bool)
    out["all_colliding"] = np.zeros((b1, b2), dtype=bool)
    seam = np.zeros((b1, b2), dtype=bool)
    seam[0, 3] = seam[-1, 3] = True                     # joined only through the joint_1 seam
    seam[b1 // 2, 0] = seam[b1 // 2, -1] = True         # only through the joint_2 seam
    out["seams"] = seam
    corner = np.zeros((b1, b2), dtype=bool)
    corner[0, 0] = corner[0, -1] = corner[-1, 0] = corner[-1, -1] = True   # one component only on the torus
    out["corners"] = corner
    return out


def grid_of_env(m, env_id0, envs_per_grid, n_grids):
    """grid of motion / pose m: ((env_id0 + m) // envs_per_grid) % n_grids (ag_check_motion's rule)"""
    return ((env_id0 + np.arange(m, dtype=np.int64)) // envs_per_grid) % n_grids


def component_of_numpy(labels, q, grids, lo, step, wrap):
    """labels [n_grids, b1, b2]; q [M, 2] float64; grids [M]: the label at the nearest lattice pose, -1 off the lattice.
    Per axis k = floor((q - lo) / step + 0.5) in float64; a wrapping axis takes k mod b, any other needs 0 <= k < b; a NaN
    or infinite q gives -1."""
    labels = np.asarray(labels)
    q = np.asarray(q, dtype=np.float64).reshape(-1, 2)
    ok = np.ones(len(q), dtype=bool)
    ks = []
    with np.errstate(invalid="ignore", over="ignore"):
        for a in range(2):
            b = labels.shape[1 + a]
            k = np.floor((q[:, a] - np.float64(lo[a])) / np.float64(step[a]) + 0.5)
            ok &= np.isfinite(k)
            if wrap >> a & 1:
                k = np.fmod(k, b)
                k = np.where(k < 0, k + b, k)
            else:
                ok &= (k >= 0) & (k < b)
            ks.append(np.where(ok, k, 0).astype(np.int64))
    out = labels[np.asarray(grids), ks[0], ks[1]]
    return np.where(ok, out, -1).astype(np.int32)


def composed_components(free, wrap):
    """free: bool torch tensor [n_grids, b1, b2] on the device -> (int32 labels, outer iterations).  Each iteration takes
    the minimum label over a pose and its 4 neighbours, then jumps L = L[L] until fixpoint; it stops when an iteration
    changes nothing.  Labels are global indices during the loop (so L[L] can index), grid-local at the end."""
    import torch
    n, b1, b2 = free.shape
    N = free.numel()
    dt = torch.int32 if N < 2 ** 31 - 1 else torch.int64
    big = torch.tensor([N], dtype=dt, device=free.device)                # colliding poses: larger than any index
    idx = torch.arange(N, dtype=dt, device=free.device).view(n, b1, b2)
    L = torch.where(free, idx, big)
    iters = 0
    while True:
        iters += 1
        M = L
        for dim, bit, b in ((1, 1, b1), (2, 2, b2)):
            for shift in (1, -1):
                nb = torch.roll(L, shift, dim)
                if not wrap & bit:                      # the rolled-in row / column is across a seam that does not exist
                    nb.narrow(dim, 0 if shift == 1 else b - 1, 1).fill_(N)
                M = torch.minimum(M, nb)
        M = torch.where(free, M, big).flatten()
        ext = torch.cat([M, big])
        while True:
            up = ext[ext]
            if torch.equal(up, ext):
                break
            ext = up
        M = ext[:N].view(n, b1, b2)
        if torch.equal(M, L):
            break
        L = M
    return torch.where(free, L - (idx // (b1 * b2)) * (b1 * b2), -1).to(torch.int32), iters


def pack_words(colliding):
    """bool torch [..., b1, b2] (True = colliding) -> int32 words [..., b1, ceil(b2/32)], the layout of
    cspace_occupancy(packed=True), padding bits 0"""
    import torch
    b2 = colliding.shape[-1]
    w = (b2 + 31) // 32
    pad = torch.zeros(colliding.shape[:-1] + (w * 32,), dtype=torch.int64, device=colliding.device)
    pad[..., :b2] = colliding
    words = (pad.view(colliding.shape[:-1] + (w, 32)) << torch.arange(32, device=colliding.device)).sum(dim=-1)
    return torch.where(words >= 1 << 31, words - (1 << 32), words).to(torch.int32)


def unpack_free(words, b2):
    """int32 words [..., b1, W] -> bool [..., b1, b2], True = free"""
    import torch
    shifts = torch.arange(32, dtype=torch.int32, device=words.device)
    bits = ((words.unsqueeze(-1) >> shifts) & 1).reshape(words.shape[:-1] + (-1,))[..., :b2]
    return bits == 0
