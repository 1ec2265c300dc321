"""Reference forms of the free-space distance and the lattice descent (ag_cspace_distance / ag_cspace_descend /
BatchedScene.cspace_distance / cspace_path):
- distance_numpy: a multi-source unweighted scipy.sparse.csgraph.dijkstra(min_only=True) on the lattice graph (the
  4-neighbour edges of components_reference, seams where requested), -1 colliding, -2 free and unreachable;
- descend_numpy: the first-neighbour descent rule, pose by pose in Python;
- composed_distance: the form a user would write in torch: a level-synchronous BFS, the frontier moved one step with
  torch.roll per level (the seams masked where an axis does not wrap), until a level adds nothing.
tests/test_distance_cpu.py holds distance_numpy to a plain BFS; tests/test_distance_gpu.py and tools/distance_bench.py
hold the kernels to these."""
import numpy as np

from components_reference import _edges


def distance_numpy(free, goals, wrap):
    """free, goals: bool [..., b1, b2] -> int32 distances of the same shape.  Goals on colliding poses seed nothing."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import dijkstra
    free = np.asarray(free, dtype=bool)
    goals = np.asarray(goals, dtype=bool) & free
    n = free.size
    out = np.where(free.ravel(), -2, -1).astype(np.int64)
    src = np.flatnonzero(goals.ravel())
    if len(src):
        a, b = _edges(np.arange(n, dtype=np.int64).reshape(free.shape), free, wrap)
        g = coo_matrix((np.ones(len(a)), (a, b)), shape=(n, n)).tocsr()
        d = dijkstra(g, directed=False, indices=src, unweighted=True, min_only=True)
        reach = np.isfinite(d)
        out[reach] = d[reach].astype(np.int64)
    return out.astype(np.int32).reshape(free.shape)


def neighbours(i, j, b1, b2, wrap):
    """the neighbours of pose (i, j) in the descent order (i+1, j), (i-1, j), (i, j+1), (i, j-1); a seam only where the
    axis wraps"""
    out = []
    for u, v in ((i + 1, j), (i - 1, j), (i, j + 1), (i, j - 1)):
        if u in (-1, b1):
            if not wrap & 1:
                continue
            u %= b1
        if v in (-1, b2):
            if not wrap & 2:
                continue
            v %= b2
        out.append((u, v))
    return out


def descend_numpy(dist, start, grid, max_len, wrap):
    """dist int32 [n_grids, b1, b2]; start int [M] grid-local indices; grid int [M] -> (path int32 [M, max_len],
    length int32 [M])"""
    dist = np.asarray(dist)
    n_grids, b1, b2 = dist.shape
    m = len(start)
    path = np.full((m, max_len), -1, dtype=np.int32)
    length = np.zeros(m, dtype=np.int32)
    for q in range(m):
        g, s = int(grid[q]), int(start[q])
        if not (0 <= g < n_grids and 0 <= s < b1 * b2) or dist[g].flat[s] < 0:
            continue
        i, j = divmod(s, b2)
        d = int(dist[g, i, j])
        path[q, 0], k = s, 1
        while d > 0 and k < max_len:
            i, j = next((u, v) for u, v in neighbours(i, j, b1, b2, wrap) if dist[g, u, v] == d - 1)
            d -= 1
            path[q, k] = i * b2 + j
            k += 1
        length[q] = k
    return path, length


def composed_distance(free, goals, wrap):
    """free, goals: bool torch tensors [n_grids, b1, b2] on the device -> (int32 distances, BFS levels)"""
    import torch
    n, b1, b2 = free.shape
    front = goals & free
    dist = torch.where(free, -2, -1).to(torch.int32)
    dist[front] = 0
    unseen = free & ~front
    level = 0
    while True:
        nb = torch.zeros_like(front)
        for dim, bit, b in ((1, 1, b1), (2, 2, b2)):
            for shift in (1, -1):
                r = torch.roll(front, shift, dim)
                if not wrap & bit:                      # the rolled-in row / column is across a seam that does not exist
                    r.narrow(dim, 0 if shift == 1 else b - 1, 1).fill_(False)
                nb |= r
        front = nb & unseen
        if not bool(front.any()):
            return dist, level
        level += 1
        dist[front] = level
        unseen &= ~front
