// ag_cdist.cu -- distance fields and lattice paths over the free poses of a configuration-space occupancy image, per grid
// (ag_cspace_distance, ag_cspace_descend; DESIGN.md "Configuration-space distance").
//
// Input: the words ag_cspace_occupancy writes, [n_grids][b1][W] uint32, W = ceil(b2/32), 1 = colliding, and a goal image
// in the same layout, 1 = goal; padding bits are ignored.  Adjacency is that of ag_cspace_components (4 neighbours, the
// seams where wrap asks for them, grids never connect).
// Output: dist [n_grids][b1][b2] int32: -1 colliding, -2 free but no free goal in its component, else the fewest steps
// through free poses to a free goal -- the multi-source BFS distance, unique, so independent of scheduling.
//
// Tile relaxation, three kernels:
//   k_dist_init   -- 0 at free goals, INT32_MAX at other free poses, -1 at colliding ones.
//   k_dist_relax  -- one pass: a warp loads a T x T tile of dist and its one-pose halo ring (seams included) into shared
//                    memory, alternates row and column min-scans d = min(d, d_nbr + 1) until nothing in the tile changes,
//                    writes back the poses it lowered and stamps the tile with the pass number.  From the second pass on,
//                    a tile is processed only when one of its four neighbour tiles (itself across a seam of a one-tile
//                    axis) was stamped by the previous pass, and the whole pass returns at once when the previous pass
//                    changed nothing.
//   k_dist_finish -- INT32_MAX becomes -2; the largest distance of each grid (max_dist).
// Why the fixpoint is the BFS distance: every value is the length of a real path to a goal, and values only decrease, so a
// stale halo read (another warp lowering that pose in the same pass) only delays a decrease; it never makes a value wrong.
// A tile is written by its own warp only.  When tile B lowers a pose in its last changing pass q, every neighbour A sees
// B's stamp q throughout pass q + 1 and relaxes against B's final values; later decreases of A keep d_A <= d_B + 1.  So
// when a pass changes nothing, d_u <= d_v + 1 holds on every edge, which with d = 0 exactly at the free goals and every
// value a path length is the BFS distance.
//
// The host launches passes in groups of AG_DIST_SYNC_PASSES and reads the change count of the group's last pass after
// each group (one cudaMemcpyAsync + cudaStreamSynchronize), stopping when it is 0.
//
// k_dist_descend -- one thread per query: from the start, the first neighbour in the order (i+1, j), (i-1, j),
// (i, j+1), (i, j-1) whose distance is one less, until distance 0 or max_len poses.
#include <climits>

#include "ag_rollout.cuh"

using namespace agd;

namespace {

constexpr int T = 32;                        // tile side (one lane per row, then per column)
constexpr int SP = T + 3;                    // shared row pitch: odd, so the row and the column scans are conflict-free
constexpr int WARPS = 4;                     // tiles per block of k_dist_relax
constexpr int32_t WALL = INT32_MAX;          // colliding, or no pose (in shared memory)
constexpr int32_t UNSEEN = INT32_MAX - 1;    // free, no goal reached yet (INT32_MAX in global memory)
constexpr int CHUNK = 16 * AG_BLOCK;         // poses per block iteration of k_dist_init / k_dist_finish
constexpr int64_t MAX_BLOCKS = 1 << 20;
constexpr int RING = 4;                      // change counters: pass p adds to slot p % 4 and clears slot (p + 1) % 4
constexpr int AG_DIST_SYNC_PASSES = 16;

struct DistDev {
    const uint32_t *bits, *goals;            // [n_grids][b1][W]
    int32_t *dist;                           // [n_grids][b1][b2]
    int32_t *max_dist;                       // [n_grids] or nullptr (set to -1 before k_dist_finish)
    int32_t *stamp;                          // [n_grids][tiles_r][tiles_c]: the last pass that changed the tile, -1 none
    unsigned int *count;                     // [RING] tiles changed per pass
    int64_t n_grids, poses;                  // poses per grid: b1 * b2 (< 2^31 - 1)
    int32_t b1, b2, W, wrap;
    int32_t tiles_r, tiles_c;
};

__global__ void __launch_bounds__(AG_BLOCK) k_dist_init(const __grid_constant__ DistDev D) {
    const int64_t chunks = (D.poses + CHUNK - 1) / CHUNK;
    for (int64_t C = blockIdx.x; C < D.n_grids * chunks; C += gridDim.x) {
        const int64_t g = C / chunks;
        const int32_t p1 = (int32_t)min(D.poses, (C % chunks + 1) * CHUNK);
        for (int32_t p = (int32_t)(C % chunks) * CHUNK + threadIdx.x; p < p1; p += blockDim.x) {
            const int32_t i = p / D.b2, j = p % D.b2;
            const int64_t o = (g * D.b1 + i) * D.W + (j >> 5);
            AG_CHECK_INDEX(o, D.n_grids * D.b1 * D.W);
            const uint32_t col = (D.bits[o] >> (j & 31)) & 1u, goal = (D.goals[o] >> (j & 31)) & 1u;
            AG_CHECK_INDEX(g * D.poses + p, D.n_grids * D.poses);
            D.dist[g * D.poses + p] = col ? -1 : (goal ? 0 : INT32_MAX);
        }
    }
}

// dist of pose (i, j) of one grid, i in [-1, b1], j in [-1, b2] (-1 and b are across the seams), in the shared encoding
__device__ __forceinline__ int32_t load_pose(const DistDev &D, const int32_t *G, int32_t i, int32_t j) {
    if (i < 0 || i == D.b1) {
        if (!(D.wrap & 1)) return WALL;
        i = i < 0 ? D.b1 - 1 : 0;
    }
    if (j < 0 || j == D.b2) {
        if (!(D.wrap & 2)) return WALL;
        j = j < 0 ? D.b2 - 1 : 0;
    }
    AG_CHECK_INDEX((int64_t)i * D.b2 + j, D.poses);
    const int32_t v = G[(int64_t)i * D.b2 + j];
    return v < 0 ? WALL : (v == INT32_MAX ? UNSEEN : v);
}

// whether tile (tr, tc) has a neighbour tile, across a seam where the axis wraps, that pass `prev` changed
__device__ __forceinline__ bool neighbour_changed(const DistDev &D, const int32_t *stamp, int tr, int tc, int32_t prev) {
    const int lane = threadIdx.x & 31;
    bool hit = false;
    if (lane < 4) {
        int r = tr + (lane == 0) - (lane == 1), c = tc + (lane == 2) - (lane == 3);
        const bool wr = (D.wrap & 1) && D.b1 > 1, wc = (D.wrap & 2) && D.b2 > 1;
        bool ok = true;
        if (r < 0 || r == D.tiles_r) { ok = wr; r = r < 0 ? D.tiles_r - 1 : 0; }
        if (c < 0 || c == D.tiles_c) { ok = ok && wc; c = c < 0 ? D.tiles_c - 1 : 0; }
        if (ok) {
            AG_CHECK_INDEX(r * D.tiles_c + c, (int64_t)D.tiles_r * D.tiles_c);
            hit = stamp[r * D.tiles_c + c] == prev;
        }
    }
    return __any_sync(0xFFFFFFFFu, hit);
}

// d = min(d, previous + 1) along one line of n free-or-wall poses, both ways; the ends see the poses before and after
__device__ __forceinline__ bool scan_line(int32_t *s, int stride, int n) {
    bool ch = false;
    int32_t prev = s[0];
    for (int k = 1; k <= n; ++k) {
        int32_t v = s[k * stride];
        const int32_t cand = min(prev, UNSEEN) + 1;          // WALL and UNSEEN neighbours offer nothing
        if (v != WALL && cand < v) { v = cand; s[k * stride] = v; ch = true; }
        prev = v;
    }
    prev = s[(n + 1) * stride];
    for (int k = n; k >= 1; --k) {
        int32_t v = s[k * stride];
        const int32_t cand = min(prev, UNSEEN) + 1;
        if (v != WALL && cand < v) { v = cand; s[k * stride] = v; ch = true; }
        prev = v;
    }
    return ch;
}

// one relaxation pass; one warp per tile, tiles numbered grid by grid
__global__ void __launch_bounds__(WARPS * 32) k_dist_relax(const __grid_constant__ DistDev D, int32_t pass) {
    __shared__ int32_t s_tile[WARPS][(T + 2) * SP];
    if (blockIdx.x == 0 && threadIdx.x == 0) D.count[(pass + 1) % RING] = 0u;
    if (pass > 0 && D.count[(pass - 1) % RING] == 0u) return;       // converged: the previous pass changed nothing
    const int lane = threadIdx.x & 31;
    int32_t *s = s_tile[threadIdx.x >> 5];
    const int64_t tiles = (int64_t)D.tiles_r * D.tiles_c;
    for (int64_t Ti = (int64_t)blockIdx.x * WARPS + (threadIdx.x >> 5); Ti < D.n_grids * tiles;
         Ti += (int64_t)gridDim.x * WARPS) {
        const int64_t g = Ti / tiles;
        const int t = (int)(Ti % tiles), tr = t / D.tiles_c, tc = t % D.tiles_c;
        if (pass > 0 && !neighbour_changed(D, D.stamp + g * tiles, tr, tc, pass - 1)) continue;   // warp-uniform
        const int32_t i0 = tr * T, j0 = tc * T;
        const int nr = min(T, D.b1 - i0), nc = min(T, D.b2 - j0);
        int32_t *G = D.dist + g * D.poses;
        // the tile (WALL outside the grid), then its halo ring; lane = column
        int32_t orig[T];
#pragma unroll
        for (int r = 0; r < T; ++r) {
            orig[r] = (r < nr && lane < nc) ? load_pose(D, G, i0 + r, j0 + lane) : WALL;
            s[(r + 1) * SP + lane + 1] = orig[r];
        }
        __syncwarp();
        if (lane < nc) {
            s[lane + 1] = load_pose(D, G, i0 - 1, j0 + lane);
            s[(nr + 1) * SP + lane + 1] = load_pose(D, G, i0 + nr, j0 + lane);
        }
        if (lane < nr) {
            s[(lane + 1) * SP] = load_pose(D, G, i0 + lane, j0 - 1);
            s[(lane + 1) * SP + nc + 1] = load_pose(D, G, i0 + lane, j0 + nc);
        }
        __syncwarp();
        bool changed = false;
        for (;;) {
            bool ch = lane < nr && scan_line(s + (lane + 1) * SP, 1, nc);       // row lane + 1
            __syncwarp();
            ch |= lane < nc && scan_line(s + lane + 1, SP, nr);                  // column lane + 1
            __syncwarp();
            if (!__any_sync(0xFFFFFFFFu, ch)) break;
            changed = true;
        }
        if (changed) {                                                           // warp-uniform
#pragma unroll
            for (int r = 0; r < T; ++r) {
                const int32_t v = s[(r + 1) * SP + lane + 1];
                if (r < nr && lane < nc && v != orig[r]) {
                    const int64_t o = (int64_t)(i0 + r) * D.b2 + j0 + lane;
                    AG_CHECK_INDEX(o, D.poses);
                    G[o] = v;
                }
            }
            if (lane == 0) {
                AG_CHECK_INDEX(g * tiles + t, D.n_grids * tiles);
                D.stamp[g * tiles + t] = pass;
                atomicAdd(D.count + pass % RING, 1u);
            }
        }
        __syncwarp();                                                            // s is rewritten by the next tile
    }
}

__global__ void __launch_bounds__(AG_BLOCK) k_dist_finish(const __grid_constant__ DistDev D) {
    __shared__ int s_max;
    const int64_t chunks = (D.poses + CHUNK - 1) / CHUNK;
    if (threadIdx.x == 0) s_max = -1;
    __syncthreads();
    for (int64_t C = blockIdx.x; C < D.n_grids * chunks; C += gridDim.x) {
        const int64_t g = C / chunks;
        int32_t *G = D.dist + g * D.poses;
        const int64_t p1 = min(D.poses, (C % chunks + 1) * CHUNK);
        int m = -1;
        for (int64_t p = (C % chunks) * CHUNK + threadIdx.x; p < p1; p += blockDim.x) {
            const int32_t v = G[p];
            if (v == INT32_MAX) G[p] = -2;
            else m = max(m, v);
        }
        if (D.max_dist != nullptr) {                                             // block-uniform
            m = __reduce_max_sync(0xFFFFFFFFu, m);
            if ((threadIdx.x & 31) == 0 && m >= 0) atomicMax(&s_max, m);
            __syncthreads();
            if (threadIdx.x == 0 && s_max >= 0) {
                AG_CHECK_INDEX(g, D.n_grids);
                atomicMax(D.max_dist + g, s_max);
                s_max = -1;
            }
            __syncthreads();
        }
    }
}

struct DescendDev {
    const int32_t *dist;                     // [n_grids][b1][b2]
    const int32_t *start;                    // [m] grid-local row-major indices
    const int64_t *grid;                     // [m]
    int32_t *path;                           // [m][max_len]
    int32_t *length;                         // [m]
    int64_t n_grids, poses, m;
    int32_t b1, b2, wrap, max_len;
};

__global__ void __launch_bounds__(AG_BLOCK) k_dist_descend(const __grid_constant__ DescendDev D) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= D.m) return;
    int32_t *path = D.path + q * D.max_len;
    const int64_t g = D.grid[q];
    int32_t cur = D.start[q], len = 0;
    if (g >= 0 && g < D.n_grids && cur >= 0 && cur < D.poses) {
        const int32_t *G = D.dist + g * D.poses;
        AG_CHECK_INDEX(cur, D.poses);
        int32_t d = G[cur];
        if (d >= 0) {
            path[0] = cur;
            len = 1;
            while (d > 0 && len < D.max_len) {
                const int32_t i = cur / D.b2, j = cur % D.b2;
                int32_t next = -1;
                for (int k = 0; k < 4 && next < 0; ++k) {
                    int32_t u = i + (k == 0) - (k == 1), v = j + (k == 2) - (k == 3);
                    if (u < 0 || u == D.b1) {
                        if (!(D.wrap & 1)) continue;
                        u = u < 0 ? D.b1 - 1 : 0;
                    }
                    if (v < 0 || v == D.b2) {
                        if (!(D.wrap & 2)) continue;
                        v = v < 0 ? D.b2 - 1 : 0;
                    }
                    AG_CHECK_INDEX(u * D.b2 + v, D.poses);
                    if (G[u * D.b2 + v] == d - 1) next = u * D.b2 + v;
                }
                if (next < 0) break;                 // not a distance field: no neighbour is one step closer
                cur = next;
                --d;
                AG_CHECK_INDEX(len, D.max_len);
                path[len++] = cur;
            }
        }
    }
    for (int32_t k = len; k < D.max_len; ++k) path[k] = -1;
    D.length[q] = len;
}

template <typename Kernel, typename Dev>
ag_status launch(Kernel k, int64_t work, const Dev &D, cudaStream_t s) {
    k<<<(unsigned)(work < MAX_BLOCKS ? work : MAX_BLOCKS), AG_BLOCK, 0, s>>>(D);
    return launched();
}

// the shape checks both entry points share
ag_status check_lattice(int64_t n_grids, int32_t b1, int32_t b2) {
    if (n_grids < 0 || b1 < 1 || b2 < 1) return AG_ERR_SHAPE;
    const int64_t poses = (int64_t)b1 * b2;
    if (poses > INT32_MAX - 1 || (n_grids > 0 && poses > INT64_MAX / n_grids)) return AG_ERR_SHAPE;   // distances < poses
    return AG_OK;
}

ag_status relax_until_stable(const DistDev &D, cudaStream_t s) {
    const int64_t tiles = D.n_grids * D.tiles_r * D.tiles_c;
    int resident = 0;
    ag_status st = resident_blocks(k_dist_relax, WARPS * 32, 0, &resident);
    if (st != AG_OK) return st;
    const int64_t want = (tiles + WARPS - 1) / WARPS;
    const unsigned blocks = (unsigned)(want < resident ? want : (resident > 0 ? resident : 1));
    unsigned int changed = 1u;
    for (int32_t pass = 0; changed != 0u;) {
        for (int k = 0; k < AG_DIST_SYNC_PASSES; ++k, ++pass) {
            k_dist_relax<<<blocks, WARPS * 32, 0, s>>>(D, pass);
            st = launched();
            if (st != AG_OK) return st;
        }
        cudaError_t e = cudaMemcpyAsync(&changed, D.count + (pass - 1) % RING, sizeof(changed), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return (ag_status)e;
    }
    return AG_OK;
}

}  // namespace

extern "C" ag_status ag_cspace_distance(const uint32_t *bits, const uint32_t *goals, int64_t n_grids, int32_t b1, int32_t b2,
                                        int32_t wrap, int32_t *dist, int32_t *max_dist, void *stream) {
    ag_status st = check_lattice(n_grids, b1, b2);
    if (st != AG_OK) return st;
    if (wrap & ~3) return AG_ERR_MODE;
    if (n_grids == 0) return AG_OK;
    if (!bits || !goals || !dist) return AG_ERR_NULL;
    if (((uintptr_t)bits % 4) || ((uintptr_t)goals % 4) || ((uintptr_t)dist % 4) || ((uintptr_t)max_dist % 4))
        return AG_ERR_ALIGN;
    cudaStream_t s = (cudaStream_t)stream;
    // convergence is read back on the host: nothing of this call can be captured in a graph
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaError_t e = cudaStreamIsCapturing(s, &cap);
    if (e != cudaSuccess) return (ag_status)e;
    if (cap != cudaStreamCaptureStatusNone) return (ag_status)cudaErrorStreamCaptureUnsupported;
    DistDev D;
    D.bits = bits; D.goals = goals; D.dist = dist; D.max_dist = max_dist;
    D.n_grids = n_grids; D.poses = (int64_t)b1 * b2;
    D.b1 = b1; D.b2 = b2; D.W = (b2 + 31) / 32; D.wrap = wrap;
    D.tiles_r = (b1 + T - 1) / T; D.tiles_c = (b2 + T - 1) / T;
    const int64_t tiles = n_grids * D.tiles_r * D.tiles_c;
    unsigned int *scratch = nullptr;                 // RING change counters, then the tile stamps
    e = cudaMallocAsync(&scratch, (size_t)(RING + tiles) * 4, s);
    if (e != cudaSuccess) return (ag_status)e;
    D.count = scratch;
    D.stamp = reinterpret_cast<int32_t *>(scratch + RING);
    e = cudaMemsetAsync(D.count, 0, RING * 4, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(D.stamp, 0xFF, (size_t)tiles * 4, s);
    if (e == cudaSuccess && max_dist != nullptr) e = cudaMemsetAsync(max_dist, 0xFF, (size_t)n_grids * 4, s);
    st = (ag_status)e;
    const int64_t chunks = n_grids * ((D.poses + CHUNK - 1) / CHUNK);
    if (st == AG_OK) st = launch(k_dist_init, chunks, D, s);
    if (st == AG_OK) st = relax_until_stable(D, s);
    if (st == AG_OK) st = launch(k_dist_finish, chunks, D, s);
    cudaFreeAsync(scratch, s);
    return st;
}

extern "C" ag_status ag_cspace_descend(const int32_t *dist, int64_t n_grids, int32_t b1, int32_t b2, int32_t wrap,
                                       const int32_t *start, const int64_t *grid, int64_t m, int32_t max_len, int32_t *path,
                                       int32_t *length, void *stream) {
    ag_status st = check_lattice(n_grids, b1, b2);
    if (st != AG_OK) return st;
    if (m < 0 || max_len < 1 || m > INT64_MAX / max_len) return AG_ERR_SHAPE;
    if (wrap & ~3) return AG_ERR_MODE;
    if (m == 0) return AG_OK;
    if (!dist || !start || !grid || !path || !length) return AG_ERR_NULL;
    if (((uintptr_t)dist % 4) || ((uintptr_t)start % 4) || ((uintptr_t)grid % 8) || ((uintptr_t)path % 4) ||
        ((uintptr_t)length % 4))
        return AG_ERR_ALIGN;
    DescendDev D;
    D.dist = dist; D.start = start; D.grid = grid; D.path = path; D.length = length;
    D.n_grids = n_grids; D.poses = (int64_t)b1 * b2; D.m = m;
    D.b1 = b1; D.b2 = b2; D.wrap = wrap; D.max_len = max_len;
    k_dist_descend<<<blocks_for(m), AG_BLOCK, 0, (cudaStream_t)stream>>>(D);
    return launched();
}
