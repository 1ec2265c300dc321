// ag_ccl.cu -- connected components of the free poses of a configuration-space occupancy image, per grid
// (ag_cspace_components, DESIGN.md "Free-space components").
//
// Input: the words ag_cspace_occupancy writes, [n_grids][b1][W] uint32, W = ceil(b2/32), pose (i, j) = bit j % 32 of
// word j / 32, 1 = colliding; padding bits (j >= b2) are ignored.  Free poses are 4-neighbour adjacent, with the seam
// row b1-1 | row 0 when wrap bit 0 is set and column b2-1 | column 0 when wrap bit 1 is set.  Grids never connect.
// Output: labels [n_grids][b1][b2] int32, -1 for a colliding pose, else the smallest grid-local row-major index
// i * b2 + j of its component.
//
// Lock-free union-find whose parents live in `labels` itself (no scratch memory, no host synchronisation), block-based
// as in Playne & Hawick (TPDS 2018) and Allegretti, Bolelli & Grana (TPDS 2020).  Three kernels:
//   k_ccl_local    -- a block labels one TH x TC tile in shared memory: each horizontal run of free poses is linked
//                     to its first pose by bit arithmetic on the words, vertical neighbours are unioned with shared
//                     atomicMin, and every free pose's root is written back as a grid-local index.  Inside a tile,
//                     local row-major order is the grid's row-major order, so the tile's minimum is a grid minimum.
//   k_ccl_border   -- unions across the tile borders and the requested seams, in global memory.
//   k_ccl_compress -- every free pose's label becomes its root; roots (label == own index) are counted per grid.
//
// Why the final root is the component's minimum: every parent is <= its node.  It holds initially (a run start is
// left of its run, a tile root is its tile's minimum), and a union only ever writes atomicMin(&parent[hi], lo) with
// lo < hi.  Following parents therefore never increases the index, so a root is <= every node of its tree.  A union
// whose atomicMin lands on a node that another union has just linked elsewhere retries with that node's new parent
// (Playne & Hawick's union), so when every union has returned, each component is one tree, and its root is its
// minimum: the label does not depend on scheduling.
#include <climits>

#include "ag_rollout.cuh"

using namespace agd;

namespace {

constexpr int TW = 4;              // words per tile row
constexpr int TC = 32 * TW;        // tile columns
constexpr int TH = 32;             // tile rows
constexpr int TP = TH * TC;        // poses per tile (16 per thread)
constexpr int CHUNK = 16 * AG_BLOCK;   // border pairs or poses per block iteration of the other two kernels
constexpr int64_t MAX_BLOCKS = 1 << 20;

struct CclDev {
    const uint32_t *bits;                      // [n_grids][b1][W]
    int32_t *labels;                           // [n_grids][b1][b2]
    unsigned long long *n_components;          // [n_grids] or nullptr (zeroed before the launch)
    int64_t n_grids, poses;                    // poses per grid: b1 * b2 (< 2^31)
    int32_t b1, b2, W;
    int32_t tiles_r, tiles_c;                  // tiles per grid along joint_1 and joint_2
    int32_t nh, nv;                            // row borders (incl. the joint_1 seam), column borders (incl. joint_2's)
    int64_t border_items;                      // nh * b2 + nv * b1 pairs per grid
};

// Parents are read with volatile loads: another block may lower them at any time, and a cached or hoisted value
// would let find() spin on, or return, a stale root.
__device__ __forceinline__ int32_t find_root(const volatile int32_t *L, int32_t x) {
    int32_t p = L[x];
    while (p != x) {
        x = p;
        p = L[x];
    }
    return x;
}

// link the trees of a and b, the larger root under the smaller; on a lost race (the larger root was linked elsewhere
// between find and atomicMin) continue from its new parent
__device__ __forceinline__ void unite(int32_t *L, int32_t a, int32_t b) {
    for (;;) {
        a = find_root(L, a);
        b = find_root(L, b);
        if (a == b) return;
        if (a > b) { const int32_t t = a; a = b; b = t; }
        const int32_t old = atomicMin(L + b, a);
        if (old == b) return;
        b = old;
    }
}

__device__ __forceinline__ bool is_free(const CclDev &D, int64_t row_base, int32_t i, int32_t j) {
    const int64_t o = (row_base + i) * D.W + (j >> 5);
    AG_CHECK_INDEX(o, D.n_grids * D.b1 * D.W);
    return !((D.bits[o] >> (j & 31)) & 1u);
}

// one tile per block iteration; tiles are numbered grid by grid
__global__ void __launch_bounds__(AG_BLOCK, 8) k_ccl_local(const __grid_constant__ CclDev D) {
    __shared__ uint32_t s_free[TH * TW];       // 1 = free; padding and poses outside the grid read as colliding
    __shared__ int32_t s_lab[TP];              // tile-local parents, -1 colliding
    const int64_t tiles = (int64_t)D.tiles_r * D.tiles_c;
    for (int64_t T = blockIdx.x; T < D.n_grids * tiles; T += gridDim.x) {
        const int64_t g = T / tiles;
        const int t = (int)(T % tiles);
        const int i0 = (t / D.tiles_c) * TH, j0 = (t % D.tiles_c) * TC;
        for (int k = threadIdx.x; k < TH * TW; k += blockDim.x) {
            const int r = k / TW, w = (j0 >> 5) + k % TW;
            uint32_t f = 0u;
            if (i0 + r < D.b1 && w < D.W) {
                const int64_t o = (g * D.b1 + i0 + r) * D.W + w;
                AG_CHECK_INDEX(o, D.n_grids * D.b1 * D.W);
                f = ~D.bits[o];
                const int valid = D.b2 - (w << 5);
                if (valid < 32) f &= (1u << valid) - 1u;
            }
            s_free[k] = f;
        }
        __syncthreads();
        // each free pose points at the first pose of its run: the highest colliding bit left of it, + 1
        for (int p = threadIdx.x; p < TP; p += blockDim.x) {
            const int r = p / TC, c = p % TC, w = c >> 5, b = c & 31;
            const uint32_t *row = s_free + r * TW;
            int32_t lab = -1;
            if ((row[w] >> b) & 1u) {
                const uint32_t blocked = ~row[w] & ((1u << b) - 1u);
                int start = w << 5;
                if (blocked) {
                    start += 32 - __clz(blocked);
                } else {
                    for (int v = w - 1; v >= 0; --v) {
                        const uint32_t bv = ~row[v];
                        start = v << 5;
                        if (bv) { start += 32 - __clz(bv); break; }
                    }
                }
                lab = r * TC + start;
            }
            s_lab[p] = lab;
        }
        __syncthreads();
        // vertical unions; where the pair to the left is free too, both runs are already joined through it
        for (int p = threadIdx.x + TC; p < TP; p += blockDim.x) {
            const int r = p / TC, c = p % TC, w = c >> 5, b = c & 31;
            const uint32_t both = s_free[r * TW + w] & s_free[(r - 1) * TW + w];
            if ((both >> b) & 1u) {
                const bool left = b ? ((both >> (b - 1)) & 1u)
                                    : (w > 0 && ((s_free[r * TW + w - 1] & s_free[(r - 1) * TW + w - 1]) >> 31));
                if (!left) unite(s_lab, p, p - TC);
            }
        }
        __syncthreads();
        // roots back to global memory, as grid-local indices
        const int64_t base = g * D.poses;
        for (int p = threadIdx.x; p < TP; p += blockDim.x) {
            const int i = i0 + p / TC, j = j0 + p % TC;
            if (i < D.b1 && j < D.b2) {
                int32_t out = -1;
                const int32_t lab = s_lab[p];
                if (lab >= 0) {
                    const int32_t root = find_root(s_lab, lab);
                    out = (i0 + root / TC) * D.b2 + j0 + root % TC;
                }
                const int64_t o = base + (int64_t)i * D.b2 + j;
                AG_CHECK_INDEX(o, D.n_grids * D.poses);
                D.labels[o] = out;
            }
        }
        __syncthreads();                       // s_free / s_lab are rewritten by the next tile
    }
}

// Border pair k of a grid: k < nh * b2 is column j of row border k / b2 (rows (k/b2 + 1) * TH - 1 and + TH, or the
// joint_1 seam b1-1 | 0); the rest are row i of column border (k - nh * b2) / b1 (likewise).  A pair whose
// neighbours one step back along the border are both free is skipped when the two steps from them lie inside tiles:
// the local pass joined those, and the pair one step back is joined here (or skipped by the same rule).
__global__ void __launch_bounds__(AG_BLOCK) k_ccl_border(const __grid_constant__ CclDev D) {
    const int64_t chunks = (D.border_items + CHUNK - 1) / CHUNK;
    for (int64_t C = blockIdx.x; C < D.n_grids * chunks; C += gridDim.x) {
        const int64_t g = C / chunks, rb0 = g * D.b1;
        int32_t *L = D.labels + g * D.poses;
        const int64_t k1 = min(D.border_items, (C % chunks + 1) * CHUNK);
        for (int64_t k = (C % chunks) * CHUNK + threadIdx.x; k < k1; k += blockDim.x) {
            int32_t ia, ja, ib, jb;
            bool inner;
            if (k < (int64_t)D.nh * D.b2) {
                const int32_t h = (int32_t)(k / D.b2);
                ja = jb = (int32_t)(k % D.b2);
                ia = h < D.tiles_r - 1 ? (h + 1) * TH - 1 : D.b1 - 1;
                ib = h < D.tiles_r - 1 ? (h + 1) * TH : 0;
                inner = ja % TC != 0 && is_free(D, rb0, ia, ja - 1) && is_free(D, rb0, ib, ja - 1);
            } else {
                const int64_t kv = k - (int64_t)D.nh * D.b2;
                const int32_t v = (int32_t)(kv / D.b1);
                ia = ib = (int32_t)(kv % D.b1);
                ja = v < D.tiles_c - 1 ? (v + 1) * TC - 1 : D.b2 - 1;
                jb = v < D.tiles_c - 1 ? (v + 1) * TC : 0;
                inner = ia % TH != 0 && is_free(D, rb0, ia - 1, ja) && is_free(D, rb0, ia - 1, jb);
            }
            if (!inner && is_free(D, rb0, ia, ja) && is_free(D, rb0, ib, jb)) {
                AG_CHECK_INDEX(ia * D.b2 + ja, D.poses);
                AG_CHECK_INDEX(ib * D.b2 + jb, D.poses);
                unite(L, ia * D.b2 + ja, ib * D.b2 + jb);
            }
        }
    }
}

__global__ void __launch_bounds__(AG_BLOCK, 8) k_ccl_compress(const __grid_constant__ CclDev D) {
    __shared__ unsigned int s_roots;
    const int64_t chunks = (D.poses + CHUNK - 1) / CHUNK;
    if (threadIdx.x == 0) s_roots = 0u;
    __syncthreads();
    for (int64_t C = blockIdx.x; C < D.n_grids * chunks; C += gridDim.x) {
        const int64_t g = C / chunks;
        int32_t *L = D.labels + g * D.poses;
        const int64_t p1 = min(D.poses, (C % chunks + 1) * CHUNK);
        unsigned int roots = 0u;
        for (int64_t p = (C % chunks) * CHUNK + threadIdx.x; p < p1; p += blockDim.x) {
            const int32_t lab = L[p];
            if (lab >= 0) {
                AG_CHECK_INDEX(lab, D.poses);
                const int32_t root = find_root(L, lab);
                if (root != lab) L[p] = root;
                roots += root == p;
            }
        }
        if (D.n_components != nullptr) {                               // block-uniform
            roots = __reduce_add_sync(0xFFFFFFFFu, roots);
            if ((threadIdx.x & 31) == 0 && roots) atomicAdd(&s_roots, roots);
            __syncthreads();
            if (threadIdx.x == 0 && s_roots) {
                AG_CHECK_INDEX(g, D.n_grids);
                atomicAdd(D.n_components + g, (unsigned long long)s_roots);
                s_roots = 0u;
            }
            __syncthreads();
        }
    }
}

template <typename Kernel>
ag_status launch(Kernel k, int64_t work, const CclDev &D, cudaStream_t s) {
    k<<<(unsigned)(work < MAX_BLOCKS ? work : MAX_BLOCKS), AG_BLOCK, 0, s>>>(D);
    return launched();
}

}  // namespace

extern "C" ag_status ag_cspace_components(const uint32_t *bits, int64_t n_grids, int32_t b1, int32_t b2, int32_t wrap,
                                          int32_t *labels, int64_t *n_components, void *stream) {
    if (n_grids < 0 || b1 < 1 || b2 < 1) return AG_ERR_SHAPE;
    const int64_t poses = (int64_t)b1 * b2;
    if (poses > INT32_MAX || (n_grids > 0 && poses > INT64_MAX / n_grids)) return AG_ERR_SHAPE;   // grid-local int32 labels
    if (wrap & ~3) return AG_ERR_MODE;
    if (n_grids == 0) return AG_OK;
    if (!bits || !labels) return AG_ERR_NULL;
    if (((uintptr_t)bits % 4) || ((uintptr_t)labels % 4) || ((uintptr_t)n_components % 8)) return AG_ERR_ALIGN;
    cudaStream_t s = (cudaStream_t)stream;
    CclDev D;
    D.bits = bits; D.labels = labels; D.n_components = reinterpret_cast<unsigned long long *>(n_components);
    D.n_grids = n_grids; D.poses = poses;
    D.b1 = b1; D.b2 = b2; D.W = (b2 + 31) / 32;
    D.tiles_r = (b1 + TH - 1) / TH; D.tiles_c = (b2 + TC - 1) / TC;
    D.nh = D.tiles_r - 1 + ((wrap & 1) && b1 > 1); D.nv = D.tiles_c - 1 + ((wrap & 2) && b2 > 1);   // a pose is never its own neighbour
    D.border_items = (int64_t)D.nh * b2 + (int64_t)D.nv * b1;
    if (n_components != nullptr) {
        const cudaError_t e = cudaMemsetAsync(n_components, 0, (size_t)n_grids * sizeof(int64_t), s);
        if (e != cudaSuccess) return (ag_status)e;
    }
    ag_status st = launch(k_ccl_local, n_grids * D.tiles_r * D.tiles_c, D, s);
    if (st == AG_OK && D.border_items > 0) st = launch(k_ccl_border, n_grids * ((D.border_items + CHUNK - 1) / CHUNK), D, s);
    if (st == AG_OK) st = launch(k_ccl_compress, n_grids * ((D.poses + CHUNK - 1) / CHUNK), D, s);
    return st;
}
