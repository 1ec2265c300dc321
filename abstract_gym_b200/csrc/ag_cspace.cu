// ag_cspace.cu -- batched configuration-space occupancy: scenario/scene_0.py:60-76 collision_check() at every pose of a
// joint-angle lattice, one bit per pose, per grid (ag_cspace_occupancy, DESIGN.md "Configuration-space occupancy").
//
// Pose (i, j) = (lo1 + i * step1, lo2 + j * step2), float64, one rounding per operation.  Its bit is K2's flag with the
// same engine.  A warp owns a unit of up to UNIT_WORDS consecutive 32-pose words of one lattice row: each lane tests one
// pose, __ballot_sync builds the word, lane 0 stores it.  Lanes past the row's end test a pose too (so the warp stays
// converged at the ballot and in the reconvergence points of the checks) and their bits are masked off.  A block works
// on one grid, which it stages once; free counts are a popcount per word, a block sum and one atomic per block.
//
// Three forms, with K2's results:
//   map form (FAST engine, where ag_cmap.cu hands the launch a configuration-space map: scene_0-class grids) -- the
//     test of cmap_needs_check (ag_cmap.cuh) with joint_1's phase hoisted out of the row; only the poses it flags go to
//     pose_collides<FAST>.
//   row form (EXACT, BRUTE) -- link 1 depends on joint_1 only, so it is tested once per unit; a unit whose link 1 hits
//     is all ones, every other pose tests link 2 only.  Both engines' flag is exactly link 1 || link 2 (arm_collides,
//     arm_brute), with the elbow of forward_kinematics, so the bits are K2's.
//   general form (FAST on every other grid) -- pose_collides<FAST> per pose.  FAST's decision is not a per-link OR
//     (the float32 filter and the float64 re-evaluation look at the arm as a whole), so it is not factored.
#include <climits>

#include "ag_cmap.cuh"
#include "ag_rollout.cuh"

using namespace agd;

namespace {

// words (of 32 poses) per unit: the row form tests link 1 once per 128 poses.  FAST shares nothing along a row, but
// single-word units made every FAST workload of tools/cspace_bench.py slower (1.4-1.7x), so it takes the same 4.
constexpr int UNIT_WORDS = 4;
constexpr int WARPS = AG_BLOCK / 32;

struct CspaceDev {
    double lo1, step1, lo2, step2;
    int32_t b1, b2, W, spans;                  // spans: units per lattice row
    int64_t units;                             // units per grid (b1 * spans)
    int64_t blocks_per_grid;
    uint32_t *bits;                            // [n_grids][b1][W]
    unsigned long long *free_count;            // [n_grids] or nullptr (zeroed before the launch)
    const uint32_t *cmap;                      // map form: the map words (global memory), copied to shared memory at cmap_off
    uint32_t cmap_off;
};

// one link of the row form: the flag of link_exact (EXACT) or of the reference's loop over every cell (BRUTE)
template <int ENGINE>
__device__ __forceinline__ bool link_hits(const GridDev &G, const GridView &V, double p0x, double p0y, double p1x, double p1y,
                                          double eps) {
    int fh = 0, axis = 0;
    if constexpr (ENGINE == AG_ENGINE_BRUTE) return link_brute<false>(G, V, p0x, p0y, p1x, p1y, eps, fh, axis);
    else return link_exact<false>(G, V, p0x, p0y, p1x, p1y, eps, fh, axis);
}

// G.envs_per_grid == 1 (set by the launcher): env id g selects grid g, and no grid index overflows an env id.
// Two blocks per SM fit the row form without spills; the FAST forms need more than 128 registers (see DESIGN.md).
template <int ENGINE, bool MAP>
__global__ void __launch_bounds__(AG_BLOCK, ENGINE == AG_ENGINE_FAST ? 1 : 2)
k_cspace(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G,
         const __grid_constant__ FastConst C, const __grid_constant__ CspaceDev D) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    __shared__ unsigned long long s_free;
    const int64_t g = (int64_t)blockIdx.x / D.blocks_per_grid, part = (int64_t)blockIdx.x % D.blocks_per_grid;
    BlockCtx B;
    B.V = stage_grid(G, g, smem);
    B.fl = nullptr;
    if (ENGINE == AG_ENGINE_FAST && G.stage) {
        build_fast_list(G, B.V, &s_fl);
        B.fl = &s_fl;
    }
    if constexpr (MAP) cmap_to_shared(smem + D.cmap_off, D.cmap, blockDim.x);   // the map: global -> shared, once per block
    if (threadIdx.x == 0) s_free = 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t cmap_a = MAP ? smem_u32(smem + D.cmap_off) : 0u;
    unsigned long long free = 0;
    for (int64_t u = part * WARPS + (threadIdx.x >> 5); u < D.units; u += D.blocks_per_grid * WARPS) {
        const int64_t i = u / D.spans;
        const int w0 = (int)(u % D.spans) * UNIT_WORDS, w1 = min(w0 + UNIT_WORDS, D.W);
        const double q1 = __dadd_rn(D.lo1, __dmul_rn((double)i, D.step1));
        // row form: link 1, once per unit (every lane has the same joint_1, so this is warp-uniform work)
        bool row_hit = false;
        if constexpr (ENGINE != AG_ENGINE_FAST) {
            const Arm A = forward_kinematics(q1, 0.0, P.link_1, P.link_2);
            row_hit = link_hits<ENGINE>(G, B.V, 0.0, 0.0, A.ex, A.ey, P.section_eps);
        }
        const uint32_t x1 = MAP ? cmap_phase(q1) : 0u;
        const bool in1 = cmap_in_range(q1);
        for (int w = w0; w < w1; ++w) {
            const int j = (w << 5) + lane;
            const double q2 = __dadd_rn(D.lo2, __dmul_rn((double)j, D.step2));
            bool hit;
            if constexpr (MAP) {
                const bool slow = cmap_bit(cmap_a, x1, cmap_phase(q2)) || !in1 || !cmap_in_range(q2);
                hit = slow && pose_hit<ENGINE>(P, G, B, C, q1, q2);
            } else if constexpr (ENGINE == AG_ENGINE_FAST) {
                hit = pose_hit<ENGINE>(P, G, B, C, q1, q2);
            } else {
                hit = row_hit;
                if (!row_hit) {                                                  // warp-uniform branch
                    const Arm A = forward_kinematics(q1, q2, P.link_1, P.link_2);
                    hit = link_hits<ENGINE>(G, B.V, A.ex, A.ey, A.gx, A.gy, P.section_eps);
                }
            }
            const uint32_t valid = __ballot_sync(0xFFFFFFFFu, j < D.b2);
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, hit) & valid;
            if (lane == 0) {
                const int64_t o = (g * D.b1 + i) * D.W + w;
                AG_CHECK_INDEX(o, (int64_t)G.n_grids * D.b1 * D.W);
                D.bits[o] = word;
                free += (unsigned)__popc(valid & ~word);
            }
        }
    }
    if (D.free_count != nullptr) {
        if (lane == 0 && free != 0) atomicAdd(&s_free, free);
        __syncthreads();
        if (threadIdx.x == 0 && s_free != 0) {
            AG_CHECK_INDEX(g, G.n_grids);
            atomicAdd(&D.free_count[g], s_free);
        }
    }
}

template <int ENGINE, bool MAP>
ag_status launch(const ag_params &P, const GridDev &G, const CspaceDev &D0, size_t smem, cudaStream_t s) {
    auto k = k_cspace<ENGINE, MAP>;
    ag_status st = set_smem(k, smem);
    if (st != AG_OK) return st;
    int slots = 0;
    st = resident_blocks(k, AG_BLOCK, smem, &slots);
    if (st != AG_OK) return st;
    // Blocks per grid: one unit per warp at most; otherwise about one wave of blocks in all (map form: every block
    // copies the 32 KB map once) or four (the other forms: grids differ in cost, so finer blocks balance better).
    // The total stays below 2^31: it is at most max(n_grids, 4 * slots + n_grids).
    const int64_t waves = MAP ? 1 : 4, want = waves * (slots > 0 ? slots : 1);
    CspaceDev D = D0;
    const int64_t per_grid = (want + G.n_grids - 1) / G.n_grids, most = (D.units + WARPS - 1) / WARPS;
    D.blocks_per_grid = per_grid < most ? per_grid : most;
    k<<<(unsigned)(D.blocks_per_grid * G.n_grids), AG_BLOCK, smem, s>>>(P, G, make_fast_const(P, G), D);
    return launched();
}

}  // namespace

// ag_cspace_occupancy after argument validation (ag_kernels.cu): smem = the staged grid's bytes (make_grid_dev, env_id0 0)
ag_status launch_cspace_occupancy(const ag_params &P, const GridDev &G0, int32_t max_occupied, double lo1, double step1,
                                  int32_t b1, double lo2, double step2, int32_t b2, uint32_t *bits, int64_t *free_count,
                                  int32_t engine, size_t smem, cudaStream_t s) {
    CspaceDev D;
    D.lo1 = lo1; D.step1 = step1; D.lo2 = lo2; D.step2 = step2;
    D.b1 = b1; D.b2 = b2; D.W = (b2 + 31) / 32; D.spans = (D.W + UNIT_WORDS - 1) / UNIT_WORDS;
    D.units = (int64_t)b1 * D.spans; D.blocks_per_grid = 1;
    D.bits = bits; D.free_count = reinterpret_cast<unsigned long long *>(free_count);
    D.cmap = nullptr; D.cmap_off = 0;
    GridDev G = G0;
    G.envs_per_grid = 1;                                                         // blocks address grids by index
    if (free_count != nullptr) {
        const cudaError_t e = cudaMemsetAsync(free_count, 0, (size_t)G.n_grids * sizeof(int64_t), s);
        if (e != cudaSuccess) return (ag_status)e;
    }
    switch (engine) {
        case AG_ENGINE_FAST: {
            CmapLaunch cm;
            const ag_status st = cspace_map_for_launch(P, G0, max_occupied, smem, s, &cm);
            if (st != AG_OK) return st;
            D.cmap = cm.map; D.cmap_off = cm.off;
            return cm.map ? launch<AG_ENGINE_FAST, true>(P, G, D, cm.smem, s) : launch<AG_ENGINE_FAST, false>(P, G, D, smem, s);
        }
        case AG_ENGINE_EXACT: return launch<AG_ENGINE_EXACT, false>(P, G, D, smem, s);
        case AG_ENGINE_BRUTE: return launch<AG_ENGINE_BRUTE, false>(P, G, D, smem, s);
        default: return AG_ERR_MODE;
    }
}
