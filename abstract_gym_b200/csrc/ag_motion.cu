// ag_motion.cu -- batched joint-space motion checking: robot/two_joint_robot.py:49-62 move_to_joint_pose() with the
// collision check of scenario/scene_0.py:60-76 at every intermediate pose (ag_check_motion, DESIGN.md "Motion checking").
//
// Motion i walks pose_k = pose_{k-1} + inc (k = 1 .. steps[i], the reference's operation order, float64, never
// contracted) and stops at its first colliding pose.  One thread per motion; the lanes of a warp run their own walks
// and the warp lasts as long as its longest walk (DESIGN.md records the measured lane utilisation of that choice).
//
// Two forms of the per-pose test, with identical results:
//   map form (FAST engine, where ag_cmap.cu hands the launch a configuration-space map: scene_0-class grids) -- 2 DADD
//     for the pose and cmap_needs_check (ag_cmap.cuh), the test of k_rollout_lut's hot loop; only the poses it flags go
//     to pose_collides<FAST>.  Persistent blocks: each copies the 32 KB map once and walks many motions.
//   general form (every other grid or engine) -- pose_collides<ENGINE> at every pose: the obstacle list, the bit-grid
//     and two-level traversals of the FAST engine, EXACT, BRUTE.
// first_hit is computed once per motion, at its first colliding pose, with the EXACT (or BRUTE) arithmetic of K2.
#include <climits>

#include "ag_cmap.cuh"
#include "ag_rollout.cuh"

using namespace agd;

namespace {

struct MotionDev {
    const double *j1, *j2, *goal;   // start [m], [m]; goal [m][2]
    const int32_t *steps;           // [m]
    int32_t *first_collision;       // [m]
    int32_t *first_hit;             // [m] or nullptr
    double *last_free;              // [m][2] or nullptr
    int64_t m, env_id0;
    const uint32_t *cmap;           // map form: the map words (global memory), copied to shared memory at cmap_off
    uint32_t cmap_off;
};

// K2's first_hit at one pose (EXACT arithmetic; BRUTE for the BRUTE engine), -1 if it does not collide.  Out of line: it
// runs once per motion, and inlined next to the walk's own check it would push the walk's registers into local memory.
template <int ENGINE>
__device__ __noinline__ int first_hit_at(const ag_params &P, const GridDev &G, const BlockCtx &B, const FastConst &C, double q1,
                                         double q2) {
    int fh = INT_MAX, axis = 0;
    return pose_collides<ENGINE, true>(P, G, B, C, q1, q2, fh, axis) ? fh : -1;
}

// MAP: the map form (ENGINE == FAST, staged obstacle-list grid).  Every thread walks motions i, i + stride, ...; the
// general form is launched with one motion per thread, so a thread's grid is the one block_prologue staged or chose.
template <int ENGINE, bool MAP>
__global__ void __launch_bounds__(AG_BLOCK, 1) k_check_motion(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G,
                                                           const __grid_constant__ FastConst C, const __grid_constant__ MotionDev M) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    const BlockCtx B = block_prologue<ENGINE>(G, M.env_id0, M.m, smem, &s_fl);
    uint32_t cmap_a = 0u;
    if constexpr (MAP) {                                                         // the map: global -> shared, once per block
        cmap_to_shared(smem + M.cmap_off, M.cmap, blockDim.x);
        __syncthreads();
        cmap_a = smem_u32(smem + M.cmap_off);
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M.m; i += (int64_t)gridDim.x * blockDim.x) {
        AG_CHECK_INDEX(i, M.m);
        double q1 = M.j1[i], q2 = M.j2[i];
        const double2 goal = reinterpret_cast<const double2 *>(M.goal)[i];
        const int n = M.steps[i];
        int fc = -2;                                                             // steps < 1: nothing checked
        double inc1 = 0.0, inc2 = 0.0;
        if (n >= 1) {
            const double alpha = __ddiv_rn(1.0, (double)n);                      // two_joint_robot.py:57
            inc1 = __dmul_rn(alpha, __dsub_rn(goal.x, q1));
            inc2 = __dmul_rn(alpha, __dsub_rn(goal.y, q2));
            fc = -1;
#pragma unroll 1
            for (int k = 1; k <= n; ++k) {
                const double p1 = __dadd_rn(q1, inc1), p2 = __dadd_rn(q2, inc2);   // :61-62
                const bool slow = !MAP || cmap_needs_check(cmap_a, p1, p2);
                if (slow && pose_hit<ENGINE, MAP ? BP_LIST : BP_ANY>(P, G, B, C, p1, p2)) { fc = k; break; }
                q1 = p1; q2 = p2;
            }
        }
        M.first_collision[i] = fc;
        if (M.first_hit != nullptr)
            M.first_hit[i] = fc > 0 ? first_hit_at<ENGINE>(P, G, B, C, __dadd_rn(q1, inc1), __dadd_rn(q2, inc2)) : -1;
        if (M.last_free != nullptr) reinterpret_cast<double2 *>(M.last_free)[i] = make_double2(q1, q2);
    }
}

template <int ENGINE, bool MAP>
ag_status launch(const ag_params &P, const GridDev &G, const MotionDev &M, size_t smem, cudaStream_t s) {
    auto k = k_check_motion<ENGINE, MAP>;
    ag_status st = set_smem(k, smem);
    if (st != AG_OK) return st;
    unsigned blocks = blocks_for(M.m);
    if (MAP) {                                                                   // persistent: as many blocks as fit at once
        int slots = 0;
        st = resident_blocks(k, AG_BLOCK, smem, &slots);
        if (st != AG_OK) return st;
        blocks = blocks < (unsigned)slots ? blocks : (unsigned)slots;
    }
    k<<<blocks, AG_BLOCK, smem, s>>>(P, G, make_fast_const(P, G), M);
    return launched();
}

}  // namespace

extern "C" ag_status ag_check_motion(const ag_params *p, const ag_grid *g, const double *j1, const double *j2,
                                     const double *goal, const int32_t *steps, int32_t *first_collision, int32_t *first_hit,
                                     double *last_free, int64_t m, int64_t env_id0, int32_t engine, void *stream) {
    if (m < 0) return AG_ERR_SHAPE;
    if (!p || !g) return AG_ERR_NULL;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, env_id0, engine, &G, &smem);
    if (st) return st;
    if (m == 0) return AG_OK;
    if (!j1 || !j2 || !goal || !steps || !first_collision) return AG_ERR_NULL;
    if (((uintptr_t)goal % 16) || ((uintptr_t)last_free % 16)) return AG_ERR_ALIGN;
    cudaStream_t s = (cudaStream_t)stream;
    MotionDev M;
    M.j1 = j1; M.j2 = j2; M.goal = goal; M.steps = steps;
    M.first_collision = first_collision; M.first_hit = first_hit; M.last_free = last_free;
    M.m = m; M.env_id0 = env_id0; M.cmap = nullptr; M.cmap_off = 0;
    switch (engine) {
        case AG_ENGINE_FAST: {
            CmapLaunch cm;
            st = cspace_map_for_launch(*p, G, g->max_occupied, smem, s, &cm);
            if (st != AG_OK) return st;
            M.cmap = cm.map; M.cmap_off = cm.off;
            return cm.map ? launch<AG_ENGINE_FAST, true>(*p, G, M, cm.smem, s) : launch<AG_ENGINE_FAST, false>(*p, G, M, smem, s);
        }
        case AG_ENGINE_EXACT: return launch<AG_ENGINE_EXACT, false>(*p, G, M, smem, s);
        case AG_ENGINE_BRUTE: return launch<AG_ENGINE_BRUTE, false>(*p, G, M, smem, s);
        default: return AG_ERR_MODE;
    }
}
