// ag_kernels.cu -- kernels K1..K5 of the scene_0 hot path and their extern "C" launchers.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 (abstract_gym_b200/build.py).
#include <atomic>
#include <climits>
#include <cstring>

#include "ag_rollout.cuh"

using namespace agd;

namespace {

#ifndef AG_FAST_BLOCKS_PER_SM
#define AG_FAST_BLOCKS_PER_SM 4
#endif
std::atomic<long long> g_launches{0};

// ------------------------------------------------------------------------------------------- K5
// environment/occupancy_grid.py:35-37,85-90: matrix -> set of occupied cells, here one bit per cell.
__global__ void k_grid_pack(const uint8_t *__restrict__ occ, int S, int wpr, int n_grids, uint32_t *__restrict__ bits,
                            int64_t stride_words) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t per_grid = (int64_t)S * wpr;
    if (i >= per_grid * n_grids) return;
    const int64_t g = i / per_grid;
    const int r = (int)((i % per_grid) / wpr), w = (int)(i % wpr);
    const uint8_t *row = occ + (g * S + r) * (int64_t)S;
    uint32_t word = 0;
    const int c_end = min(S, (w + 1) * 32);
    for (int c = w * 32; c < c_end; ++c) word |= (row[c] != 0 ? 1u : 0u) << (c & 31);
    bits[g * stride_words + (int64_t)r * wpr + w] = word;
}

// bits -> the two-level form (ag_grid.hier): one thread per 8x8 tile; the summary bitmap is zeroed by the launcher
__global__ void k_grid_pack_hier(const uint32_t *__restrict__ bits, int S, int wpr, int n_grids, int64_t stride_words,
                                 unsigned char *__restrict__ hier, int T, int cwpr, int64_t tiles_bytes, int64_t coarse_words,
                                 int64_t hier_bytes) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * T * n_grids) return;
    const int64_t g = i / ((int64_t)T * T);
    const int R = (int)((i % ((int64_t)T * T)) / T), Cc = (int)(i % T);
    const uint32_t *gb = bits + g * stride_words;
    unsigned long long tile = 0;
    for (int dr = 0; dr < 8; ++dr) {
        const int r = R * 8 + dr;
        if (r >= S) break;
        const uint32_t byte = (gb[(int64_t)r * wpr + (Cc >> 2)] >> ((Cc & 3) * 8)) & 0xFFu;   // columns 8Cc .. 8Cc+7 of row r
        tile |= (unsigned long long)byte << (dr * 8);
    }
    unsigned char *gh = hier + g * hier_bytes;
    reinterpret_cast<unsigned long long *>(gh)[(int64_t)R * T + Cc] = tile;
    if (tile) {
        uint32_t *coarse = reinterpret_cast<uint32_t *>(gh + tiles_bytes);
        atomicOr(coarse + R * cwpr + (Cc >> 5), 1u << (Cc & 31));
        atomicOr(coarse + coarse_words + Cc * cwpr + (R >> 5), 1u << (R & 31));
    }
}

// ------------------------------------------------------------------------- predicate / FK arrays
__global__ void k_segment_square(const double *__restrict__ seg, const double *__restrict__ sq, double eps,
                                 uint8_t *__restrict__ hit, double *__restrict__ abc, double *__restrict__ corner_values,
                                 unsigned long long *axis_aligned, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double4 s = reinterpret_cast<const double4 *>(seg)[i];
    const double4 q = reinterpret_cast<const double4 *>(sq)[i];
    int axis = 0;
    const LineD L = make_line(s.x, s.y, s.z, s.w);       // utils/collision_checker.py:21
    hit[i] = segment_square_exact(L, q.x, q.y, q.z, q.w, eps, axis) ? 1 : 0;
    if (abc) { abc[3 * i] = L.a; abc[3 * i + 1] = L.b; abc[3 * i + 2] = L.c; }
    if (corner_values) {                                 // utils/collision_checker.py:27-30
        const double ax0 = __dmul_rn(L.a, q.x), ax1 = __dmul_rn(L.a, q.z);
        const double by0 = __dmul_rn(L.b, q.y), by1 = __dmul_rn(L.b, q.w);
        corner_values[4 * i] = __dadd_rn(__dadd_rn(ax0, by0), L.c);
        corner_values[4 * i + 1] = __dadd_rn(__dadd_rn(ax0, by1), L.c);
        corner_values[4 * i + 2] = __dadd_rn(__dadd_rn(ax1, by0), L.c);
        corner_values[4 * i + 3] = __dadd_rn(__dadd_rn(ax1, by1), L.c);
    }
    if (axis && axis_aligned) atomicAdd(axis_aligned, (unsigned long long)axis);
}

__global__ void k_forward_kinematics(ag_params P, const double *__restrict__ j1, const double *__restrict__ j2,
                                     double *__restrict__ out, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Arm A = forward_kinematics(j1[i], j2[i], P.link_1, P.link_2);
    reinterpret_cast<double4 *>(out)[i] = make_double4(A.ex, A.ey, A.gx, A.gy);
}

// robot/two_joint_robot.py:74-113 inverse_kinematic() over arrays (not on the step/reset path; SURVEY 8f.3).
// sol: [n][4] = (j1_1, j2_1, j1_2, j2_2); valid: [n].  corrected: alpha = atan2(y, x) instead of arccos(x/r).
__global__ void k_inverse_kinematics(ag_params P, const double *__restrict__ target, double *__restrict__ sol,
                                     uint8_t *__restrict__ valid, int corrected, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2 t = reinterpret_cast<const double2 *>(target)[i];
    const double l1 = P.link_1, l2 = P.link_2;
    const double radius = sqrt(__dadd_rn(__dmul_rn(t.x, t.x), __dmul_rn(t.y, t.y)));                   // :82
    const bool ok = (fabs(__dsub_rn(l1, l2)) < radius) && (radius <= __dadd_rn(l1, l2)) && radius != 0.0;   // :80-86,:96
    valid[i] = ok ? 1 : 0;
    double4 out = make_double4(0.0, 0.0, 0.0, 0.0);
    if (ok) {
        const double r2 = __dmul_rn(radius, radius), a2 = __dmul_rn(l1, l1), b2 = __dmul_rn(l2, l2);
        const double cos_theta = __ddiv_rn(__dsub_rn(__dadd_rn(r2, a2), b2), __dmul_rn(__dmul_rn(2.0, l1), radius));   // :99
        const double theta = acos(cos_theta);                                                                        // :100
        const double alpha = corrected ? atan2(t.y, t.x) : acos(__ddiv_rn(t.x, radius));                             // :101-102
        const double cos_beta = __ddiv_rn(__dsub_rn(__dadd_rn(a2, b2), r2), __dmul_rn(__dmul_rn(2.0, l1), l2));      // :105
        const double inner = __dsub_rn(3.141592653589793, acos(cos_beta));
        out.x = __dsub_rn(alpha, theta);                                   // :103
        out.z = __dadd_rn(alpha, theta);                                   // :104
        out.y = __dadd_rn(inner, out.x);                                   // :106
        out.w = __dsub_rn(out.z, inner);                                   // :107
    }
    reinterpret_cast<double4 *>(sol)[i] = out;
}

// robot/two_joint_robot.py:49-62 move_to_joint_pose(): `steps` increments alpha*(target - init) added one by one
// (no intermediate collision checks, like the reference)
__global__ void k_move_to_joint_pose(double *__restrict__ j1, double *__restrict__ j2, const double *__restrict__ target,
                                     int steps, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2 t = reinterpret_cast<const double2 *>(target)[i];
    double a = j1[i], b = j2[i];
    const double alpha = __ddiv_rn(1.0, (double)steps);                    // :57
    const double inc1 = __dmul_rn(alpha, __dsub_rn(t.x, a)), inc2 = __dmul_rn(alpha, __dsub_rn(t.y, b));
    for (int k = 0; k < steps; ++k) { a = __dadd_rn(a, inc1); b = __dadd_rn(b, inc2); }                 // :61-62
    j1[i] = a; j2[i] = b;
}

// ------------------------------------------------------------------------------------------- K2
template <int ENGINE, bool WANT_FIRST>
__global__ void __launch_bounds__(AG_BLOCK) k_collision(const ag_params P, const GridDev G,
                                                        const double *__restrict__ j1, const double *__restrict__ j2,
                                                        uint8_t *__restrict__ hit, int32_t *__restrict__ first_hit,
                                                        int64_t n, int64_t env_id0) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    const BlockCtx B = block_prologue<ENGINE>(G, env_id0, n, smem, &s_fl);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const FastConst C = make_fast_const(P, G);
    int fh = INT_MAX, axis = 0;
    const bool h = pose_collides<ENGINE, WANT_FIRST>(P, G, B, C, j1[e], j2[e], fh, axis);
    hit[e] = h ? 1 : 0;
    if (WANT_FIRST) first_hit[e] = h ? fh : -1;
}

// ------------------------------------------------------------------------------------------- K3
// scenario/scene_0.py:105-113 (clear_flags) / :174-181
template <int ENGINE, bool HAS_RESET_U>
__global__ void __launch_bounds__(AG_BLOCK) k_reset(const ag_params P, const GridDev G, double *__restrict__ j1,
                                                    double *__restrict__ j2, float *__restrict__ reward,
                                                    uint8_t *__restrict__ flags, uint32_t *__restrict__ reset_ctr,
                                                    const uint8_t *__restrict__ mask, const double *__restrict__ reset_u,
                                                    int32_t R, uint64_t seed, int clear_flags, unsigned long long *stats,
                                                    int64_t n, int64_t env_id0) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    __shared__ unsigned long long s_acc[AG_ST_COUNT];
    if (threadIdx.x < AG_ST_COUNT) s_acc[threadIdx.x] = 0;
    const BlockCtx B = block_prologue<ENGINE>(G, env_id0, n, smem, &s_fl);
    __syncthreads();
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n && (mask == nullptr || mask[e] != 0)) {
        const FastConst C = make_fast_const(P, G);
        double q1 = j1[e], q2 = j2[e];
        uint32_t rc = reset_ctr[e];
        int fh = 0, axis = 0;
        const bool h = pose_collides<ENGINE, false>(P, G, B, C, q1, q2, fh, axis);
        if (axis) acc32(s_acc, AG_ST_AXIS_ALIGNED, axis);
        resample_pose<ENGINE, HAS_RESET_U>(P, G, B, C, h, q1, q2, rc, HAS_RESET_U ? reset_u + (int64_t)e * R * 2 : nullptr,
                                           R, seed, (uint64_t)(env_id0 + e), s_acc);
        j1[e] = q1; j2[e] = q2; reset_ctr[e] = rc;
        if (clear_flags) { reward[e] = 0.0f; flags[e] = 0; }       // scene_0.py:111-113
    }
    stats_flush(s_acc, stats);
}

// -------------------------------------------------------------------------------------- K1 / K6
// One env step per thread: Scene.step (scene_0.py:88-103) behind ag_step, and the gym-style step of
// scenario/vector_env.py behind ag_step_obs, which adds the terminal observation, the episode statistics and
// Scene.reset() of experiment_0.py:30-34 (same-step auto-reset), and the observation of the pose the env continues from.
// obs / final_obs: [n][AG_OBS_DIM] float64 = (joint_1, joint_2, EE_x, EE_y, |target_x - EE_x|, |target_y - EE_y|); crop:
// [n][c][c] uint8 occupancy of the c x c cells centred on the end effector's cell (1 = occupied, 2 = outside the grid),
// row 0 = top.
struct StepDev {
    double *j1, *j2;                       // in/out
    const void *actions;                   // [n][2] float32 (ACT_F32) or float64
    float *reward;                         // in/out, sticky
    uint8_t *flags;                        // in/out, sticky
    const double *targets;                 // optional per-env cartesian targets [n][2], or nullptr
    unsigned long long *stats;             // or nullptr
    int64_t n, env_id0;
    // optional outputs of ag_step: the stepped pose's end effector and goal distances [n][2], K2's first_hit [n]
    double *ee, *dist;
    int32_t *first_hit;                    // WANT_FIRST only
    // optional outputs of ag_step_obs: this step's return values, the observations, the crop; reset_ctr with auto_reset
    uint32_t *reset_ctr, *ep_len;
    double *obs, *final_obs;
    float *reward_out;
    uint8_t *terminated, *collision, *crop;
    int32_t crop_size, auto_reset;
    uint64_t seed;
};

__device__ __forceinline__ void write_obs(double *o, double q1, double q2, const Arm &A, double tx, double ty) {
    reinterpret_cast<double2 *>(o)[0] = make_double2(q1, q2);
    reinterpret_cast<double2 *>(o)[1] = make_double2(A.gx, A.gy);
    reinterpret_cast<double2 *>(o)[2] = make_double2(fabs(__dsub_rn(tx, A.gx)), fabs(__dsub_rn(ty, A.gy)));
}

// WANT_FIRST: the collision flag and first_hit with the EXACT (or BRUTE) arithmetic of K2; the launcher runs the EXACT
// kernel for the FAST engine
template <int ENGINE, bool ACT_F32, bool WANT_FIRST>
__global__ void __launch_bounds__(AG_BLOCK) k_step(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G,
                                                   const __grid_constant__ StepDev D) {
    static_assert(!(WANT_FIRST && ENGINE == AG_ENGINE_FAST), "first_hit runs the EXACT kernel");
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    __shared__ unsigned long long s_acc[AG_ST_COUNT];
    if (threadIdx.x < AG_ST_COUNT) s_acc[threadIdx.x] = 0;
    const BlockCtx B = block_prologue<ENGINE>(G, D.env_id0, D.n, smem, &s_fl);
    __syncthreads();
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < D.n) {
        const FastConst C = make_fast_const(P, G);
        double tx = P.target_x, ty = P.target_y;
        if (D.targets) { const double2 tg = reinterpret_cast<const double2 *>(D.targets)[e]; tx = tg.x; ty = tg.y; }
        double d1, d2;
        if (ACT_F32) { const float2 a = reinterpret_cast<const float2 *>(D.actions)[e]; d1 = (double)a.x; d2 = (double)a.y; }
        else { const double2 a = reinterpret_cast<const double2 *>(D.actions)[e]; d1 = a.x; d2 = a.y; }
        double q1 = __dadd_rn(D.j1[e], d1), q2 = __dadd_rn(D.j2[e], d2);      // two_joint_robot.py:71-72
        float rw = D.reward[e];
        uint32_t fl = D.flags[e];
        Arm A = forward_kinematics(q1, q2, P.link_1, P.link_2);
        int fh = INT_MAX, axis = 0;
        bool h;
        if constexpr (ENGINE == AG_ENGINE_FAST) h = fast_arm_collides(P, G, B.V, B.fl, C, A, axis);
        else h = arm_collides<ENGINE, WANT_FIRST>(G, B.V, A, P.section_eps, fh, axis);
        if (h) { rw = (float)P.reward_collision; fl |= AG_FLAG_COLLISION; }      // scene_0.py:95-97
        const bool reached = P.choose_j_tar ? target_reached_joint(P, q1, q2)
                                            : (fabs(__dsub_rn(tx, A.gx)) < P.reach_eps && fabs(__dsub_rn(ty, A.gy)) < P.reach_eps);
        if (reached) { rw = (float)P.reward_reach; fl |= AG_FLAG_DONE; }         // :98-100
        if (WANT_FIRST) D.first_hit[e] = h ? fh : -1;
        if (D.ee) reinterpret_cast<double2 *>(D.ee)[e] = make_double2(A.gx, A.gy);
        if (D.dist) reinterpret_cast<double2 *>(D.dist)[e] = make_double2(fabs(__dsub_rn(tx, A.gx)), fabs(__dsub_rn(ty, A.gy)));
        if (D.reward_out) D.reward_out[e] = rw;
        if (D.terminated) D.terminated[e] = fl != 0 ? 1 : 0;
        if (D.collision) D.collision[e] = (fl & AG_FLAG_COLLISION) ? 1 : 0;
        if (D.final_obs) write_obs(D.final_obs + e * AG_OBS_DIM, q1, q2, A, tx, ty);
        uint32_t el = (D.ep_len ? D.ep_len[e] : 0u) + 1;
        acc32(s_acc, AG_ST_ENV_STEPS, 1);
        if (fl != 0 && D.auto_reset) {                                           // experiment_0.py:30-34
            acc32(s_acc, AG_ST_EPISODES, 1);
            if (fl & AG_FLAG_COLLISION) acc32(s_acc, AG_ST_COLLISIONS, 1);
            if (fl & AG_FLAG_DONE) acc32(s_acc, AG_ST_SUCCESSES, 1);
            atomicAdd(&s_acc[AG_ST_EP_LEN_SUM], (unsigned long long)el);
            acc32(s_acc, AG_ST_RETURN_MILLI, __float2int_rn(rw * 1e-3f));
            if (h) {                                                             // Scene.reset(): resample only while colliding
                uint32_t rc = D.reset_ctr[e];
                resample_pose<ENGINE, false>(P, G, B, C, true, q1, q2, rc, nullptr, 0, D.seed, (uint64_t)(D.env_id0 + e), s_acc);
                D.reset_ctr[e] = rc;
                A = forward_kinematics(q1, q2, P.link_1, P.link_2);
            }
            rw = 0.0f; fl = 0; el = 0;                                           // scene_0.py:111-113
        }
        if (axis) acc32(s_acc, AG_ST_AXIS_ALIGNED, axis);
        D.j1[e] = q1; D.j2[e] = q2; D.reward[e] = rw; D.flags[e] = (uint8_t)fl;
        if (D.ep_len) D.ep_len[e] = el;
        if (D.obs) write_obs(D.obs + e * AG_OBS_DIM, q1, q2, A, tx, ty);
        if (D.crop) {                                                            // local occupancy around the end effector
            // the end effector's own cell, not clamped to [-1, S] as row_of / col_of do for the traversal: an arm
            // that reaches past the grid sees only cells outside it
            const int64_t r0 = (int64_t)(floor((G.half - A.gy) * G.inv_side) + 1.0), c0 = (int64_t)floor((A.gx + G.half) * G.inv_side);
            const int hc = D.crop_size / 2;
            uint8_t *o = D.crop + e * (int64_t)D.crop_size * D.crop_size;
            for (int dr = 0; dr < D.crop_size; ++dr)
                for (int dc = 0; dc < D.crop_size; ++dc) {
                    const int64_t r = r0 - hc + dr, c = c0 - hc + dc;
                    uint8_t v = 2;
                    if (r >= 0 && r < G.S && c >= 0 && c < G.S) v = (B.V.bits[r * G.wpr + (c >> 5)] >> (c & 31)) & 1u;
                    o[dr * D.crop_size + dc] = v;
                }
        }
    }
    stats_flush(s_acc, D.stats);
}

// ------------------------------------------------------------------------------------------- K4
// experiment/experiment_0.py:20-34 fused over K steps; env state lives in registers for the
// whole launch, the only per-step HBM traffic is the action read and the record write.
//
// Register discipline: the hot loop keeps (q1, q2, reward, flags, ep_len, prefetched action) live;
// everything an episode end needs (reset counter, Philox key, candidate list) is re-derived
// inside the out-of-line cold_terminal(), so the loop fits the register budget without spills.
template <int ENGINE, int BP>
__device__ __forceinline__ int step_decide(const ag_params &P, const GridDev &G, const BlockCtx &B,
                                           const FastConst &C, double q1, double q2, const double *tgt) {
    if constexpr (ENGINE == AG_ENGINE_FAST) {
        return fast_decide<BP>(P, G, B.V, B.fl, C, q1, q2, true, tgt);
    } else {
        const Arm A = forward_kinematics(q1, q2, P.link_1, P.link_2);
        int fh = 0, axis = 0;
        const bool h = arm_collides<ENGINE, false>(G, B.V, A, P.section_eps, fh, axis);
        return (h ? 1 : 0) | (target_reached_at(P, q1, q2, A, tgt) ? 2 : 0) | (axis << 2);
    }
}

// Everything thread-private that the hot loop carries.  It lives in registers inside the inner loops and is
// parked in this shared-memory block (structure of arrays: conflict-free) only around the out-of-line cold
// section, so that no value is live across the ABI call: that is what keeps the inner loop spill-free under a
// 64-register budget (DESIGN.md "register allocation of K4").  It used to be a struct in local memory; ncu
// counted 37 M local-memory sectors per launch for it -- as much L2 traffic as the action and record streams.
template <int BLOCK>
struct HotShared {
    double q1[BLOCK], q2[BLOCK];
    const float2 *act[BLOCK];   // action row of step t + AG_RING - 1: the next one to prefetch
    int64_t o[BLOCK];           // record offset of step t
    float rw[BLOCK];
    uint32_t flags[BLOCK];
    int el_off[BLOCK];          // episode length after step t = el_off + t + 1
    int t[BLOCK], d[BLOCK];
    int undecided[BLOCK];       // 0, or 16 | c | r << 2: the float32 filter's verdicts (2 = undecided) of step t
};

// Action prefetch ring: every thread streams its own actions global -> shared with cp.async (LDGSTS), AG_RING - 1
// steps ahead of their use, so that no register and no warp ever waits for a DRAM round trip (with a
// register prefetch one step ahead, 37 % of all stall samples were long-scoreboard waits on that load:
// profiles/r1g).  Slot (t mod AG_RING) of row threadIdx.x holds the action of step t.
constexpr int AG_RING = 4;

// Cold section, out of line: (1) finish a step whose float32 filter was undecided with the
// float64 reference arithmetic, (2) episode end (experiment_0.py:30-34): statistics + Scene.reset().
template <int ENGINE, int BP, bool HAS_RESET_U, bool RECORD, int BLOCK>
__device__ __noinline__ void cold_section(const ag_params &P, const GridDev &G, const FastConst &C, const RolloutDev &A,
                                          HotShared<BLOCK> &hs, const FastList *fl_list, unsigned long long *s_acc) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int x = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + x;
    double q1 = hs.q1[x], q2 = hs.q2[x];
    float rw = hs.rw[x];
    uint32_t fl = hs.flags[x];
    int d = hs.d[x];
    const int t = hs.t[x], und = hs.undecided[x];
    BlockCtx B;
    B.V = thread_view(G, smem, A.env_id0 + e);
    B.fl = fl_list;
    if (und) {
        acc32(s_acc, AG_ST_COUNT + AG_DIAG_EXACT_STEPS, 1);
        double txd = P.target_x, tyd = P.target_y;
        if (A.targets != nullptr) { const double2 tg = reinterpret_cast<const double2 *>(A.targets)[e]; txd = tg.x; tyd = tg.y; }
        d = cold_exact_decide_at(P, G, B.V, B.fl, q1, q2, und & 3, (und >> 2) & 3, txd, tyd);  // the filter's verdicts
        if (d & 1) { rw = (float)P.reward_collision; fl |= AG_FLAG_COLLISION; }   // scene_0.py:95-97
        if (d & 2) { rw = (float)P.reward_reach; fl |= AG_FLAG_DONE; }            // :98-100
        store_record<RECORD>(A, hs.o[x], q1, q2, rw, fl);                         // experiment_0.py:23-25
        emit_event(A, e, t, rw, fl);
    }
    if (d >> 2) acc32(s_acc, AG_ST_AXIS_ALIGNED, d >> 2);
    if (fl) {                                                                     // experiment_0.py:30-34
        acc32(s_acc, AG_ST_EPISODES, 1);
        if (fl & AG_FLAG_COLLISION) acc32(s_acc, AG_ST_COLLISIONS, 1);
        if (fl & AG_FLAG_DONE) acc32(s_acc, AG_ST_SUCCESSES, 1);
        atomicAdd(&s_acc[AG_ST_EP_LEN_SUM], (unsigned long long)(uint32_t)(hs.el_off[x] + t + 1));
        acc32(s_acc, AG_ST_RETURN_MILLI, __float2int_rn(rw * 1e-3f));
        if (d & 1) {   // Scene.reset(): the pose is unchanged since the step, so collision_check() == (d & 1)
            uint32_t rc = A.reset_ctr[e];
            resample_pose<ENGINE, HAS_RESET_U, BP>(P, G, B, C, true, q1, q2, rc,
                                                   HAS_RESET_U ? A.reset_u + e * A.R * 2 : nullptr, A.R, A.seed,
                                                   (uint64_t)(A.env_id0 + e), s_acc);
            A.reset_ctr[e] = rc;
        }
        rw = 0.0f; fl = 0; hs.el_off[x] = -(t + 1);                               // scene_0.py:111-113
    }
    hs.q1[x] = q1; hs.q2[x] = q2; hs.rw[x] = rw; hs.flags[x] = fl;
    hs.t[x] = t + 1; hs.o[x] += A.row_stride;
}

// Three nested loops, warp-synchronous (every lane of a warp is at the same step t, so action loads and
// record stores stay coalesced):
//   inner  : uneventful steps only -- float32 FK, broad_list(), the reach pre-test and the record of
//            an uneventful step (reward 0, flags 0); branch-free, call-free, ~150 instructions that stay
//            resident in the instruction cache.  A lane is "slow" when a link's box comes within the margin
//            of a square, the end effector is within the margin of the target box, its angles are out of the
//            filter's range or its sticky state is not clean; the warp leaves the loop when ANY lane is slow.
//   middle : the narrow phase for the slow lanes (inline, placed after the inner loop); if no lane has an
//            event -- collision, target reached, undecided filter, axis-aligned evaluation -- the warp
//            goes straight back into the inner loop.
//   outer  : event lanes run the out-of-line cold_section() (the only call; registers are exchanged
//            through HotShared), then the warp re-enters in lockstep.
// The EXACT / BRUTE reference engines have no pre-test (every step is "slow"); the FAST engine on grids that need
// the cell traversal runs k_rollout_async instead.
template <int ENGINE, int BP, bool HAS_ACT, bool HAS_RESET_U, bool RECORD, bool FULL, int BLOCK>
__global__ void __launch_bounds__(BLOCK, (ENGINE == AG_ENGINE_FAST ? (BP == BP_LIST ? AG_FAST_BLOCKS_PER_SM : 2) : 1) * (AG_BLOCK / BLOCK))
k_rollout(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G, const __grid_constant__ FastConst C,
          const __grid_constant__ RolloutDev A) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    __shared__ unsigned long long s_acc[AG_ST_COUNT + AG_DIAG_COUNT];
    __shared__ HotShared<BLOCK> hs;
    __shared__ __align__(16) float2 s_ring[HAS_ACT ? AG_RING * BLOCK : 1];
    __shared__ __align__(16) float4 s_arm[(ENGINE == AG_ENGINE_FAST && BP == BP_LIST) ? BLOCK : 1];   // float32 arm of a slow lane
    if (threadIdx.x < AG_ST_COUNT + AG_DIAG_COUNT) s_acc[threadIdx.x] = 0;
    const BlockCtx B0 = block_prologue<ENGINE>(G, A.env_id0, A.n, smem, &s_fl);
    __syncthreads();
    constexpr bool LIST = (ENGINE == AG_ENGINE_FAST && BP == BP_LIST);
    const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e0 < A.n) {
        const int x = threadIdx.x;
        hs.q1[x] = A.j1[e0]; hs.q2[x] = A.j2[e0]; hs.rw[x] = A.reward[e0]; hs.flags[x] = A.flags[e0];
        hs.el_off[x] = (int)A.ep_len[e0];
        hs.act[x] = nullptr;
        const uint32_t ring0 = smem_u32(&s_ring[HAS_ACT ? threadIdx.x : 0]);     // this thread's column of the ring
        if (HAS_ACT) {                                                           // steps 0 .. AG_RING-2 in flight
            const float2 *p = reinterpret_cast<const float2 *>(A.actions) + e0;
#pragma unroll
            for (int i = 0; i < AG_RING - 1; ++i) {
                if (i < A.K) cp_async8(ring0 + (uint32_t)i * (BLOCK * 8), p);
                cp_async_commit();
                p += A.row_stride;
            }
            hs.act[x] = p;
        }
        hs.o[x] = e0; hs.t[x] = 0; hs.d[x] = 0; hs.undecided[x] = 0;
        const uint32_t lane_mask = __activemask();
        if (RECORD && LIST && A.zfill) zero_fill_warp(A, e0 - (threadIdx.x & 31));
        const uint32_t sc0 = A.step_ctr[e0];
        A.step_ctr[e0] = sc0 + (uint32_t)A.K;
        const float reach_thr_clean = C.reach_eps + (AG_DELTA_P + 2.0e-7f);      // reach_fast()'s margin
        const double *tgt = A.targets ? A.targets + 2 * e0 : nullptr;            // per-env target override
        float ltx = C.tx, lty = C.ty;
        if (tgt != nullptr) { ltx = (float)tgt[0]; lty = (float)tgt[1]; }
        for (;;) {                                                               // ---- outer
            // hot state: struct -> registers
            double q1 = hs.q1[x], q2 = hs.q2[x];
            float rw = hs.rw[x];
            uint32_t fl = hs.flags[x];
            const uint32_t warp_mask = FULL ? 0xFFFFFFFFu : lane_mask;   // FULL: n % 32 == 0, every warp is complete
            const float2 *act = hs.act[x];
            int64_t o = hs.o[x];
            int t = hs.t[x], d = 0, cr = 0;
            bool undecided = false, event = false;
            // a lane whose sticky state is not clean (flags / reward left by earlier step() calls) is
            // forced through the slow branch: an infinite threshold makes its reach pre-test fire
            float reach_thr = ((fl != 0) | (rw != 0.0f)) ? __int_as_float(0x7f800000) : reach_thr_clean;
            BlockCtx B;
            B.V = B0.V; B.fl = LIST ? &s_fl : B0.fl;
            const uint64_t gid = (uint64_t)(A.env_id0 + e0);
            for (;;) {                                                           // ---- middle
                bool slow = true;
#pragma unroll 1
                for (; t < A.K; ++t, o += A.row_stride) {                        // ---- inner
                    double d1, d2;
                    if (HAS_ACT) {
                        if (t + (AG_RING - 1) < A.K)                             // refill the slot consumed last step
                            cp_async8(ring0 + ((uint32_t)(t + AG_RING - 1) & (AG_RING - 1)) * (BLOCK * 8), act);
                        cp_async_commit();
                        act += A.row_stride;
                        cp_async_wait<AG_RING - 1>();                            // this step's action has landed
                        const float2 an = s_ring[((uint32_t)t & (AG_RING - 1)) * BLOCK + threadIdx.x];
                        d1 = (double)an.x; d2 = (double)an.y;
                    } else {
                        philox_action(P, A.seed, gid, sc0 + (uint32_t)t, d1, d2);
                    }
                    q1 = __dadd_rn(q1, d1); q2 = __dadd_rn(q2, d2);              // two_joint_robot.py:71-72
                    if constexpr (LIST) {
                        bool ok;
                        const ArmF a = fast_forward_kinematics(q1, q2, C, ok);
                        const float sep = broad_list(s_fl, a);
                        const float worst = fmaxf(fabsf(ltx - a.gx), fabsf(lty - a.gy));
                        slow = !(sep >= s_fl.hm) | !(worst >= reach_thr) | !ok;             // NaN-safe: NaN is slow
                        if (P.choose_j_tar) slow |= target_reached_joint(P, q1, q2);
                        if (slow) s_arm[threadIdx.x] = make_float4(a.ex, a.ey, ok ? a.gx : __int_as_float(0x7fc00000), a.gy);
                        store_uneventful<RECORD>(A, o, q1, q2);                  // slow lanes rewrite theirs
                    }
                    if (__any_sync(warp_mask, slow)) break;
                }
                if (t >= A.K) break;
                event = false;
                // Narrow phase of the slow lanes, warp-cooperative when the warp is complete: a slow lane has at most
                // 2 * AG_LIST_MAX = 16 (link, square) pairs, so lane L of the warp takes pair (link L & 1, square L >> 1)
                // of the slow lane's stashed arm and one pass of narrow_f32 settles them all (instead of one lane
                // looping over its candidates while 31 wait).
                int c_coop = 0;
                if constexpr (LIST && FULL) {
                    uint32_t todo = __ballot_sync(0xFFFFFFFFu, slow);
                    const int lane = threadIdx.x & 31, m2 = 2 * s_fl.m;
                    while (todo) {                                               // warp-uniform: usually one pass
                        const int src = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const float4 af = s_arm[(threadIdx.x & ~31) + src];
                        int v = 0;
                        if (lane < m2) {
                            const float4 q = s_fl.sq[lane >> 1];
                            const bool second = (lane & 1) != 0;
                            const LinkF L = make_link_f(second ? af.x : 0.0f, second ? af.y : 0.0f, second ? af.z : af.x,
                                                        second ? af.w : af.y, C.side);
                            v = narrow_f32(L, q.x, q.y, q.z, q.w);
                        }
                        const uint32_t hit = __ballot_sync(0xFFFFFFFFu, v == 1), und = __ballot_sync(0xFFFFFFFFu, v == 2);
                        if (lane == src) c_coop = hit ? 1 : (und ? 2 : 0);
                    }
                }
                if (slow) {
                    if constexpr (LIST) {
                        const float4 af = s_arm[threadIdx.x];                    // stashed by this lane in the inner loop
                        ArmF a;                                                  // (keeping it in registers costs spills there)
                        a.ex = af.x; a.ey = af.y; a.gx = af.z; a.gy = af.w;
                        const bool ok = (af.z == af.z);                          // NaN marks angles outside the filter's range
                        const int c = (ok && s_fl.m >= 0) ? (FULL ? c_coop : arm_fast_list(&s_fl, a, C)) : 2;
                        int r;
                        if (P.choose_j_tar) r = target_reached_joint(P, q1, q2) ? 1 : 0;
                        else r = ok ? reach_fast_at(C, a, ltx, lty) : 2;
                        undecided = ((c | r) & 2) != 0;
                        cr = c | (r << 2);
                        d = (c & 1) | ((r & 1) << 1);
                    } else {
                        d = step_decide<ENGINE, BP>(P, G, B, C, q1, q2, tgt);
                    }
                    event = undecided;
                    if (!undecided) {
                        if (d & 1) { rw = (float)P.reward_collision; fl |= AG_FLAG_COLLISION; }   // scene_0.py:95-97
                        if (d & 2) { rw = (float)P.reward_reach; fl |= AG_FLAG_DONE; }            // :98-100
                        if (!LIST || fl != 0 || rw != 0.0f) {                                      // else: already recorded
                            store_record<RECORD>(A, o, q1, q2, rw, fl);                            // experiment_0.py:23-25
                            emit_event(A, e0, t, rw, fl);
                        }
                        event = (fl | (d >> 2)) != 0;
                        reach_thr = (rw != 0.0f) ? __int_as_float(0x7f800000) : reach_thr_clean;
                    }
                }
                if (__any_sync(warp_mask, event)) break;                         // warp-uniform exit to the cold section
                ++t; o += A.row_stride;
            }
            // registers -> struct
            hs.q1[x] = q1; hs.q2[x] = q2; hs.rw[x] = rw; hs.flags[x] = fl;
            if (t >= A.K) break;
            hs.act[x] = act; hs.o[x] = o; hs.t[x] = t; hs.d[x] = d; hs.undecided[x] = undecided ? (cr | 16) : 0;
            if (event) {
                acc32(s_acc, AG_ST_COUNT + AG_DIAG_COLD_CALLS, 1);
                cold_section<ENGINE, BP, HAS_RESET_U, RECORD, BLOCK>(P, G, C, A, hs, B0.fl, s_acc);
            } else { hs.t[x] = t + 1; hs.o[x] = o + A.row_stride; }
            if ((threadIdx.x & 31) == 0) acc32(s_acc, AG_ST_COUNT + AG_DIAG_WARP_EXITS, 1);
        }
        acc32(s_acc, AG_ST_ENV_STEPS, A.K);
        A.j1[e0] = hs.q1[x]; A.j2[e0] = hs.q2[x]; A.reward[e0] = hs.rw[x]; A.flags[e0] = (uint8_t)hs.flags[x];
        A.ep_len[e0] = (uint32_t)(hs.el_off[x] + A.K);
    }
    stats_flush(s_acc, A.stats);
    if (A.diag != nullptr && threadIdx.x < AG_DIAG_COUNT) {
        const unsigned long long v = s_acc[AG_ST_COUNT + threadIdx.x];
        if (v != 0) atomicAdd(&A.diag[threadIdx.x], v);
    }
}

// ------------------------------------------------------------------------------------------- K4, dense maps
// Lane-asynchronous form of the same loop for grids that go through the cell traversal (high-resolution
// and per-batch maps, BASELINE configs 4/5).  There an episode ends every second or third step and
// Scene.reset() needs ~3 candidates on average, so a warp-synchronous kernel idles most lanes: a step
// costs 1 pose check but the warp waits for the slowest lane's rejection loop (the maximum of 32 geometric
// draws, ~9 checks).  Here every lane is a small state machine -- STEP (consume the action of its own step t)
// or RESET (consume its next reset candidate) -- and each loop iteration runs exactly ONE pose check per lane,
// so the expensive part (FK + traversal + narrow phase) is executed by all 32 lanes together whatever their
// mode.  Lanes drift apart in t, so action loads / record stores are per-lane (sector-granular); this path
// is bound by the traversal (thousands of instructions per check), not by memory.
#ifndef AG_ASYNC_BLOCKS_PER_SM
#define AG_ASYNC_BLOCKS_PER_SM 2
#endif
template <int BP, bool HAS_ACT, bool HAS_RESET_U, bool RECORD>
__global__ void __launch_bounds__(AG_BLOCK, AG_ASYNC_BLOCKS_PER_SM)
k_rollout_async(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G, const __grid_constant__ FastConst C,
                const __grid_constant__ RolloutDev A) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FastList s_fl;
    __shared__ unsigned long long s_acc[AG_ST_COUNT + AG_DIAG_COUNT];
    if (threadIdx.x < AG_ST_COUNT + AG_DIAG_COUNT) s_acc[threadIdx.x] = 0;
    const BlockCtx B = block_prologue<AG_ENGINE_FAST>(G, A.env_id0, A.n, smem, &s_fl);
    __syncthreads();
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    long long loc[AG_ST_COUNT];
#pragma unroll
    for (int i = 0; i < AG_ST_COUNT; ++i) loc[i] = 0;
    if (e < A.n) {
        double q1 = A.j1[e], q2 = A.j2[e];
        float rw = A.reward[e];
        uint32_t fl = A.flags[e], el = A.ep_len[e], rc = A.reset_ctr[e];
        const uint32_t sc0 = A.step_ctr[e];
        A.step_ctr[e] = sc0 + (uint32_t)A.K;
        const uint64_t gid = (uint64_t)(A.env_id0 + e);
        const double *ru = HAS_RESET_U ? A.reset_u + e * A.R * 2 : nullptr;
        const double *tgt = A.targets ? A.targets + 2 * e : nullptr;             // per-env target override
        int t = 0, tries = 0;
        bool resetting = false;
        while (t < A.K || resetting) {
            const unsigned live = __activemask();                                // the lanes still in the loop
            bool stuck = false;
            if (!resetting) {                                                    // ---- STEP: experiment_0.py:21-22
                double d1, d2;
                if (HAS_ACT) {
                    const float2 a = __ldcs(reinterpret_cast<const float2 *>(A.actions) + (int64_t)t * A.row_stride + e);
                    d1 = (double)a.x; d2 = (double)a.y;
                } else {
                    philox_action(P, A.seed, gid, sc0 + (uint32_t)t, d1, d2);
                }
                q1 = __dadd_rn(q1, d1); q2 = __dadd_rn(q2, d2);                  // two_joint_robot.py:71-72
            } else if (tries >= P.max_reset_tries || (HAS_RESET_U && rc >= (uint32_t)A.R)) {
                stuck = true;                                                    // give up: keep the last candidate
            } else {                                                             // ---- RESET: scene_0.py:179-181
                reset_candidate<HAS_RESET_U>(A.seed, gid, rc, ru, q1, q2);
                ++tries;
            }
            // ---- one pose check per lane and iteration, whatever the mode, with all lanes converged
            __syncwarp(live);
            const int d = stuck ? 0 : fast_decide<BP>(P, G, B.V, B.fl, C, q1, q2, !resetting, tgt);
            __syncwarp(live);
            loc[AG_ST_AXIS_ALIGNED] += d >> 2;
            if (!resetting) {
                if (d & 1) { rw = (float)P.reward_collision; fl |= AG_FLAG_COLLISION; }   // scene_0.py:95-97
                if (d & 2) { rw = (float)P.reward_reach; fl |= AG_FLAG_DONE; }            // :98-100
                store_record<RECORD>(A, (int64_t)t * A.row_stride + e, q1, q2, rw, fl);    // experiment_0.py:23-25
                emit_event(A, e, t, rw, fl);
                ++el; ++t;
                if (fl) {                                                        // experiment_0.py:30-34
                    ++loc[AG_ST_EPISODES];
                    loc[AG_ST_COLLISIONS] += (fl & AG_FLAG_COLLISION) ? 1 : 0;
                    loc[AG_ST_SUCCESSES] += (fl & AG_FLAG_DONE) ? 1 : 0;
                    loc[AG_ST_EP_LEN_SUM] += el;
                    loc[AG_ST_RETURN_MILLI] += __float2int_rn(rw * 1e-3f);
                    rw = 0.0f; fl = 0; el = 0;                                   // scene_0.py:111-113
                    resetting = (d & 1) != 0;                                    // random_valid_pose() only while colliding
                    tries = 0;
                }
            } else if (stuck) {
                ++loc[AG_ST_STUCK_RESETS];
                resetting = false;
            } else if (!(d & 1)) {
                resetting = false;                                               // candidate accepted
            }
        }
        loc[AG_ST_ENV_STEPS] = A.K;
        A.j1[e] = q1; A.j2[e] = q2; A.reward[e] = rw; A.flags[e] = (uint8_t)fl;
        A.ep_len[e] = el; A.reset_ctr[e] = rc;
    }
    block_accumulate_stats(loc, A.stats, s_acc);
}

// ------------------------------------------------------------------------------------- host side
#define AG_DISPATCH_ENGINE(engine, ...)                                   \
    switch (engine) {                                                     \
        case AG_ENGINE_EXACT: { constexpr int E = AG_ENGINE_EXACT; __VA_ARGS__; break; } \
        case AG_ENGINE_FAST:  { constexpr int E = AG_ENGINE_FAST;  __VA_ARGS__; break; } \
        case AG_ENGINE_BRUTE: { constexpr int E = AG_ENGINE_BRUTE; __VA_ARGS__; break; } \
        default: return AG_ERR_MODE;                                      \
    }

// K1 / K2 with first_hit: the FAST engine computes the flag with the EXACT arithmetic (pose_collides, k_step), so those
// launches run the EXACT kernels
constexpr int first_hit_engine(int engine) { return engine == AG_ENGINE_FAST ? AG_ENGINE_EXACT : engine; }

template <int E, bool F32, bool WF>
ag_status launch_step_k(const ag_params &P, const GridDev &G, const StepDev &D, size_t smem, cudaStream_t s) {
    auto k = k_step<E, F32, WF>;
    ag_status st = set_smem(k, smem);
    if (st) return st;
    k<<<blocks_for(D.n), AG_BLOCK, smem, s>>>(P, G, D);
    return launched();
}

// K1 / K6: the k_step of the engine, the action dtype and first_hit (which only ag_step asks for)
ag_status launch_step(const ag_params &P, const GridDev &G, const StepDev &D, int engine, bool f32, size_t smem,
                      cudaStream_t s) {
    AG_DISPATCH_ENGINE(engine, {
        constexpr int EF = first_hit_engine(E);
        if (D.first_hit)
            return f32 ? launch_step_k<EF, true, true>(P, G, D, smem, s) : launch_step_k<EF, false, true>(P, G, D, smem, s);
        return f32 ? launch_step_k<E, true, false>(P, G, D, smem, s) : launch_step_k<E, false, false>(P, G, D, smem, s);
    });
}

template <int E, int BP, bool HA, bool HR, bool REC, bool FULL, int BLOCK>
ag_status launch_rollout_b(const ag_params &P, const GridDev &G, const RolloutDev &A, size_t smem, cudaStream_t s) {
    auto k = k_rollout<E, BP, HA, HR, REC, FULL, BLOCK>;
    ag_status st = set_smem(k, smem);
    if (st) return st;
    k<<<(unsigned)((A.n + BLOCK - 1) / BLOCK), BLOCK, smem, s>>>(P, G, make_fast_const(P, G), A);
    return launched();
}

// Block size of the rollout kernel.  A block lasts as long as its slowest warp (cold-section visits are
// Poisson-distributed per warp), and a finished warp's slot stays idle until the block retires, so
// scene_0-class launches (obstacle list: per-block set-up is ~100 instructions) use one-warp blocks;
// 256 threads remain for staged per-batch grids, where a block shares one shared-memory copy.
constexpr int AG_SMALL_BLOCK =
#ifdef AG_ROLLOUT_SMALL_BLOCK
    AG_ROLLOUT_SMALL_BLOCK;
#else
    32;
#endif

template <int E, int BP, bool HA, bool HR, bool REC>
ag_status launch_rollout_t(const ag_params &P, const GridDev &G, const RolloutDev &A, size_t smem, cudaStream_t s) {
    if constexpr (E == AG_ENGINE_FAST && BP == BP_TRAVERSAL) {       // dense maps: lane-asynchronous kernel
        auto k = k_rollout_async<BP, HA, HR, REC>;
        ag_status st = set_smem(k, smem);
        if (st) return st;
        k<<<blocks_for(A.n), AG_BLOCK, smem, s>>>(P, G, make_fast_const(P, G), A);
        return launched();
    } else if constexpr (E == AG_ENGINE_FAST) {                      // obstacle list
        if (G.n_grids == 1) {
            // complete warps only (n % 32 == 0): the warp votes use a constant full mask
            if (A.n % 32 == 0) return launch_rollout_b<E, BP, HA, HR, REC, true, AG_SMALL_BLOCK>(P, G, A, smem, s);
            return launch_rollout_b<E, BP, HA, HR, REC, false, AG_SMALL_BLOCK>(P, G, A, smem, s);
        }
        return launch_rollout_b<E, BP, HA, HR, REC, false, AG_BLOCK>(P, G, A, smem, s);
    } else {                                                         // EXACT / BRUTE
        return launch_rollout_b<E, BP, HA, HR, REC, false, AG_BLOCK>(P, G, A, smem, s);
    }
}

template <int E, int BP>
ag_status launch_rollout_e(const ag_params &P, const GridDev &G, const RolloutDev &A, size_t smem, cudaStream_t s) {
    const bool ha = A.actions != nullptr, hr = A.reset_u != nullptr, rec = A.rec_j1 != nullptr;
#define AG_RO(HA, HR, REC) return launch_rollout_t<E, BP, HA, HR, REC>(P, G, A, smem, s)
    if (ha) { if (hr) { if (rec) AG_RO(true, true, true); else AG_RO(true, true, false); }
              else    { if (rec) AG_RO(true, false, true); else AG_RO(true, false, false); } }
    else    { if (hr) { if (rec) AG_RO(false, true, true); else AG_RO(false, true, false); }
              else    { if (rec) AG_RO(false, false, true); else AG_RO(false, false, false); } }
#undef AG_RO
}

}  // namespace

void ag_note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

// the largest grid footprint (bits, transposed bits, two-level form, cell tables) a block copies to shared memory
constexpr size_t STAGE_MAX_BYTES = 32768;

ag_status make_grid_dev(const ag_params *p, const ag_grid *g, int64_t env_id0, int engine, GridDev *out,
                        size_t *smem_bytes) {
    if (!g || !g->bits || !g->min_x || !g->min_y) return AG_ERR_NULL;
    if (g->S < 2 || g->words_per_row != (g->S + 31) / 32 || g->n_grids < 1 || g->envs_per_grid < 1 ||
        g->grid_stride_words < (int64_t)g->S * g->words_per_row)
        return AG_ERR_SHAPE;
    // the FAST engine's error budget (ag_fast.cuh) assumes scene_0-class magnitudes
    if (engine == AG_ENGINE_FAST && p &&
        !(p->link_1 > 0 && p->link_2 > 0 && p->link_1 <= 1.0 && p->link_2 <= 1.0 && g->env_size <= 4.0))
        return AG_ERR_MODE;
    GridDev d;
    d.bits = g->bits; d.bits_t = g->bits_t; d.min_x = g->min_x; d.min_y = g->min_y;
    d.T = (g->S + 7) / 8; d.cwpr = (d.T + 31) / 32;
    d.hier = d.T <= AG_HIER_MAX_T ? reinterpret_cast<const unsigned char *>(g->hier) : nullptr;   // larger maps: the row walk
    d.hier_tiles_bytes = (int32_t)((((int64_t)d.T * d.T + 1) & ~(int64_t)1) * 8);
    d.hier_coarse_words = (int32_t)(((int64_t)d.T * d.cwpr + 3) & ~(int64_t)3);
    d.hier_bytes = (int32_t)ag_grid_hier_bytes(g->S);
    d.side = g->side; d.half = g->env_size / 2.0; d.inv_side = 1.0 / g->side;
    d.margin = 1e-9 * g->env_size;
    d.S = g->S; d.wpr = g->words_per_row; d.n_grids = g->n_grids;
    d.stride_words = g->grid_stride_words; d.envs_per_grid = g->envs_per_grid;
    const int spad = (g->S + 1) & ~1;
    const size_t bytes = 16 + (size_t)g->grid_stride_words * 4 * (g->bits_t ? 2 : 1) + (d.hier ? (size_t)d.hier_bytes : 0) +
                         (size_t)spad * 16;
    const bool uniform = g->n_grids == 1 || (g->envs_per_grid % AG_BLOCK == 0 && env_id0 % AG_BLOCK == 0);
    const bool aligned = ((uintptr_t)g->bits % 16 == 0) && ((uintptr_t)g->bits_t % 16 == 0) && ((uintptr_t)g->hier % 16 == 0) &&
                         (g->grid_stride_words % 4 == 0);
    d.stage = (uniform && aligned && bytes <= STAGE_MAX_BYTES) ? 1 : 0;
    *smem_bytes = d.stage ? bytes : 0;
    *out = d;
    return AG_OK;
}

ag_status ag_rollout_impl(const ag_params *p, const ag_grid *g, const ag_rollout_args *a, int64_t row_stride,
                          void *stream) {
    if (!p || !g || !a) return AG_ERR_NULL;
    if (a->n < 0 || a->K < 1 || a->K > AG_MAX_K) return AG_ERR_SHAPE;
    if (a->n == 0) return AG_OK;
    if (!a->j1 || !a->j2 || !a->reward || !a->flags || !a->step_ctr || !a->reset_ctr || !a->ep_len || !a->stats)
        return AG_ERR_NULL;
    const int nrec = (a->rec_j1 != nullptr) + (a->rec_j2 != nullptr) + (a->rec_reward != nullptr) + (a->rec_flags != nullptr);
    const bool joints_only = nrec == 2 && a->rec_j1 != nullptr && a->rec_j2 != nullptr;
    if (nrec != 0 && nrec != 4 && !joints_only) return AG_ERR_NULL;
    if (a->events != nullptr && (a->event_count == nullptr || a->event_capacity < 0)) return AG_ERR_NULL;
    if (a->reset_u && a->R < 1) return AG_ERR_SHAPE;
    if (((uintptr_t)a->actions % 8) || ((uintptr_t)a->reset_u % 16) || ((uintptr_t)a->targets % 16)) return AG_ERR_ALIGN;
    if (row_stride < a->n) return AG_ERR_SHAPE;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, a->env_id0, a->engine, &G, &smem);
    if (st) return st;
    RolloutDev A;
    A.n = a->n; A.env_id0 = a->env_id0; A.row_stride = row_stride; A.K = a->K; A.R = a->R; A.seed = a->seed;
    A.actions = a->actions; A.reset_u = a->reset_u;
    A.j1 = a->j1; A.j2 = a->j2; A.reward = a->reward; A.flags = a->flags;
    A.step_ctr = a->step_ctr; A.reset_ctr = a->reset_ctr; A.ep_len = a->ep_len;
    A.rec_j1 = a->rec_j1; A.rec_j2 = a->rec_j2; A.rec_reward = a->rec_reward; A.rec_flags = a->rec_flags;
    A.stats = reinterpret_cast<unsigned long long *>(a->stats);
    A.diag = reinterpret_cast<unsigned long long *>(a->diag);
    A.targets = a->targets; A.max_occupied = g->max_occupied;
    // warp-wide 16-byte zero fill of the reward / flags record planes needs 16-byte aligned rows
    A.zfill = (a->rec_reward != nullptr && a->n % 32 == 0 && row_stride % 16 == 0 &&
               (uintptr_t)a->rec_reward % 16 == 0 && (uintptr_t)a->rec_flags % 16 == 0) ? 1 : 0;
    if (joints_only && a->n % 32 == 0) A.zfill = 1;      // nothing to fill: the uneventful step writes its joints only
    A.events = a->events; A.event_count = reinterpret_cast<unsigned long long *>(a->event_count);
    A.event_cap = a->event_capacity; A.event_step0 = a->event_step0;
    cudaStream_t s = (cudaStream_t)stream;
    // FAST engine: the obstacle-list broad phase when the caller vouches for small sparse staged grids
    // (ag_grid.max_occupied); a block whose grid turns out not to qualify falls back to EXACT per lane.
    if (a->engine == AG_ENGINE_FAST) {
        const bool list = G.stage && g->S <= 32 && g->max_occupied >= 0 && g->max_occupied <= AG_LIST_MAX;
        if (list && rollout_lut_applies(*p, G, A)) return launch_rollout_lut(*p, G, A, smem, s);
        if (list) return launch_rollout_e<AG_ENGINE_FAST, BP_LIST>(*p, G, A, smem, s);
        return launch_rollout_e<AG_ENGINE_FAST, BP_TRAVERSAL>(*p, G, A, smem, s);
    }
    if (a->engine == AG_ENGINE_EXACT) return launch_rollout_e<AG_ENGINE_EXACT, BP_ANY>(*p, G, A, smem, s);
    if (a->engine == AG_ENGINE_BRUTE) return launch_rollout_e<AG_ENGINE_BRUTE, BP_ANY>(*p, G, A, smem, s);
    return AG_ERR_MODE;
}

extern "C" {

int64_t ag_launch_count(void) { return g_launches.load(); }

ag_status ag_grid_pack(const uint8_t *occ, int32_t S, int32_t n_grids, uint32_t *bits, int64_t grid_stride_words,
                       void *stream) {
    if (!occ || !bits) return AG_ERR_NULL;
    const int wpr = (S + 31) / 32;
    if (S < 2 || n_grids < 1 || grid_stride_words < (int64_t)S * wpr) return AG_ERR_SHAPE;
    const int64_t total = (int64_t)S * wpr * n_grids;
    k_grid_pack<<<blocks_for(total), AG_BLOCK, 0, (cudaStream_t)stream>>>(occ, S, wpr, n_grids, bits, grid_stride_words);
    return launched();
}

ag_status ag_grid_pack_hier(const uint32_t *bits, int32_t S, int32_t n_grids, int64_t grid_stride_words, void *hier,
                            void *stream) {
    if (!bits || !hier) return AG_ERR_NULL;
    const int wpr = (S + 31) / 32;
    if (S < 2 || n_grids < 1 || grid_stride_words < (int64_t)S * wpr) return AG_ERR_SHAPE;
    if ((uintptr_t)hier % 16) return AG_ERR_ALIGN;
    const int T = (S + 7) / 8, cwpr = (T + 31) / 32;
    const int64_t hb = ag_grid_hier_bytes(S), tb = (((int64_t)T * T + 1) & ~(int64_t)1) * 8;
    cudaError_t e = cudaMemsetAsync(hier, 0, (size_t)hb * n_grids, (cudaStream_t)stream);
    if (e != cudaSuccess) return (ag_status)e;
    k_grid_pack_hier<<<blocks_for((int64_t)T * T * n_grids), AG_BLOCK, 0, (cudaStream_t)stream>>>(
        bits, S, wpr, n_grids, grid_stride_words, reinterpret_cast<unsigned char *>(hier), T, cwpr, tb,
        ((int64_t)T * cwpr + 3) & ~(int64_t)3, hb);
    return launched();
}

ag_status ag_segment_square(const double *seg, const double *sq, double section_eps, uint8_t *hit, double *abc,
                            double *corner_values, int64_t *axis_aligned, int64_t n, void *stream) {
    if (n < 0) return AG_ERR_SHAPE;
    if (n == 0) return AG_OK;
    if (!seg || !sq || !hit) return AG_ERR_NULL;
    if (((uintptr_t)seg % 32) || ((uintptr_t)sq % 32)) return AG_ERR_ALIGN;
    k_segment_square<<<blocks_for(n), AG_BLOCK, 0, (cudaStream_t)stream>>>(
        seg, sq, section_eps, hit, abc, corner_values, reinterpret_cast<unsigned long long *>(axis_aligned), n);
    return launched();
}

ag_status ag_forward_kinematics(const ag_params *p, const double *j1, const double *j2, double *out, int64_t n,
                                void *stream) {
    if (n < 0) return AG_ERR_SHAPE;
    if (n == 0) return AG_OK;
    if (!p || !j1 || !j2 || !out) return AG_ERR_NULL;
    if ((uintptr_t)out % 32) return AG_ERR_ALIGN;
    k_forward_kinematics<<<blocks_for(n), AG_BLOCK, 0, (cudaStream_t)stream>>>(*p, j1, j2, out, n);
    return launched();
}

ag_status ag_inverse_kinematics(const ag_params *p, const double *target, double *sol, uint8_t *valid, int32_t corrected,
                                int64_t n, void *stream) {
    if (n < 0) return AG_ERR_SHAPE;
    if (n == 0) return AG_OK;
    if (!p || !target || !sol || !valid) return AG_ERR_NULL;
    if (((uintptr_t)target % 16) || ((uintptr_t)sol % 32)) return AG_ERR_ALIGN;
    k_inverse_kinematics<<<blocks_for(n), AG_BLOCK, 0, (cudaStream_t)stream>>>(*p, target, sol, valid, corrected, n);
    return launched();
}

ag_status ag_move_to_joint_pose(double *j1, double *j2, const double *target, int32_t steps, int64_t n, void *stream) {
    if (n < 0 || steps < 1) return AG_ERR_SHAPE;
    if (n == 0) return AG_OK;
    if (!j1 || !j2 || !target) return AG_ERR_NULL;
    if ((uintptr_t)target % 16) return AG_ERR_ALIGN;
    k_move_to_joint_pose<<<blocks_for(n), AG_BLOCK, 0, (cudaStream_t)stream>>>(j1, j2, target, steps, n);
    return launched();
}

ag_status ag_collision_check(const ag_params *p, const ag_grid *g, const double *j1, const double *j2, uint8_t *hit,
                             int32_t *first_hit, int64_t n, int64_t env_id0, int32_t engine, void *stream) {
    if (n < 0) return AG_ERR_SHAPE;
    if (!p || !g) return AG_ERR_NULL;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, env_id0, engine, &G, &smem);
    if (st) return st;
    if (n == 0) return AG_OK;
    if (!j1 || !j2 || !hit) return AG_ERR_NULL;
    cudaStream_t s = (cudaStream_t)stream;
    AG_DISPATCH_ENGINE(engine, {
        if (first_hit) {
            auto k = k_collision<first_hit_engine(E), true>;
            if ((st = set_smem(k, smem))) return st;
            k<<<blocks_for(n), AG_BLOCK, smem, s>>>(*p, G, j1, j2, hit, first_hit, n, env_id0);
        } else {
            auto k = k_collision<E, false>;
            if ((st = set_smem(k, smem))) return st;
            k<<<blocks_for(n), AG_BLOCK, smem, s>>>(*p, G, j1, j2, hit, first_hit, n, env_id0);
        }
    });
    return launched();
}

ag_status ag_step(const ag_params *p, const ag_grid *g, double *j1, double *j2, const void *actions,
                  int32_t actions_f32, float *reward, uint8_t *flags, double *ee, double *dist, int32_t *first_hit,
                  int64_t *stats, const double *targets, int64_t n, int64_t env_id0, int32_t engine, void *stream) {
    if (n < 0) return AG_ERR_SHAPE;
    if (!p || !g) return AG_ERR_NULL;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, env_id0, engine, &G, &smem);
    if (st) return st;
    if (n == 0) return AG_OK;
    if (!j1 || !j2 || !actions || !reward || !flags) return AG_ERR_NULL;
    if (((uintptr_t)actions % (actions_f32 ? 8 : 16)) || ((uintptr_t)ee % 16) || ((uintptr_t)dist % 16) ||
        ((uintptr_t)targets % 16))
        return AG_ERR_ALIGN;
    StepDev D{j1, j2, actions, reward, flags, targets, reinterpret_cast<unsigned long long *>(stats), n, env_id0, ee, dist,
              first_hit};
    return launch_step(*p, G, D, engine, actions_f32 != 0, smem, (cudaStream_t)stream);
}

ag_status ag_reset(const ag_params *p, const ag_grid *g, double *j1, double *j2, float *reward, uint8_t *flags,
                   uint32_t *reset_ctr, const uint8_t *mask, const double *reset_u, int32_t R, uint64_t seed,
                   int32_t clear_flags, int64_t *stats, int64_t n, int64_t env_id0, int32_t engine, void *stream) {
    if (n < 0) return AG_ERR_SHAPE;
    if (!p || !g) return AG_ERR_NULL;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, env_id0, engine, &G, &smem);
    if (st) return st;
    if (n == 0) return AG_OK;
    if (!j1 || !j2 || !reset_ctr || (clear_flags && (!reward || !flags))) return AG_ERR_NULL;
    if (reset_u && R < 1) return AG_ERR_SHAPE;
    if ((uintptr_t)reset_u % 16) return AG_ERR_ALIGN;
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *ust = reinterpret_cast<unsigned long long *>(stats);
#define AG_RESET(HR) { auto k = k_reset<E, HR>; if ((st = set_smem(k, smem))) return st; \
        k<<<blocks_for(n), AG_BLOCK, smem, s>>>(*p, G, j1, j2, reward, flags, reset_ctr, mask, reset_u, R, seed, clear_flags, ust, n, env_id0); }
    AG_DISPATCH_ENGINE(engine, { if (reset_u) AG_RESET(true) else AG_RESET(false) });
#undef AG_RESET
    return launched();
}

ag_status ag_step_obs(const ag_params *p, const ag_grid *g, double *j1, double *j2, const void *actions, int32_t actions_f32,
                      float *reward, uint8_t *flags, uint32_t *reset_ctr, uint32_t *ep_len, const double *targets, double *obs,
                      float *reward_out, uint8_t *terminated, uint8_t *collision, double *final_obs, uint8_t *crop,
                      int32_t crop_size, int64_t *stats, uint64_t seed, int32_t auto_reset, int64_t n, int64_t env_id0,
                      int32_t engine, void *stream) {
    if (n < 0 || (crop && (crop_size < 1 || crop_size > 63 || crop_size % 2 == 0))) return AG_ERR_SHAPE;
    if (!p || !g) return AG_ERR_NULL;
    GridDev G;
    size_t smem;
    ag_status st = make_grid_dev(p, g, env_id0, engine, &G, &smem);
    if (st) return st;
    if (n == 0) return AG_OK;
    if (!j1 || !j2 || !actions || !reward || !flags || !reset_ctr || !ep_len || !obs || !reward_out || !terminated || !collision)
        return AG_ERR_NULL;
    if (((uintptr_t)actions % (actions_f32 ? 8 : 16)) || ((uintptr_t)obs % 16) || ((uintptr_t)final_obs % 16) || ((uintptr_t)targets % 16))
        return AG_ERR_ALIGN;
    StepDev D{j1, j2, actions, reward, flags, targets, reinterpret_cast<unsigned long long *>(stats), n, env_id0};
    D.reset_ctr = reset_ctr; D.ep_len = ep_len; D.obs = obs; D.final_obs = final_obs; D.reward_out = reward_out;
    D.terminated = terminated; D.collision = collision; D.crop = crop; D.crop_size = crop_size; D.auto_reset = auto_reset;
    D.seed = seed;
    return launch_step(*p, G, D, engine, actions_f32 != 0, smem, (cudaStream_t)stream);
}

ag_status ag_rollout(const ag_params *p, const ag_grid *g, const ag_rollout_args *a, void *stream) {
    if (!a) return AG_ERR_NULL;
    return ag_rollout_impl(p, g, a, a->n, stream);
}

}  // extern "C"
