// ag_rollout.cuh -- pieces shared by the rollout kernels (ag_kernels.cu: K1..K5 and the general K4;
// ag_rollout_lut.cu: the persistent scene_0-class K4).
#pragma once
#include <climits>

#include "ag_device.cuh"
#include "ag_fast.cuh"

namespace agd {

constexpr int AG_BLOCK = 256;
static_assert(AG_BLOCK <= AG_TILEQ_COLS, "the tile queue of arm_fast_hier has one column per thread");

struct RolloutDev {
    int64_t n, env_id0, row_stride;
    int32_t K, R;
    uint64_t seed;
    const float *actions;
    const double *reset_u;
    double *j1, *j2;
    float *reward;
    uint8_t *flags;
    uint32_t *step_ctr, *reset_ctr, *ep_len;
    float *rec_j1, *rec_j2, *rec_reward;
    uint8_t *rec_flags;
    unsigned long long *stats;
    unsigned long long *diag;
    int32_t zfill;            // 1: the reward / flags planes of this launch are zero-filled up front by each warp
    int32_t max_occupied;     // ag_grid.max_occupied (hint: upper bound on occupied cells)
    const double *targets;    // optional per-env cartesian targets [n][2], or nullptr
    uint32_t *events;         // optional event sink (ag_rollout_args.events), or nullptr
    unsigned long long *event_count;
    int64_t event_cap;
    int32_t event_step0;
};

// one eventful step -> the event sink (ag_rollout_args.events): (local env, step << 8 | flags, reward bits)
__device__ __forceinline__ void emit_event(const RolloutDev &A, int64_t e, int t, float rw, uint32_t fl) {
    if (A.events != nullptr && (fl != 0 || rw != 0.0f)) {
        const unsigned long long i = atomicAdd(A.event_count, 1ull);
        if (i < (unsigned long long)A.event_cap) {
            AG_CHECK_INDEX(t, A.K); AG_CHECK_INDEX(A.event_step0 + t, 1 << 24);
            A.events[3 * i] = (uint32_t)e;
            A.events[3 * i + 1] = ((uint32_t)(A.event_step0 + t) << 8) | (fl & 0xFFu);
            A.events[3 * i + 2] = __float_as_uint(rw);
        }
    }
}

// ------------------------------------------------------------------------- per-block context
// Every kernel that reads the grid starts the same way: stage the block's grid into shared memory
// (or point at global memory), and for the FAST engine build the obstacle list of small sparse grids.
struct BlockCtx {
    GridView V;
    const FastList *fl;   // nullptr: not applicable (grid not staged / engine != FAST)
};

template <int ENGINE>
__device__ __forceinline__ BlockCtx block_prologue(const GridDev &G, int64_t env_id0, int64_t n, unsigned char *smem,
                                                   FastList *s_fl) {
    const int64_t e0 = (int64_t)blockIdx.x * blockDim.x, e = e0 + threadIdx.x;
    BlockCtx B;
    B.fl = nullptr;
    if (G.stage) {
        B.V = stage_grid(G, env_id0 + e0, smem);
        if (ENGINE == AG_ENGINE_FAST) {
            build_fast_list(G, B.V, s_fl);
            B.fl = s_fl;
        }
    } else {
        const int64_t gi = grid_of_env(G, env_id0 + min(e, n - 1)), off = gi * G.stride_words;
        B.V.bits = G.bits + off;
        B.V.bits_t = G.bits_t ? G.bits_t + off : nullptr;
        B.V.min_x = G.min_x; B.V.min_y = G.min_y;
        view_hier(B.V, G, G.hier ? G.hier + gi * (int64_t)G.hier_bytes : nullptr);
    }
    return B;
}

// Block statistics: shared-memory atomics at (rare) events, one global atomic per slot per block.
// 64-bit shared atomics compile to compare-and-swap spin loops (ATOMS.CAST.SPIN), so every slot but the
// episode-length sum is accumulated as a native 32-bit add on the low word of its 64-bit cell: a block adds at
// most blockDim * K (K <= AG_MAX_K) per slot and launch, which cannot carry.  The return slot is signed.
constexpr int AG_MAX_K = 65536;
__device__ __forceinline__ void acc32(unsigned long long *s_acc, int slot, int v) {
    atomicAdd(reinterpret_cast<unsigned int *>(&s_acc[slot]), (unsigned int)v);
}
__device__ __forceinline__ void stats_flush(unsigned long long *s_acc, unsigned long long *gstats) {
    __syncthreads();
    if (threadIdx.x < AG_ST_COUNT && gstats != nullptr) {
        unsigned long long v = s_acc[threadIdx.x];
        if (threadIdx.x == AG_ST_RETURN_MILLI) v = (unsigned long long)(long long)(int)(unsigned int)v;   // sign-extend
        if (v != 0) atomicAdd(&gstats[threadIdx.x], v);
    }
}

// collision_check of one pose for K2/K3 (flag only unless WANT_FIRST)
template <int ENGINE, bool WANT_FIRST, int BP = BP_ANY>
__device__ __forceinline__ bool pose_collides(const ag_params &P, const GridDev &G, const BlockCtx &B,
                                              const FastConst &C, double j1, double j2, int &fh, int &axis) {
    if constexpr (ENGINE == AG_ENGINE_FAST && !WANT_FIRST) {
        const int d = fast_decide<BP>(P, G, B.V, B.fl, C, j1, j2, false);
        axis += d >> 2;
        return d & 1;
    } else {
        const Arm A = forward_kinematics(j1, j2, P.link_1, P.link_2);
        return arm_collides<ENGINE == AG_ENGINE_BRUTE ? AG_ENGINE_BRUTE : AG_ENGINE_EXACT, WANT_FIRST>(
            G, B.V, A, P.section_eps, fh, axis);
    }
}

// shared by K3 and K4: scenario/scene_0.py:174-181 with a bound.  `colliding` is the
// collision_check() of the current pose.
template <int ENGINE, bool HAS_RESET_U, int BP = BP_ANY>
__device__ __forceinline__ void resample_pose(const ag_params &P, const GridDev &G, const BlockCtx &B,
                                              const FastConst &C, bool colliding, double &j1, double &j2,
                                              uint32_t &rc, const double *reset_u_env, int32_t R, uint64_t seed,
                                              uint64_t gid, unsigned long long *s_acc) {
    int tries = 0;
    while (colliding) {
        if (tries >= P.max_reset_tries || (HAS_RESET_U && rc >= (uint32_t)R)) {
            acc32(s_acc, AG_ST_STUCK_RESETS, 1);
            break;
        }
        double u0, u1;
        if (HAS_RESET_U) {
            const double2 u = reinterpret_cast<const double2 *>(reset_u_env)[rc];
            u0 = u.x; u1 = u.y;
        } else {
            philox_uniform2(seed, gid, rc, 1u, u0, u1);
        }
        ++rc; ++tries;
        j1 = __dmul_rn(__dmul_rn(u0, 3.141592653589793), 2.0);    // scene_0.py:180  rand()*pi*2.0
        j2 = __dmul_rn(__dmul_rn(u1, 3.141592653589793), 2.0);    // :181
        int fh = 0, axis = 0;
        colliding = pose_collides<ENGINE, false, BP>(P, G, B, C, j1, j2, fh, axis);
        if (axis) acc32(s_acc, AG_ST_AXIS_ALIGNED, axis);
    }
}

// this thread's view of its grid: the block's shared-memory copy (layout of stage_grid) or global memory
__device__ __forceinline__ GridView thread_view(const GridDev &G, unsigned char *smem, int64_t gid) {
    GridView V;
    if (G.stage) {
        const int spad = (G.S + 1) & ~1;
        const uint32_t bit_bytes = (uint32_t)G.stride_words * 4u;
        V.bits = reinterpret_cast<const uint32_t *>(smem + 16);
        V.bits_t = G.bits_t ? V.bits + G.stride_words : nullptr;
        const uint32_t two_bytes = G.bits_t ? 2u * bit_bytes : bit_bytes;
        view_hier(V, G, G.hier ? smem + 16 + two_bytes : nullptr);
        V.min_x = reinterpret_cast<const double *>(smem + 16 + two_bytes + (G.hier ? (uint32_t)G.hier_bytes : 0u));
        V.min_y = V.min_x + spad;
    } else {
        const int64_t gi = grid_of_env(G, gid), off = gi * G.stride_words;
        V.bits = G.bits + off;
        V.bits_t = G.bits_t ? G.bits_t + off : nullptr;
        V.min_x = G.min_x; V.min_y = G.min_y;
        view_hier(V, G, G.hier ? G.hier + gi * (int64_t)G.hier_bytes : nullptr);
    }
    return V;
}

// one step record (experiment_0.py:23-25): joint_1, joint_2, step_reward, flags, post-step / pre-reset
template <bool RECORD>
__device__ __forceinline__ void store_record(const RolloutDev &A, int64_t o, double q1, double q2, float rw, uint32_t fl) {
    if (RECORD) {
        AG_CHECK_INDEX(o, (int64_t)(A.K - 1) * A.row_stride + A.n);
        __stcs(A.rec_j1 + o, (float)q1);
        __stcs(A.rec_j2 + o, (float)q2);
        if (A.rec_reward != nullptr) {                  // joints-only records: reward / flags go to the event sink
            __stcs(A.rec_reward + o, rw);
            A.rec_flags[o] = (uint8_t)fl;
        }
    }
}

// The record of an UNEVENTFUL step has reward 0 and flags 0.  When the launch qualifies (complete warps, 16-byte
// aligned rows) every warp zero-fills its slice of those two planes once, with warp-wide 16-byte stores (20 stores
// for 64 steps), and the hot loop stores the two joints only; eventful steps rewrite all four fields.
template <bool RECORD>
__device__ __forceinline__ void store_uneventful(const RolloutDev &A, int64_t o, double q1, double q2) {
    if (RECORD) {
        AG_CHECK_INDEX(o, (int64_t)(A.K - 1) * A.row_stride + A.n);
        __stcs(A.rec_j1 + o, (float)q1);
        __stcs(A.rec_j2 + o, (float)q2);
        if (!A.zfill && A.rec_reward != nullptr) {
            __stcs(A.rec_reward + o, 0.0f);
            A.rec_flags[o] = 0;
        }
    }
}

// warp-cooperative zero fill of rows [0, K) x this warp's 32 envs of the reward (128 B per row) and flags (32 B per
// row) planes.  warp_e0: first env of the warp (a multiple of 32).
__device__ __forceinline__ void zero_fill_warp(const RolloutDev &A, int64_t warp_e0) {
    if (A.rec_reward == nullptr) return;                // joints-only records
    const int lane = threadIdx.x & 31;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int t = lane >> 3; t < A.K; t += 4)            // 8 lanes x 16 B = one 128-byte row segment; 4 rows per store
        __stcs(reinterpret_cast<float4 *>(A.rec_reward + (int64_t)t * A.row_stride + warp_e0) + (lane & 7), z4);
    const uint4 zu = make_uint4(0u, 0u, 0u, 0u);
    for (int t = lane >> 1; t < A.K; t += 16)           // 2 lanes x 16 B = one 32-byte row segment; 16 rows per store
        reinterpret_cast<uint4 *>(A.rec_flags + (int64_t)t * A.row_stride + warp_e0)[lane & 1] = zu;
    __syncwarp();                                       // orders these stores before the owners' later rewrites
}


// ------------------------------------------------------------------------- configuration-space map (ag_rollout_lut.cu)
// 2^CB1 x 2^CB2 bins over (joint_1, joint_2) mod 2pi, one bit each.  The bin of a pose with |q| < 2^20 comes from the
// joint phases x = low word of fma(q, 2^32/2pi, PHASE_MAGIC): bit ((x1 >> (32 - CB1)) << CB2) | (x2 >> (32 - CB2)) of
// the map, word bit >> 5.  CLEAR: no pose of the bin collides or reaches the target (k_cspace_build); SET: evaluate.
#ifndef AG_CMAP_B1
#define AG_CMAP_B1 10
#endif
#ifndef AG_CMAP_B2
#define AG_CMAP_B2 8
#endif
constexpr int CB1 = AG_CMAP_B1, CB2 = AG_CMAP_B2;
static_assert(CB1 >= 6 && CB2 >= 6 && CB1 + CB2 <= 20, "the map must fit shared memory");
constexpr int CMAP_WORDS = 1 << (CB1 + CB2 - 5);
constexpr double PHASE_MAGIC = 6755399441055744.0;       // 1.5 * 2^52: the add rounds to an integer in the low word
constexpr double TWO_PI = 6.283185307179586476925;

}  // namespace agd

// ag_rollout_lut.cu: the map for one launch.  cspace_map_applies: the grid is one staged grid with an obstacle list
// (S <= 32, at most AG_LIST_MAX occupied cells by ag_grid.max_occupied), the only grids the map is built for.
// cspace_map_for_launch: the library's cached map of this grid and these parameters, after enqueuing on `s` the
// k_cspace_build launch that checks it against the grid's current content on the device (and rebuilds it if it
// differs); *map = nullptr when no cache entry can be had (inside a stream capture before the grid's first uncaptured
// launch, or an allocation failure) -- the caller then takes its general form, whose results are identical.
bool cspace_map_applies(const agd::GridDev &G, int32_t max_occupied);
ag_status cspace_map_for_launch(const ag_params &P, const agd::GridDev &G, cudaStream_t s, const uint32_t **map);

namespace agd {

__device__ __forceinline__ void cp_async8(uint32_t smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }


}  // namespace agd
