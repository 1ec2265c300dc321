// ag_rollout.cuh -- pieces shared by the kernels of the library, the launch helpers every launcher uses, and the host
// functions one file calls in another: the grid prologue of every grid-taking entry point (make_grid_dev), the launch
// counter, the rollout with a row stride (ag_rollout_impl) and its dispatch to the persistent kernel.
//
// Each extern "C" entry point is defined next to its kernels:
//   ag_kernels.cu      K1..K6 and the general K4 (ag_collision_check, ag_step, ag_reset, ag_step_obs, ag_rollout, ...)
//   ag_rollout_lut.cu  the persistent scene_0-class K4, which ag_rollout dispatches to (launch_rollout_lut)
//   ag_motion.cu       ag_check_motion
//   ag_cspace.cu       ag_cspace_occupancy
//   ag_ccl.cu          ag_cspace_components
//   ag_cdist.cu        ag_cspace_distance, ag_cspace_descend
//   ag_cmap.cu         ag_cspace_map, ag_cspace_map_words (and the map cache its readers share, ag_cmap.cuh)
//   ag_host.cu         the host-only entry points and the pipelined host-buffer executor (ag_rollout_host)
#pragma once
#include <climits>

#include "ag_device.cuh"
#include "ag_fast.cuh"

void ag_note_launch();   // ag_kernels.cu: counts kernel launches (ag_launch_count)
// ag_kernels.cu: ag_rollout with an explicit action / record row stride (ag_host.cu runs it on chunks of a batch)
ag_status ag_rollout_impl(const ag_params *p, const ag_grid *g, const ag_rollout_args *a, int64_t row_stride,
                          void *stream);

namespace agd {

constexpr int AG_BLOCK = 256;
static_assert(AG_BLOCK <= AG_TILEQ_COLS, "the tile queue of arm_fast_hier has one column per thread");

// Opt a kernel in to `smem` bytes of dynamic shared memory.  Without the opt-in a launch may use 48 KB INCLUDING the
// kernel's static part (the 256-thread rollout kernels carry ~22 KB of it), so the attribute is set whenever static +
// dynamic exceeds 48 KB and the kernel's current limit.
template <typename Kernel>
ag_status set_smem(Kernel kernel, size_t smem) {
    if (smem == 0) return AG_OK;
    cudaFuncAttributes at;
    cudaError_t e = cudaFuncGetAttributes(&at, kernel);
    if (e != cudaSuccess) return (ag_status)e;
    if (smem + at.sharedSizeBytes > 48 * 1024 && (int)smem > at.maxDynamicSharedSizeBytes) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (ag_status)e;
    }
    return AG_OK;
}

// after a kernel launch: count it and return the launch's error
inline ag_status launched() {
    ag_note_launch();
    return (ag_status)cudaGetLastError();
}

// the grid of a persistent launch: blocks of `kernel` resident at once (SM count x blocks per SM at `block` threads and
// `smem` bytes of dynamic shared memory)
template <typename Kernel>
ag_status resident_blocks(Kernel kernel, int block, size_t smem, int *blocks) {
    int dev = 0, sms = 0, occ = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, block, smem);
    *blocks = sms * occ;
    return (ag_status)e;
}

// the grid of a launch with one thread per item
inline unsigned blocks_for(int64_t n) { return (unsigned)((n + AG_BLOCK - 1) / AG_BLOCK); }

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

// collision_check of one pose, out of line: the map forms of k_check_motion and k_cspace keep their loops short,
// with few live registers
template <int ENGINE, int BP = BP_ANY>
static __device__ __noinline__ bool pose_hit(const ag_params &P, const GridDev &G, const BlockCtx &B, const FastConst &C, double q1,
                                      double q2) {
    int fh = 0, axis = 0;
    return pose_collides<ENGINE, false, BP>(P, G, B, C, q1, q2, fh, axis);
}

// The in-kernel action of step counter `ctr` (scenario/scene_0.py:84-85): (rand() - 0.5) * action_scale per joint, from
// Philox stream 0.  BatchedScene.philox_actions draws the same on the host.
__device__ __forceinline__ void philox_action(const ag_params &P, uint64_t seed, uint64_t gid, uint32_t ctr, double &d1,
                                              double &d2) {
    double u0, u1;
    philox_uniform2(seed, gid, ctr, 0u, u0, u1);
    d1 = __dmul_rn(__dsub_rn(u0, 0.5), P.action_scale);
    d2 = __dmul_rn(__dsub_rn(u1, 0.5), P.action_scale);
}

// Reset candidate number rc (scenario/scene_0.py:180-181): rand()*pi*2.0 per joint, from Philox stream 1 or, with
// SCRIPTED, from the caller's uniforms reset_u_env[rc]; advances rc.
template <bool SCRIPTED>
__device__ __forceinline__ void reset_candidate(uint64_t seed, uint64_t gid, uint32_t &rc, const double *reset_u_env,
                                                double &j1, double &j2) {
    double u0, u1;
    if (SCRIPTED) {
        const double2 u = reinterpret_cast<const double2 *>(reset_u_env)[rc];
        u0 = u.x; u1 = u.y;
    } else {
        philox_uniform2(seed, gid, rc, 1u, u0, u1);
    }
    ++rc;
    j1 = __dmul_rn(__dmul_rn(u0, 3.141592653589793), 2.0);
    j2 = __dmul_rn(__dmul_rn(u1, 3.141592653589793), 2.0);
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
        reset_candidate<HAS_RESET_U>(seed, gid, rc, reset_u_env, j1, j2);
        ++tries;
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

__device__ __forceinline__ void cp_async8(uint32_t smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

}  // namespace agd

// make_grid_dev (ag_kernels.cu): the grid prologue of every entry point that takes an ag_grid.  Checks the grid
// (NULL pointers -> AG_ERR_NULL, inconsistent shape or stride -> AG_ERR_SHAPE; the FAST engine outside its error
// budget -> AG_ERR_MODE, other engine values are the caller's to check) and fills *out; *smem_bytes = the dynamic shared
// memory of a block that stages its grid (0: the grid is read from global memory).  Touches no device.
ag_status make_grid_dev(const ag_params *p, const ag_grid *g, int64_t env_id0, int engine, agd::GridDev *out,
                        size_t *smem_bytes);
// ag_rollout_lut.cu: the persistent kernel for scene_0-class grids (obstacle list, one grid, cartesian target)
bool rollout_lut_applies(const ag_params &P, const agd::GridDev &G, const agd::RolloutDev &A);
ag_status launch_rollout_lut(const ag_params &P, const agd::GridDev &G, const agd::RolloutDev &A, size_t smem, cudaStream_t s);
