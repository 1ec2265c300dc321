// ag_rollout_lut.cu -- K4 for scene_0-class grids (obstacle list, one grid, cartesian target): the rollout loop
// experiment/experiment_0.py:20-34 fused over K steps, persistent warps.  DESIGN.md "K4, scene_0 class".
//
// The general kernel (ag_kernels.cu, k_rollout) is instruction-issue-bound at ~236 warp-instructions per warp-step;
// ~145 of them are the float32 filter of an uneventful step (99.5 % of all env-steps).  This kernel has two forms of a
// much cheaper test for "this step is certainly uneventful"; both use the joint phase
//
//   x = low word of fma(q, 2^32/2pi, 1.5*2^52)            one DFMA per joint: the turn fraction as a 32-bit integer
//
// CMAP form (the default; scene-wide target): one bit of a configuration-space map in shared memory, indexed by the top
//   bits of (x1, x2), says whether ANY pose of that bin can touch an obstacle or the target box -- no forward kinematics
//   in the hot loop at all (k_cspace_build below explains how the map is made conservative, and how it is cached and
//   validated against the current grid on the device at every launch).
// table-arm form (per-env targets, or no map available): the float32 arm comes from two shared-memory tables,
//   entry  = lut[x >> (32-B)]                            (c, s) * length at the bin centre, 8 bytes
//   d      = (x mod 2^(32-B)) * 2pi/2^32 - pi/2^B        angle from the bin centre, one LOP3 + one FFMA
//   point  = (1 - d*d/2) * (c, s) + d * (-s, c)          second-order Taylor step: FMUL + FFMA + FMUL2 + 2 FFMA
//   With 2048 bins for link 1 and 512 for link 2, emulated op for op in numpy over 1.2e7 angles up to +-2^20 rad, the
//   elbow is within 8.9e-8 m and the end effector within 2.1e-7 m of the float64 values: inside the error budget
//   AG_DELTA_P = 3e-7 m the float32 filter of ag_fast.cuh was derived for.  Link 1 depends on joint_1 only: its test is
//   one hazard bit per bin (hazard_interval), link 2 is a box test against the squares, the target a box pre-test.
//
// A lane that clears the test is certainly uneventful; every other lane ("slow", ~0.5 % of env-steps) goes through the
// float32 narrow phase, the float64 filter and the reference arithmetic exactly as in the general kernel (level 1 in the
// loop, level 2 = settle_step).  Results are therefore identical to the general kernel's and the reference's;
// tests/test_gpu_parity.py runs all forms.
//
// Structure: a persistent grid (one 512-thread block per SM); every warp draws 32-env tiles from a global counter.
// Per tile: state -> registers, the next valid reset pose is drawn up front by all 32 lanes together (draw_valid_pose;
// consumed on collision), then K steps of
//   action (cp.async ring, RING - 1 rows ahead) -> 2 DADD -> test -> record (2 F2F + 2 STG) -> vote.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "ag_rollout.cuh"

using namespace agd;

void ag_note_launch();

namespace {

#ifndef AG_LUT_B1
#define AG_LUT_B1 11
#endif
#ifndef AG_LUT_B2
#define AG_LUT_B2 9
#endif
#ifndef AG_LUT_BLOCKS_PER_SM
#define AG_LUT_BLOCKS_PER_SM 1
#endif

// configuration-space map (CMAP form of the kernel): CB1, CB2, CMAP_WORDS in ag_rollout.cuh
constexpr int CMAP_HDR_WORDS = 64;                       // 256-byte header in front of the map words
constexpr int CMAP_SLOTS = 16;
struct CmapHeader {
    unsigned long long key;                              // hash of everything the map depends on; 0 = never built
    unsigned int done[CMAP_SLOTS];                       // blocks finished, one counter per in-flight build
};
static_assert(sizeof(CmapHeader) <= CMAP_HDR_WORDS * 4, "header");

constexpr int B1 = AG_LUT_B1, B2 = AG_LUT_B2;            // bins: 2^B1 for link 1 (also the resolution of its hazard bit), 2^B2 for link 2
constexpr int N1 = 1 << B1, N2 = 1 << B2;
static_assert(B1 >= 9 && B2 >= 9 && B1 <= 11 && B2 <= 11, "sub-bin phase must fit 23 bits; tables must fit static shared memory");
// One 512-thread block per SM: the same 16 warps as two blocks of 256, but one copy of the map, of the obstacle list and
// of the block's bookkeeping per SM (+3 %; 640 threads at 96 registers spill and lose 6 %).
#ifndef AG_LUT_BLOCK
#define AG_LUT_BLOCK 512
#endif
constexpr int LB = AG_LUT_BLOCK, LW = LB / 32;
// Action prefetch ring: every lane streams its own actions global -> shared with cp.async (LDGSTS), RING - 1 steps
// ahead of their use; slot (t mod RING) of the warp's ring holds row t.  (Register prefetch does not work here: ptxas
// gives all in-flight LDGs of the loop ONE scoreboard slot, so a consumer waits for every outstanding load and the
// effective distance is a single step: profiles/r2b.)
// 8 rows for the map form; the table-arm form keeps 20 KB of tables in static shared memory next to the rings (static
// shared memory is capped at 48 KB) and stays at 4.  [Moving the rings into the dynamic segment measured 5-9 % slower.]
#ifndef AG_LUT_RING
#define AG_LUT_RING 4
#endif
#ifndef AG_CMAP_RING
#define AG_CMAP_RING 8
#endif
static_assert((AG_LUT_RING & (AG_LUT_RING - 1)) == 0 && AG_LUT_RING >= 4, "ring slots: a power of two");
#ifndef AG_CMAP_LAZY_DRAW
#define AG_CMAP_LAZY_DRAW 1
#endif
static_assert((AG_CMAP_RING & (AG_CMAP_RING - 1)) == 0 && AG_CMAP_RING >= 4, "ring slots: a power of two");

constexpr float RAD_PER_UNIT = (float)(TWO_PI / 4294967296.0);   // one phase unit (2^-32 turn) in radians
// d = fma(2^23 + frac, RAD_PER_UNIT, C0): removes the 2^23 of the integer -> float trick and half a bin
__host__ __device__ constexpr float lut_c0(int bits) { return (float)(-(8388608.0 * (double)RAD_PER_UNIT + TWO_PI / (double)(2 << bits))); }
constexpr float C0_1 = lut_c0(B1), C0_2 = lut_c0(B2);

struct LutConst {
    double phase_scale;     // 2^32 / 2pi
    float thr_c;            // reach_eps + AG_DELTA_P + 2e-7: reach pre-test threshold (reach_fast's margin)
    int64_t n_tiles;
    uint32_t ss_off;        // byte offset of SlowShared in dynamic shared memory (after the staged grid)
    uint32_t slot;          // this launch's pair of tile / done counters (g_tile_sched)
    uint32_t cmap_off;      // CMAP: byte offset of the map's shared-memory copy in the dynamic segment
    const uint32_t *cmap;   // CMAP: the map words in global memory (k_cspace_build)
};

// Dynamic tile scheduling: warps draw 32-env tiles from a device-global counter, so no warp idles while tiles remain
// (a static split leaves 13 % of all warp-time parked at the end: profiles/r2a).  Each launch uses the next of
// AG_TILE_SLOTS counter pairs (host round-robin); the last block to finish zeroes its pair again.  Launches in flight
// at the same time on one device must therefore number fewer than AG_TILE_SLOTS.
constexpr int AG_TILE_SLOTS = 256;
__device__ unsigned int g_tile_sched[2 * AG_TILE_SLOTS];    // [2*slot] next tile, [2*slot+1] blocks done

// per-thread state that only the slow path touches (one slot per thread: no sharing, no conflicts)
struct SlowShared {
    double cq1[LB], cq2[LB];   // the pre-drawn reset pose
    float rw[LB];              // sticky Scene.step_reward
    uint32_t fl[LB];           // sticky flags
    uint32_t rc[LB];           // reset draw counter
    uint32_t crc[LB];          // reset draw counter after the pre-drawn pose
    uint32_t cinfo[LB];        // PoseDraw::info of the pre-drawn pose, 0 = consumed
    int el_off[LB];            // episode length after step t = el_off + t + 1
    // the hot loop's registers, parked here around the slow section: that section makes out-of-line calls, and any
    // value live in a register across a call is spilled where it is DEFINED, i.e. inside the hot loop
    double q1[LB], q2[LB];
    float thr[LB], tx[LB], ty[LB];
    int t[LB];
    int cr[LB];                // level 1's verdicts for level 2: 0 = no event, else 16 | c | r << 2
    uint32_t sc0[LB];          // action draw counter at the start of the launch (Philox actions)
    // Episode statistics of the current tile, one private cell per lane (no atomics: 64-bit shared atomics are
    // compare-and-swap loops, five of them per episode end cost 3 % of the kernel -- profiles/r2); the warp folds
    // them into its own row of s_wacc when the tile ends.
    unsigned long long len_sum[LB];
    uint32_t n_ep[LB], n_col[LB], n_suc[LB], n_cold[LB], n_exact[LB];
    int ret[LB];
};
enum { WA_EPISODES = 0, WA_COLLISIONS, WA_SUCCESSES, WA_LEN_SUM, WA_RETURN, WA_ENV_STEPS, WA_COLD, WA_EXACT, WA_EXITS, WA_COUNT };

__device__ __forceinline__ void add64(unsigned long long *s_acc, int slot, long long v) {
    atomicAdd(&s_acc[slot], (unsigned long long)v);
}

// scenario/scene_0.py:174-181 with a bound, entered with a colliding pose: draw candidates until one is free.
// Nothing is counted here (the pose may never be used); the caller applies `info` when it consumes the pose.
struct PoseDraw {
    double j1, j2;
    uint32_t rc;
    uint32_t info;   // bit0 valid, bit1 at least one candidate drawn (j1, j2 meaningful), bit2 gave up; bits 8..: axis-aligned evaluations
};
enum { PD_VALID = 1, PD_DREW = 2, PD_STUCK = 4 };

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// cmap_a: shared-window address of the configuration-space map, or 0.  A candidate whose bin is CLEAR is certainly
// collision-free (the map's guarantee): accepted without any arithmetic on the arm.
AG_COLD PoseDraw draw_valid_pose(const ag_params &P, const GridDev &G, const FastConst &C,
                                                 const unsigned char *smem_grid, const FastList *fl, uint32_t rc,
                                                 const double *reset_u_env, int32_t R, uint64_t seed, uint64_t gid,
                                                 uint32_t cmap_a = 0u) {
    const GridView V = thread_view(G, const_cast<unsigned char *>(smem_grid), (int64_t)gid);
    PoseDraw o;
    o.j1 = 0.0; o.j2 = 0.0; o.info = PD_VALID;
    int tries = 0, axis = 0;
    bool colliding = true;
    while (colliding) {
        if (tries >= P.max_reset_tries || (reset_u_env != nullptr && rc >= (uint32_t)R)) { o.info |= PD_STUCK; break; }
        double u0, u1;
        if (reset_u_env != nullptr) {
            const double2 u = reinterpret_cast<const double2 *>(reset_u_env)[rc];
            u0 = u.x; u1 = u.y;
        } else {
            philox_uniform2(seed, gid, rc, 1u, u0, u1);
        }
        ++rc; ++tries;
        o.j1 = __dmul_rn(__dmul_rn(u0, 3.141592653589793), 2.0);    // scene_0.py:180  rand()*pi*2.0
        o.j2 = __dmul_rn(__dmul_rn(u1, 3.141592653589793), 2.0);    // :181
        if (cmap_a != 0u && o.j1 < 1048576.0 && o.j2 < 1048576.0) {        // candidates are in [0, 2 pi) unless scripted
            const uint32_t x1 = (uint32_t)__double2loint(fma(o.j1, 4294967296.0 / TWO_PI, PHASE_MAGIC));
            const uint32_t x2 = (uint32_t)__double2loint(fma(o.j2, 4294967296.0 / TWO_PI, PHASE_MAGIC));
            const uint32_t bit = ((x1 >> (32 - CB1)) << CB2) | (x2 >> (32 - CB2));
            if (((lds_u32(cmap_a + ((bit >> 3) & ~3u)) >> (bit & 31u)) & 1u) == 0u) { colliding = false; continue; }
        }
        const int d = fast_decide<BP_LIST>(P, G, V, fl, C, o.j1, o.j2, false);
        axis += d >> 2;
        colliding = (d & 1) != 0;
    }
    if (tries) o.info |= PD_DREW;
    o.info |= (uint32_t)axis << 8;
    o.rc = rc;
    return o;
}

// Level 2 of the slow path, for one lane with an event: (1) float64 filter / reference arithmetic for what the
// float32 narrow phase could not settle, (2) reward / flags (scene_0.py:95-100), record rewrite, (3) episode end
// (experiment_0.py:30-34): statistics + Scene.reset() from the pre-drawn pose.
// Works on the lane's parked state (SlowShared: q1, q2, t, cr in; q1, q2, thr out).
template <bool RECORD>
__device__ __forceinline__ void settle_step(const ag_params &P, const GridDev &G, const FastConst &C, const RolloutDev &A,
                                            SlowShared &ss, const FastList *fl, unsigned long long *s_acc,
                                            const unsigned char *smem_grid, float thr_clean, int64_t e, uint32_t cmap_a) {
    const int x = threadIdx.x;
    const int t = ss.t[x] - 1;                                                   // the step being settled (ss.t: where the loop resumes)
    const int c = ss.cr[x] & 3, r = (ss.cr[x] >> 2) & 3;                         // the float32 verdicts: 0 / 1 certain, 2 undecided
    double q1 = ss.q1[x], q2 = ss.q2[x];
    int d = (c & 1) | ((r & 1) << 1);
    bool cold = false;
    if ((c | r) & 2) {                                                           // undecided: float64
        double txd = P.target_x, tyd = P.target_y;
        if (A.targets != nullptr) {
            const double2 tg = reinterpret_cast<const double2 *>(A.targets)[e];
            txd = tg.x; tyd = tg.y;
        }
        const GridView V = thread_view(G, const_cast<unsigned char *>(smem_grid), A.env_id0 + e);
        d = cold_exact_decide_at(P, G, V, fl, q1, q2, c, r, txd, tyd);
        cold = true;
        ss.n_exact[x] += 1;
    }
    float rw = ss.rw[x];
    uint32_t f = ss.fl[x];
    if (d & 1) { rw = (float)P.reward_collision; f |= AG_FLAG_COLLISION; }       // scene_0.py:95-97
    if (d & 2) { rw = (float)P.reward_reach; f |= AG_FLAG_DONE; }                // :98-100
    if (d >> 2) add64(s_acc, AG_ST_AXIS_ALIGNED, d >> 2);
    if (RECORD && A.rec_reward != nullptr && (f != 0 || rw != 0.0f)) {           // experiment_0.py:23-25 (joints already stored)
        const int64_t o = (int64_t)t * A.row_stride + e;
        __stcs(A.rec_reward + o, rw);
        A.rec_flags[o] = (uint8_t)f;
    }
    emit_event(A, e, t, rw, f);
    if (f) {                                                                     // experiment_0.py:30-34
        cold = true;
        ss.n_ep[x] += 1;
        if (f & AG_FLAG_COLLISION) ss.n_col[x] += 1;
        if (f & AG_FLAG_DONE) ss.n_suc[x] += 1;
        ss.len_sum[x] += (unsigned long long)((long long)ss.el_off[x] + t + 1);
        ss.ret[x] += __float2int_rn(rw * 1e-3f);
        if (d & 1) {   // Scene.reset(): the pose is unchanged since the step, so collision_check() == (d & 1)
            uint32_t info = ss.cinfo[x];
            if (info & PD_VALID) {
                if (info & PD_DREW) { q1 = ss.cq1[x]; q2 = ss.cq2[x]; }
                ss.rc[x] = ss.crc[x];
                ss.cinfo[x] = 0;
            } else {                                                             // second collision of this tile: draw now
                const PoseDraw pd = draw_valid_pose(P, G, C, smem_grid, fl, ss.rc[x],
                                                    A.reset_u ? A.reset_u + e * A.R * 2 : nullptr, A.R, A.seed,
                                                    (uint64_t)(A.env_id0 + e), cmap_a);
                if (pd.info & PD_DREW) { q1 = pd.j1; q2 = pd.j2; }
                ss.rc[x] = pd.rc;
                info = pd.info;
            }
            if (info & PD_STUCK) add64(s_acc, AG_ST_STUCK_RESETS, 1);
            if (info >> 8) add64(s_acc, AG_ST_AXIS_ALIGNED, info >> 8);
        }
        rw = 0.0f; f = 0; ss.el_off[x] = -(t + 1);                               // scene_0.py:111-113
    }
    if (cold) ss.n_cold[x] += 1;
    ss.rw[x] = rw; ss.fl[x] = f;
    ss.q1[x] = q1; ss.q2[x] = q2;
    ss.thr[x] = (f != 0 || rw != 0.0f) ? __int_as_float(0x7f800000) : thr_clean;
}

__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}

// point = (1 - d*d/2) * (c, s) + d * (-s, c): the table entry's vector turned by the small angle d
__device__ __forceinline__ float2 taylor_turn(float2 t, float d) {
    const float u = fmaf(d * d, -0.5f, 1.0f);
    const float2 ut = mul2(t, splat2(u));
    return make_float2(fmaf(-d, t.y, ut.x), fmaf(d, t.x, ut.y));
}

// The directions in which link 1 (origin -> length l1) comes within `mg` of the closed square sq = (min_x, min_y, max_x,
// max_y): the angular extent of (inflated square) n (disc of radius l1) seen from the origin.  That set is convex and,
// unless the origin lies inside the inflated square, does not contain the origin, so its extent is spanned by its
// vertices: corners inside the disc and circle / edge crossings (a ray from the centre is never tangent to the circle).
// half < 0: never; half >= pi: always.
__device__ void hazard_interval(double X0, double Y0, double X1, double Y1, double l1, float &mid, float &half);
__device__ void hazard_interval(float4 sq, double l1, double mg, float &mid, float &half) {
    hazard_interval((double)sq.x - mg, (double)sq.y - mg, (double)sq.z + mg, (double)sq.w + mg, l1, mid, half);
}
// the same for an (already inflated) box X0..X1 x Y0..Y1
__device__ void hazard_interval(double X0, double Y0, double X1, double Y1, double l1, float &mid, float &half) {
    if (X0 <= 0.0 && X1 >= 0.0 && Y0 <= 0.0 && Y1 >= 0.0) { mid = 0.0f; half = 4.0f; return; }
    const double r2 = l1 * l1;
    const double ref = atan2(0.5 * (Y0 + Y1), 0.5 * (X0 + X1));
    double lo = 1.0e9, hi = -1.0e9;
    auto take = [&](double px, double py) {
        double a = atan2(py, px) - ref;
        a -= TWO_PI * rint(a / TWO_PI);
        lo = fmin(lo, a); hi = fmax(hi, a);
    };
    const double XS[2] = {X0, X1}, YS[2] = {Y0, Y1};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j)
            if (XS[i] * XS[i] + YS[j] * YS[j] <= r2) take(XS[i], YS[j]);
    for (int i = 0; i < 2; ++i) {
        if (fabs(XS[i]) <= l1) {
            const double y = sqrt(r2 - XS[i] * XS[i]);
            if (y >= Y0 && y <= Y1) take(XS[i], y);
            if (-y >= Y0 && -y <= Y1) take(XS[i], -y);
        }
        if (fabs(YS[i]) <= l1) {
            const double xx = sqrt(r2 - YS[i] * YS[i]);
            if (xx >= X0 && xx <= X1) take(xx, YS[i]);
            if (-xx >= X0 && -xx <= X1) take(-xx, YS[i]);
        }
    }
    if (hi < lo) { mid = 0.0f; half = -1.0f; return; }
    mid = (float)(ref + 0.5 * (lo + hi));
    half = (float)(0.5 * (hi - lo));
}

// Fill a table of n bins with (c, s) * len at the bin centres (b + 1/2) * 2pi/n, eight symmetric entries per
// float64 sincospi.  hz != nullptr: bit 0 of .x is link 1's hazard bit (hz: [m][2] = (mid, half) intervals), else 0.
__device__ void fill_table(float2 *lut, int n, double len, const float *hz, int m, bool all_hazard) {
    const float hw = (float)(TWO_PI / (double)(2 * n)) + 2.0e-6f;                // half a bin + phase / float rounding
    for (int i = threadIdx.x; i < n / 8; i += blockDim.x) {
        double sd, cd;
        sincospi((2.0 * i + 1.0) / (double)n, &sd, &cd);                         // angle (i + 1/2) * 2pi/n in (0, pi/4)
        const float c = (float)(len * cd), s = (float)(len * sd);
        const int q4 = n / 4;
        const int bins[8] = {i, q4 - 1 - i, q4 + i, 2 * q4 - 1 - i, 2 * q4 + i, 3 * q4 - 1 - i, 3 * q4 + i, n - 1 - i};
        const float xs[8] = {c, s, -s, -c, -c, -s, s, c};
        const float ys[8] = {s, c, c, s, -s, -c, -c, -s};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int b = bins[j];
            uint32_t bit = 0;
            if (hz != nullptr) {
                bit = all_hazard ? 1u : 0u;
                const float th = ((float)b + 0.5f) * (float)(TWO_PI / (double)n);
                for (int k = 0; k < m; ++k) {
                    float dlt = th - hz[2 * k];
                    dlt -= (float)TWO_PI * rintf(dlt * (float)(1.0 / TWO_PI));
                    if (fabsf(dlt) <= hz[2 * k + 1] + hw) bit = 1u;
                }
            }
            const float vx = hz != nullptr ? __uint_as_float((__float_as_uint(xs[j]) & ~1u) | bit) : xs[j];
            lut[b] = make_float2(vx, ys[j]);
        }
    }
}

// ------------------------------------------------------------------------- configuration-space map (CMAP)
// One bit per bin of (joint_1, joint_2) mod 2pi: CLEAR = for every pose of the bin both links stay farther than CMAP_MG
// from every occupied square and the end effector stays outside the target box (scene_0.py:129-130) by more than
// CMAP_MG, i.e. the step is certainly uneventful and the hot loop needs no forward kinematics at all -- two DFMA for
// the phases, one shared-memory word, one bit test.  SET = "look closer": the lane takes the slow path, which decides
// exactly as before.  So the map only has to be CONSERVATIVE; it is built from lower bounds of distances:
//   * over a bin, joint_1 in [a1-d1, a1+d1] and joint_2 in [a2-d2, a2+d2], the elbow stays within the sagitta
//     l1(1-cos d1) of the chord Ea..Eb and link 2's direction vector within l2(1-cos d2) of the triangle 0, Ua, Ub, so
//     link 2 sweeps a subset of the convex polygon hull({Ea,Eb} + {0,Ua,Ub}) inflated by the two sagittas;
//   * the distance from that polygon to a square is bounded from below by the largest separation along a finite set
//     of unit axes (every axis gives a valid lower bound; the set -- box normals, the link normals at the bin's centre
//     and edges, the chord normal, and the directions from the square's corners to the centre pose's elbow and end
//     effector -- makes the bound tight for edge/vertex and vertex/vertex contacts);
//   * link 1 depends on joint_1 only and uses the exact angular intervals of hazard_interval().
// 2.0e-6 m covers the rounding of the phase (< 1e-9 rad), of this float64 construction, and the reference's own
// rounding noise (< 1e-12 m): the same margin the float32 broad phase uses.
// The map depends on the grid, the link lengths, the target and its tolerance.  It lives in a library-owned device
// buffer that is reused between launches: every launch re-derives a 64-bit key from the CURRENT grid words and
// parameters on the device (thread 0 of each block, ~100 words) and rebuilds the map only when the stored key differs.
constexpr double CMAP_MG = 2.0e-6;
constexpr int CMAP_BUILD_BLOCKS = 128;
constexpr uint32_t CMAP_VERSION = 1;

struct V2 { double x, y; };

__device__ __forceinline__ unsigned long long mix64(unsigned long long h, unsigned long long v) {
    h ^= v;
    h *= 0x100000001B3ull;                                                       // FNV-1a over 64-bit words
    return h ^ (h >> 29);
}

// separation of the point set P and the box (centre c, half extents hx, hy) along the unit axis n (negative: overlap)
template <int NP>
__device__ __forceinline__ double axis_gap(V2 n, const V2 (&P)[NP], V2 c, double hx, double hy) {
    double lo = 1.0e300, hi = -1.0e300;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        const double d = n.x * P[i].x + n.y * P[i].y;
        lo = fmin(lo, d); hi = fmax(hi, d);
    }
    const double cc = n.x * c.x + n.y * c.y, r = fabs(n.x) * hx + fabs(n.y) * hy;
    return fmax(lo - (cc + r), (cc - r) - hi);
}

__global__ void __launch_bounds__(256)
k_cspace_build(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G, uint32_t *buf, uint32_t slot) {
    __shared__ unsigned long long s_key;
    __shared__ int s_skip, s_m;
    __shared__ double s_sq[AG_LIST_MAX][4];
    __shared__ float s_hz[2 * AG_LIST_MAX];
    CmapHeader *H = reinterpret_cast<CmapHeader *>(buf);
    if (threadIdx.x == 0) {
        unsigned long long h = 0xCBF29CE484222325ull;
        h = mix64(h, ((unsigned long long)CMAP_VERSION << 48) | ((unsigned long long)CB1 << 40) | ((unsigned long long)CB2 << 32) | (unsigned)G.S);
        const double par[6] = {P.link_1, P.link_2, P.target_x, P.target_y, P.reach_eps, G.side};
        for (int i = 0; i < 6; ++i) h = mix64(h, (unsigned long long)__double_as_longlong(par[i]));
        int m = 0;
        for (int r = 0; r < G.S; ++r) {
            h = mix64(h, (unsigned long long)__double_as_longlong(G.min_y[r]));
            h = mix64(h, (unsigned long long)__double_as_longlong(G.min_x[r]));
            for (int w = 0; w < G.wpr; ++w) {
                uint32_t word = G.bits[r * G.wpr + w];
                h = mix64(h, word);
                while (word) {
                    const int c = (w << 5) + __ffs(word) - 1;
                    word &= word - 1;
                    if (m < AG_LIST_MAX && c < G.S) {
                        const double mnx = G.min_x[c], mny = G.min_y[r];
                        s_sq[m][0] = mnx; s_sq[m][1] = mny;
                        s_sq[m][2] = __dadd_rn(mnx, G.side); s_sq[m][3] = __dadd_rn(mny, G.side);   // occupancy_grid.py:66-67
                    }
                    ++m;
                }
            }
        }
        h |= 1ull;                                                               // 0 means "never built"
        s_key = h;
        s_m = m > AG_LIST_MAX ? -1 : m;                                          // no obstacle list: every bin is slow
        s_skip = (*reinterpret_cast<volatile unsigned long long *>(&H->key) == h) ? 1 : 0;
    }
    __syncthreads();
    if (!s_skip) {
        const int m = s_m;
        if ((int)threadIdx.x < m)
            hazard_interval(s_sq[threadIdx.x][0] - CMAP_MG, s_sq[threadIdx.x][1] - CMAP_MG, s_sq[threadIdx.x][2] + CMAP_MG,
                            s_sq[threadIdx.x][3] + CMAP_MG, P.link_1, s_hz[2 * threadIdx.x], s_hz[2 * threadIdx.x + 1]);
        __syncthreads();
        constexpr int N1c = 1 << CB1, N2c = 1 << CB2;
        const double l1 = P.link_1, l2 = P.link_2;
        double sd, cd;
        sincospi(1.0 / (double)N1c, &sd, &cd);
        const double sag1 = l1 * (1.0 - cd);
        sincospi(1.0 / (double)N2c, &sd, &cd);
        const double sag2 = l2 * (1.0 - cd);
        const double infl = sag1 + sag2 + CMAP_MG;
        const float hw1 = (float)(TWO_PI / (double)(2 * N1c)) + 2.0e-6f;          // half a bin of joint_1 + rounding
        for (int bin = blockIdx.x * 256 + threadIdx.x; bin < N1c * N2c; bin += gridDim.x * 256) {   // a warp = 32 bins of joint_2
            const int b1 = bin >> CB2, b2 = bin & (N2c - 1);
            bool haz = m < 0;
            // ---- link 1: exact angular intervals
            const float th1 = ((float)b1 + 0.5f) * (float)(TWO_PI / (double)N1c);
            for (int k = 0; k < m; ++k) {
                float dlt = th1 - s_hz[2 * k];
                dlt -= (float)TWO_PI * rintf(dlt * (float)(1.0 / TWO_PI));
                if (fabsf(dlt) <= s_hz[2 * k + 1] + hw1) haz = true;
            }
            // ---- link 2: the swept polygon against every square
            V2 Ea, Eb, Ec, Ua, Ub, Uc;
            sincospi(2.0 * (double)b1 / (double)N1c, &Ea.y, &Ea.x);
            sincospi(2.0 * (double)(b1 + 1) / (double)N1c, &Eb.y, &Eb.x);
            sincospi((2.0 * (double)b1 + 1.0) / (double)N1c, &Ec.y, &Ec.x);
            sincospi(2.0 * (double)b2 / (double)N2c, &Ua.y, &Ua.x);
            sincospi(2.0 * (double)(b2 + 1) / (double)N2c, &Ub.y, &Ub.x);
            sincospi((2.0 * (double)b2 + 1.0) / (double)N2c, &Uc.y, &Uc.x);
            const V2 n1c = {Ec.x, Ec.y};                                          // normal of the elbow chord = link 1's direction
            const V2 n2a = {-Ua.y, Ua.x}, n2b = {-Ub.y, Ub.x}, n2c = {-Uc.y, Uc.x};   // link 2's normals at the bin's edges / centre
            const V2 ea = {l1 * Ea.x, l1 * Ea.y}, eb = {l1 * Eb.x, l1 * Eb.y}, ec = {l1 * Ec.x, l1 * Ec.y};
            const V2 ua = {l2 * Ua.x, l2 * Ua.y}, ub = {l2 * Ub.x, l2 * Ub.y};
            const V2 gc = {ec.x + l2 * Uc.x, ec.y + l2 * Uc.y};
            const V2 poly[6] = {ea, eb, {ea.x + ua.x, ea.y + ua.y}, {ea.x + ub.x, ea.y + ub.y},
                                {eb.x + ua.x, eb.y + ua.y}, {eb.x + ub.x, eb.y + ub.y}};
            for (int k = 0; k < m && !haz; ++k) {
                const V2 c = {0.5 * (s_sq[k][0] + s_sq[k][2]), 0.5 * (s_sq[k][1] + s_sq[k][3])};
                const double hx = 0.5 * (s_sq[k][2] - s_sq[k][0]), hy = 0.5 * (s_sq[k][3] - s_sq[k][1]);
                double gap = axis_gap(V2{1.0, 0.0}, poly, c, hx, hy);
                gap = fmax(gap, axis_gap(V2{0.0, 1.0}, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n2c, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n2a, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n2b, poly, c, hx, hy));
                gap = fmax(gap, axis_gap(n1c, poly, c, hx, hy));
#pragma unroll 1
                for (int j = 0; j < 8; ++j) {                                     // corner -> centre pose's end effector / elbow
                    const double qx = (j & 1) ? s_sq[k][2] : s_sq[k][0], qy = (j & 2) ? s_sq[k][3] : s_sq[k][1];
                    const V2 from = (j & 4) ? ec : gc;
                    const double vx = from.x - qx, vy = from.y - qy, nv = sqrt(vx * vx + vy * vy);
                    if (nv > 1.0e-9) gap = fmax(gap, axis_gap(V2{vx / nv, vy / nv}, poly, c, hx, hy) * (1.0 - 1.0e-12));
                }
                if (!(gap > infl)) haz = true;
            }
            // ---- the target box (scene_0.py:129-130) against the box of the swept end effector
            {
                const double gx0 = fmin(fmin(poly[2].x, poly[3].x), fmin(poly[4].x, poly[5].x)) - infl;
                const double gx1 = fmax(fmax(poly[2].x, poly[3].x), fmax(poly[4].x, poly[5].x)) + infl;
                const double gy0 = fmin(fmin(poly[2].y, poly[3].y), fmin(poly[4].y, poly[5].y)) - infl;
                const double gy1 = fmax(fmax(poly[2].y, poly[3].y), fmax(poly[4].y, poly[5].y)) + infl;
                const double e = fabs(P.reach_eps);
                if (!(gx0 > P.target_x + e || gx1 < P.target_x - e || gy0 > P.target_y + e || gy1 < P.target_y - e)) haz = true;
            }
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, haz);
            if ((threadIdx.x & 31) == 0) buf[CMAP_HDR_WORDS + (bin >> 5)] = word;
        }
    }
    // the last block of this launch publishes the key (blocks that skipped count too: the map they saw was complete)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(&H->done[slot], 1u) == gridDim.x - 1) {
            H->done[slot] = 0;
            *reinterpret_cast<volatile unsigned long long *>(&H->key) = s_key;
            __threadfence();
        }
    }
}


// The float32 arm from the tables (see the header of this file): elbow, half of link 2, link 1's hazard bit.
struct TableArm { float2 ev, hv; uint32_t hazard; };
__device__ __forceinline__ TableArm table_arm(double q1, double q2, double phase_scale, uint32_t lut1_a, uint32_t lut2_a) {
    const uint32_t x1 = (uint32_t)__double2loint(fma(q1, phase_scale, PHASE_MAGIC));
    const uint32_t x2 = (uint32_t)__double2loint(fma(q2, phase_scale, PHASE_MAGIC));
    const float2 t1 = lds_f2(lut1_a + ((x1 >> (29 - B1)) & (uint32_t)((N1 - 1) << 3)));
    const float2 t2 = lds_f2(lut2_a + ((x2 >> (29 - B2)) & (uint32_t)((N2 - 1) << 3)));
    const float dA = fmaf(__uint_as_float((x1 & ((1u << (32 - B1)) - 1u)) | 0x4B000000u), RAD_PER_UNIT, C0_1);
    const float dB = fmaf(__uint_as_float((x2 & ((1u << (32 - B2)) - 1u)) | 0x4B000000u), RAD_PER_UNIT, C0_2);
    TableArm a;
    a.ev = taylor_turn(t1, dA);
    a.hv = taylor_turn(t2, dB);
    a.hazard = __float_as_uint(t1.x) & 1u;
    return a;
}

// CMAP = true: the hot loop consults the configuration-space map instead of computing the table arm (scene-wide target only)
template <bool HAS_ACT, bool RECORD, bool M3, bool CMAP>
__global__ void __launch_bounds__(LB, AG_LUT_BLOCKS_PER_SM)
k_rollout_lut(const __grid_constant__ ag_params P, const __grid_constant__ GridDev G, const __grid_constant__ FastConst C,
              const __grid_constant__ RolloutDev A, const __grid_constant__ LutConst L) {
    extern __shared__ __align__(16) unsigned char smem_grid[];  // the staged grid (layout of stage_grid), then SlowShared
    __shared__ __align__(16) float2 s_lut1[CMAP ? 1 : N1], s_lut2[CMAP ? 1 : N2];
    constexpr int RING = CMAP ? AG_CMAP_RING : AG_LUT_RING;     // the table-arm form keeps its tables in static shared memory
    __shared__ __align__(16) float2 s_ring[LW][RING][32];   // action rows t .. t+RING-1 of each warp's tile (cp.async)
    __shared__ FastList s_fl;
    __shared__ float s_hz[2 * AG_LIST_MAX];
    __shared__ unsigned long long s_acc[AG_ST_COUNT + AG_DIAG_COUNT];
    __shared__ long long s_wacc[LW][WA_COUNT];                  // per-warp totals over its tiles (lane 0 owns the row)
    __shared__ unsigned int s_done;
    __shared__ int64_t s_tile[LW];                              // each warp's current tile
    __shared__ int s_exits[LW];                                 // diagnostics: exits of the hot loop, per warp
    SlowShared &ss = *reinterpret_cast<SlowShared *>(smem_grid + L.ss_off);     // dynamic: static shared memory is capped at 48 KB
    if (threadIdx.x < AG_ST_COUNT + AG_DIAG_COUNT) s_acc[threadIdx.x] = 0;
    if (threadIdx.x < LW * WA_COUNT) (&s_wacc[0][0])[threadIdx.x] = 0;
    if (threadIdx.x == 0) s_done = 0;
    if (threadIdx.x < LW) s_exits[threadIdx.x] = 0;
    {
        const GridView V = stage_grid(G, A.env_id0, smem_grid);                  // one grid: block-uniform
        build_fast_list(G, V, &s_fl);
    }
    if constexpr (CMAP) {                                                        // ---- the map: global -> shared
        const uint4 *src = reinterpret_cast<const uint4 *>(L.cmap);
        uint4 *dst = reinterpret_cast<uint4 *>(smem_grid + L.cmap_off);
        for (int i = threadIdx.x; i < CMAP_WORDS / 4; i += LB) dst[i] = src[i];
    } else {                                                                     // ---- the two tables
        const int m = s_fl.m;
        if ((int)threadIdx.x < m) hazard_interval(s_fl.sq[threadIdx.x], P.link_1, 2.0e-6, s_hz[2 * threadIdx.x], s_hz[2 * threadIdx.x + 1]);
        __syncthreads();
        fill_table(s_lut1, N1, P.link_1, s_hz, m < 0 ? 0 : m, m < 0 || (M3 && m > 3));   // no list / more squares than promised: all slow
        fill_table(s_lut2, N2, 0.5 * P.link_2, nullptr, 0, false);
    }
    __syncthreads();

    const int x = threadIdx.x, lane = x & 31;
    const float INF = __int_as_float(0x7f800000);
    const float2 zero2 = make_float2(0.f, 0.f);

    for (;;) {
        // ================================================================ draw a tile, global state -> SlowShared
        {
            int64_t tile = 0;
            if (lane == 0) tile = (int64_t)atomicAdd(&g_tile_sched[2 * L.slot], 1u);
            tile = __shfl_sync(0xFFFFFFFFu, tile, 0);
            if (tile >= L.n_tiles) break;
            if (lane == 0) s_tile[x >> 5] = tile;
            const int64_t e = tile * 32 + lane;
            const bool active = RECORD ? true : (e < A.n);                       // RECORD launches have complete tiles (zfill)
            const int64_t ec = active ? e : A.n - 1;                             // inactive lanes shadow the last env, store nothing
            ss.q1[x] = A.j1[ec]; ss.q2[x] = A.j2[ec];
            const float rw0 = A.reward[ec];
            const uint32_t fl0 = A.flags[ec];
            ss.rw[x] = rw0; ss.fl[x] = fl0; ss.el_off[x] = (int)A.ep_len[ec];
            const uint32_t rc0 = A.reset_ctr[ec];
            ss.rc[x] = rc0;
            const uint32_t sc0 = A.step_ctr[ec];
            ss.sc0[x] = sc0;
            if (active) A.step_ctr[e] = sc0 + (uint32_t)A.K;
            float tx = C.tx, ty = C.ty;
            if (A.targets != nullptr) {
                const double2 tg = reinterpret_cast<const double2 *>(A.targets)[ec];
                tx = (float)tg.x; ty = (float)tg.y;
            }
            ss.tx[x] = tx; ss.ty[x] = ty;
            // a lane whose sticky state is not clean (flags / reward left by earlier step() calls) is slow until an
            // episode end clears it: an infinite threshold makes its reach pre-test fire
            ss.thr[x] = (fl0 != 0 || rw0 != 0.0f) ? INF : L.thr_c;
            ss.t[x] = 0;
            ss.len_sum[x] = 0; ss.n_ep[x] = 0; ss.n_col[x] = 0; ss.n_suc[x] = 0; ss.n_cold[x] = 0; ss.n_exact[x] = 0; ss.ret[x] = 0;
            if (HAS_ACT) {                                                       // rows 0 .. RING-2 in flight
                const uint32_t ring_lane = smem_u32(&s_ring[x >> 5][0][lane]);
                const float2 *ap = reinterpret_cast<const float2 *>(A.actions) + e;
#pragma unroll
                for (int i = 0; i < RING - 1; ++i) {
                    if (i < A.K && active) cp_async8(ring_lane + (uint32_t)(i << 8), ap);
                    cp_async_commit();
                    ap += A.row_stride;
                }
            }
            if (RECORD && A.zfill) zero_fill_warp(A, tile * 32);
            if constexpr (CMAP && AG_CMAP_LAZY_DRAW) {
                // Map form: no pose is drawn ahead.  6 % of the lanes collide during a tile; the lane that does draws
                // then (settle_step), and 86 % of its candidates are accepted by one look at the map.
                ss.cinfo[x] = 0;
            } else {
                // the next valid reset pose, drawn by all lanes together
                const PoseDraw pd = draw_valid_pose(P, G, C, smem_grid, &s_fl, rc0,
                                                    A.reset_u ? A.reset_u + ec * A.R * 2 : nullptr, A.R, A.seed,
                                                    (uint64_t)(A.env_id0 + ec));
                ss.cq1[x] = pd.j1; ss.cq2[x] = pd.j2; ss.crc[x] = pd.rc; ss.cinfo[x] = pd.info;
            }
            __syncwarp();
        }
        for (;;) {   // ---- resume loop: one pass per entry into the hot loop (fresh tile, or after a level-2 call)
        // ================================================================ set-up
        // Everything the hot loop keeps in registers is (re)derived HERE from kernel parameters and shared memory -- for a
        // fresh tile and again after every level-2 call.  A value live in a register across a call is spilled where it
        // is defined and reloaded where it is used, i.e. inside the hot loop; this way nothing is live across a call.
        // The asm statements keep the compiler from merging these values with copies computed before the call.
        int64_t tile = s_tile[x >> 5];
        asm volatile("" : "+l"(tile));
        const int K = A.K;
        const int64_t e = tile * 32 + lane;
        const bool active = RECORD ? true : (e < A.n);
        const uint64_t gid = (uint64_t)(A.env_id0 + (active ? e : A.n - 1));
        const uint32_t sc0 = HAS_ACT ? 0u : ss.sc0[x];
        // Table addresses: ptxas otherwise re-derives a shared-memory symbol's address (cluster rank << 24 | offset: S2UR
        // + 4 uniform ops + 2 moves) at every use.  Row strides in bytes: otherwise re-read from the constant bank and
        // re-shifted at every step.
        uint32_t lut1_a, lut2_a, ring_lane;
        asm volatile("mov.u32 %0, %1;" : "=r"(lut1_a) : "r"(smem_u32(s_lut1)));
        asm volatile("mov.u32 %0, %1;" : "=r"(lut2_a) : "r"(smem_u32(s_lut2)));
        asm volatile("mov.u32 %0, %1;" : "=r"(ring_lane) : "r"(smem_u32(&s_ring[x >> 5][0][lane])));
        uint32_t cmap_a;
        asm volatile("mov.u32 %0, %1;" : "=r"(cmap_a) : "r"(smem_u32(smem_grid + L.cmap_off)));
        int64_t sa = A.row_stride * (int64_t)sizeof(float2), sr = A.row_stride * (int64_t)sizeof(float);
        asm volatile("" : "+l"(sa));
        asm volatile("" : "+l"(sr));
        float hm = s_fl.hm;                                                      // side/2 + AG_M_BROAD (INF without a list)
        asm volatile("" : "+f"(hm));
        // square centres of the 3-obstacle map (occupancy_grid.py:45-47) live in registers
        float2 o0, o1, o2;
        if (M3) {
            const float2 far = make_float2(1.0e9f, 1.0e9f);
            o0 = s_fl.m > 0 ? s_fl.ctr[0] : far; o1 = s_fl.m > 1 ? s_fl.ctr[1] : far; o2 = s_fl.m > 2 ? s_fl.ctr[2] : far;
        }
        double q1 = ss.q1[x], q2 = ss.q2[x];
        float thr = ss.thr[x];
        const float tx = ss.tx[x], ty = ss.ty[x];
        int t = ss.t[x];
        char *p1 = reinterpret_cast<char *>(A.rec_j1 + e + (int64_t)t * A.row_stride);          // record row t
        char *p2 = reinterpret_cast<char *>(A.rec_j2 + e + (int64_t)t * A.row_stride);
        const char *pa = reinterpret_cast<const char *>(reinterpret_cast<const float2 *>(A.actions) + e + (int64_t)(t + RING - 1) * A.row_stride);   // next row to fetch

        // what the last step leaves for level 1: the table arm, the box measures of link 2 (3-square form), the reach
        // measure, link 1's hazard bit, angles in range
        float l_ex = 0.f, l_ey = 0.f, l_gx = 0.f, l_gy = 0.f, l_s0 = 0.f, l_s1 = 0.f, l_s2 = 0.f, l_worst = 0.f;
        bool l_haz = false, l_inr = false;
        // one step up to the vote: true = this lane is slow
        auto step = [&](float2 a, int t) -> bool {
            double d1, d2;
            if (HAS_ACT) {
                d1 = (double)a.x; d2 = (double)a.y;
            } else {
                double u0, u1;
                philox_uniform2(A.seed, gid, sc0 + (uint32_t)t, 0u, u0, u1);
                d1 = __dmul_rn(__dsub_rn(u0, 0.5), P.action_scale);              // scene_0.py:84
                d2 = __dmul_rn(__dsub_rn(u1, 0.5), P.action_scale);              // :85
            }
            q1 = __dadd_rn(q1, d1); q2 = __dadd_rn(q2, d2);                      // two_joint_robot.py:71-72
            const bool inr = (fabs(q1) < 1048576.0) && (fabs(q2) < 1048576.0);   // NaN-safe: NaN is slow
            if constexpr (CMAP) {
                const uint32_t x1 = (uint32_t)__double2loint(fma(q1, L.phase_scale, PHASE_MAGIC));
                const uint32_t x2 = (uint32_t)__double2loint(fma(q2, L.phase_scale, PHASE_MAGIC));
                const uint32_t bit = ((x1 >> (32 - CB1)) << CB2) | (x2 >> (32 - CB2));
                const uint32_t w = lds_u32(cmap_a + ((bit >> 3) & ~3u));
                l_inr = inr;
                if (RECORD) {
                    __stcs(reinterpret_cast<float *>(p1), (float)q1);
                    __stcs(reinterpret_cast<float *>(p2), (float)q2);
                    p1 += sr; p2 += sr;
                }
                // a set bit, sticky state (thr == INF), or an angle outside the phase's range (also NaN)
                return (((w >> (bit & 31u)) & 1u) != 0) || !(thr < INF) || !inr;
            }
            const TableArm ta = table_arm(q1, q2, L.phase_scale, lut1_a, lut2_a);
            const float2 ev = ta.ev, hv = ta.hv;
            const float c2x = ev.x + hv.x, c2y = ev.y + hv.y;                    // centre of link 2's box; half extents |hv|
            const float gx = fmaf(2.0f, hv.x, ev.x), gy = fmaf(2.0f, hv.y, ev.y);
            const float hx = fabsf(hv.x), hy = fabsf(hv.y);
            float sep;
            if (M3) {
                const float s0 = fmaxf(fabsf(c2x - o0.x) - hx, fabsf(c2y - o0.y) - hy);
                const float s1 = fmaxf(fabsf(c2x - o1.x) - hx, fabsf(c2y - o1.y) - hy);
                const float s2 = fmaxf(fabsf(c2x - o2.x) - hx, fabsf(c2y - o2.y) - hy);
                sep = fminf(fminf(s0, s1), s2);
                l_s0 = s0; l_s1 = s1; l_s2 = s2;
            } else {
                sep = 1.0e30f;
                const int m = s_fl.m;
#pragma unroll 1
                for (int k = 0; k < m; ++k) {
                    const float2 o = s_fl.ctr[k];
                    sep = fminf(sep, fmaxf(fabsf(c2x - o.x) - hx, fabsf(c2y - o.y) - hy));
                }
            }
            const float worst = fmaxf(fabsf(tx - gx), fabsf(ty - gy));
            l_ex = ev.x; l_ey = ev.y; l_gx = gx; l_gy = gy; l_worst = worst; l_haz = ta.hazard != 0; l_inr = inr;
            if (RECORD) {                                                        // RECORD launches have complete tiles
                __stcs(reinterpret_cast<float *>(p1), (float)q1);                // and zero-filled reward / flags planes
                __stcs(reinterpret_cast<float *>(p2), (float)q2);
                p1 += sr; p2 += sr;
            }
            // NaN-safe: an unordered comparison is slow.  Inactive lanes (ragged last tile, STATS mode only) are
            // masked on the rare path.
            return (ta.hazard != 0) || !(sep >= hm) || !(worst >= thr) || !inr;
        };
        // Ring slot of step t: ring_lane + (t mod RING) * 256.  Invariant at the top of the loop: rows t .. t+RING-2 are
        // in flight or landed in their slots, pa points at row t+RING-1.
        auto issue_row = [&](int row) {                                          // row `row` -> its slot, if it exists
            if (HAS_ACT) {
                if (row < K && active) cp_async8(ring_lane + (((uint32_t)row & (RING - 1)) << 8), pa);
                cp_async_commit();
                pa += sa;
            }
        };
        auto fetch_row = [&](int t) -> float2 {                                  // this step's action, after its copy has landed
            if (!HAS_ACT) return zero2;
            cp_async_wait<RING - 1>();
            return lds_f2(ring_lane + (((uint32_t)t & (RING - 1)) << 8));
        };
        bool need_level2 = false, event = false;
        int cr = 0;
        for (;;) {
            bool slow = false;
            // ---- hot loop: uneventful steps only; the warp leaves it when ANY lane is slow
#pragma unroll 1
            for (; t < K; ++t) {
                issue_row(t + RING - 1);
                slow = step(fetch_row(t), t);
                if (__any_sync(0xFFFFFFFFu, slow)) break;
            }
            if (t >= K) break;
            {

            // Step t is recorded as uneventful.  Level 1 (no calls: the loop state stays in registers): the float32
            // narrow phase of the slow lanes on the step's table arm; usually it clears them all.
            cr = 0;
            event = false;
            if (slow && active) {
                int c = 2, r = 2;
                if (CMAP) {                                                      // the hot loop had no arm: float32 FK now
                    bool ok;
                    const ArmF a = fast_forward_kinematics(q1, q2, C, ok);
                    if (ok) {
                        c = s_fl.m < 0 ? 2 : arm_fast_list(&s_fl, a, C, true);
                        r = reach_fast_at(C, a, tx, ty);
                    }
                } else if (l_inr) {
                    ArmF a;
                    a.ex = l_ex; a.ey = l_ey; a.gx = l_gx; a.gy = l_gy;
                    if (s_fl.m < 0) {
                        c = 2;
                    } else if (M3 && !l_haz) {                                   // the step's own measures name the pairs
                        const uint32_t cand = (l_s0 < hm ? 2u : 0u) | (l_s1 < hm ? 8u : 0u) | (l_s2 < hm ? 32u : 0u);
                        c = narrow_candidates(&s_fl, a, C, cand);
                    } else {
                        c = arm_fast_list(&s_fl, a, C, l_haz);
                    }
                    const float mr = AG_DELTA_P + 2.0e-7f;                       // reach_fast() on the step's measure
                    r = l_worst > C.reach_eps + mr ? 0 : (l_worst < C.reach_eps - mr ? 1 : 2);
                }
                cr = c | (r << 2);
                event = (cr != 0) || !(thr < INF);                               // a hit, target reached, undecided, or sticky state
            }
            if (A.diag != nullptr && lane == 0) s_exits[x >> 5] += 1;
            // Reconverge HERE.  The vote below only makes the fragments of a diverged warp meet for one instruction
            // (BRA.DIV + WARPSYNC.COLLECTIVE); without a real barrier the slow lanes and the others went back into
            // the hot loop as separate fragments and every instruction of it was issued twice (profiles/r2d: 21 of 32
            // threads per hot-loop instruction).
            __syncwarp();
            if (__any_sync(0xFFFFFFFFu, event)) { need_level2 = true; break; }
            ++t;
        }
        }
        if (!need_level2) {                                                      // the tile is finished: registers -> global
            if (HAS_ACT) cp_async_wait<0>();
            if (active) {
                A.j1[e] = q1; A.j2[e] = q2; A.reward[e] = ss.rw[x]; A.flags[e] = (uint8_t)ss.fl[x];
                A.ep_len[e] = (uint32_t)(ss.el_off[x] + K);
                A.reset_ctr[e] = ss.rc[x];
            }
            const int n_act = __popc(__ballot_sync(0xFFFFFFFFu, active));
            // fold the tile's per-lane counters into the warp's row
            const uint32_t ne = __reduce_add_sync(0xFFFFFFFFu, ss.n_ep[x]);
            const uint32_t ncold = __reduce_add_sync(0xFFFFFFFFu, ss.n_cold[x]);
            long long *wa = s_wacc[x >> 5];
            if (ne != 0 || ncold != 0) {                                         // warp-uniform
                const uint32_t nc = __reduce_add_sync(0xFFFFFFFFu, ss.n_col[x]), ns = __reduce_add_sync(0xFFFFFFFFu, ss.n_suc[x]);
                const uint32_t nx = __reduce_add_sync(0xFFFFFFFFu, ss.n_exact[x]);
                const int rt = __reduce_add_sync(0xFFFFFFFFu, ss.ret[x]);
                unsigned long long ls = ss.len_sum[x];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) ls += __shfl_xor_sync(0xFFFFFFFFu, ls, o);
                if (lane == 0) {
                    wa[WA_EPISODES] += ne; wa[WA_COLLISIONS] += nc; wa[WA_SUCCESSES] += ns; wa[WA_LEN_SUM] += (long long)ls;
                    wa[WA_RETURN] += rt; wa[WA_COLD] += ncold; wa[WA_EXACT] += nx;
                }
            }
            if (lane == 0) {
                wa[WA_ENV_STEPS] += (long long)n_act * K;
                wa[WA_EXITS] += s_exits[x >> 5]; s_exits[x >> 5] = 0;
            }
            break;
        }
        // ================================================================ level 2 (out-of-line calls), then resume
        ss.q1[x] = q1; ss.q2[x] = q2; ss.thr[x] = thr; ss.t[x] = t + 1; ss.cr[x] = event ? (cr | 16) : 0;
        if (event)
            settle_step<RECORD>(P, G, C, A, ss, &s_fl, s_acc, smem_grid, L.thr_c, s_tile[x >> 5] * 32 + (threadIdx.x & 31),
                                CMAP ? smem_u32(smem_grid + L.cmap_off) : 0u);
        __syncwarp();
        }   // resume loop
    }
    // ---- no block barrier at the end (a warp that runs out of tiles just leaves): the last warp of the block
    // flushes the block's counters, the last block of the grid re-arms the tile counters
    __threadfence_block();
    unsigned int prev = 0;
    if (lane == 0) prev = atomicAdd(&s_done, 1u);
    prev = __shfl_sync(0xFFFFFFFFu, prev, 0);
    if (prev == LW - 1) {
        __threadfence_block();
        // slot of s_acc -> column of s_wacc that also feeds it (-1: none)
        const int wa_of_stat[AG_ST_COUNT] = {WA_EPISODES, WA_COLLISIONS, WA_SUCCESSES, WA_ENV_STEPS, WA_LEN_SUM, WA_RETURN, -1, -1};
        const int wa_of_diag[AG_DIAG_COUNT] = {WA_EXACT, WA_COLD, WA_EXITS};
        if (lane < AG_ST_COUNT && A.stats != nullptr) {
            unsigned long long v = *reinterpret_cast<volatile unsigned long long *>(&s_acc[lane]);
            const int col = wa_of_stat[lane];
            if (col >= 0)
                for (int w = 0; w < LW; ++w) v += (unsigned long long)*reinterpret_cast<volatile long long *>(&s_wacc[w][col]);
            if (v != 0) atomicAdd(&A.stats[lane], v);
        }
        if (A.diag != nullptr && lane < AG_DIAG_COUNT) {
            unsigned long long v = *reinterpret_cast<volatile unsigned long long *>(&s_acc[AG_ST_COUNT + lane]);
            for (int w = 0; w < LW; ++w) v += (unsigned long long)*reinterpret_cast<volatile long long *>(&s_wacc[w][wa_of_diag[lane]]);
            if (v != 0) atomicAdd(&A.diag[lane], v);
        }
        unsigned int *const sched = g_tile_sched + 2 * L.slot;
        if (lane == 0 && atomicAdd(&sched[1], 1u) == gridDim.x - 1) {            // every block has drawn its last tile
            sched[0] = 0; sched[1] = 0;
            __threadfence();
        }
    }
}

int sm_slots(const void *kernel, size_t smem) {
    int dev = 0, sms = 0, occ = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, LB, smem) != cudaSuccess) return 0;
    return sms * occ;
}

template <bool HA, bool REC, bool M3, bool CM>
ag_status launch_t(const ag_params &P, const GridDev &G, const RolloutDev &A, const LutConst &L, size_t smem, cudaStream_t s) {
    auto k = k_rollout_lut<HA, REC, M3, CM>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (ag_status)e;
    const int slots = sm_slots(reinterpret_cast<const void *>(k), smem);
    if (slots <= 0) return (ag_status)cudaGetLastError();
    const int64_t want = (L.n_tiles + LW - 1) / LW;
    const unsigned blocks = (unsigned)(want < slots ? want : slots);
    k<<<blocks, LB, smem, s>>>(P, G, make_fast_const(P, G), A, L);
    ag_note_launch();
    return (ag_status)cudaGetLastError();
}

}  // namespace

// The persistent kernel serves the FAST engine on one staged small sparse grid (obstacle list), cartesian target.
bool rollout_lut_applies(const ag_params &P, const GridDev &G, const RolloutDev &A) {
    static const bool legacy = std::getenv("AG_ROLLOUT_LEGACY") != nullptr;
    const bool rec = A.rec_j1 != nullptr;   // RECORD: complete tiles and zero-filled reward / flags planes only
    // the table arm's error (2.2e-7 m per metre of link 1, 2.8e-7 per metre of link 2, 5e-8 of rounding) must stay
    // inside the float32 filter's budget AG_DELTA_P
    const bool budget = 2.2e-7 * P.link_1 + 2.8e-7 * P.link_2 + 5.0e-8 <= (double)AG_DELTA_P;
    return !legacy && cspace_map_applies(G, A.max_occupied) && !P.choose_j_tar && (!rec || A.zfill) && budget;
}

// ---- the library-owned buffers of the configuration-space maps: up to 32 entries (33 KB each) per process, found by (device, grid
// pointers, parameters); the CONTENT is validated on the device by every launch (k_cspace_build), so a grid that was
// rewritten in place, or a new grid at a recycled address, just rebuilds the entry.
namespace {
struct CmapEntry {
    int dev = -1;
    const void *bits = nullptr, *min_x = nullptr;
    double par[6] = {0, 0, 0, 0, 0, 0};
    int S = 0;
    uint32_t *buf = nullptr;
    unsigned long long last_use = 0;
};
constexpr int CMAP_ENTRIES = 32;
std::mutex g_cmap_mutex;
CmapEntry g_cmap[CMAP_ENTRIES];
unsigned long long g_cmap_clock = 0;

// the entry's device buffer (header + map), or nullptr when the map form cannot be used for this launch
uint32_t *cmap_buffer(const ag_params &P, const GridDev &G, cudaStream_t s) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cap) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    const bool capturing = cap != cudaStreamCaptureStatusNone;
    const double par[6] = {P.link_1, P.link_2, P.target_x, P.target_y, P.reach_eps, G.side};
    std::lock_guard<std::mutex> lock(g_cmap_mutex);
    CmapEntry *hit = nullptr, *lru = &g_cmap[0];
    for (CmapEntry &e : g_cmap) {
        if (e.buf != nullptr && e.dev == dev && e.bits == G.bits && e.min_x == G.min_x && e.S == G.S &&
            std::memcmp(e.par, par, sizeof(par)) == 0) { hit = &e; break; }
        if (e.last_use < lru->last_use) lru = &e;
    }
    if (hit == nullptr) {
        if (capturing) return nullptr;                        // no allocation / synchronisation inside a stream capture
        if (lru->buf != nullptr) {
            // the buffer changes hands: launches that still read the old map (any stream of its device) must be done
            int cur = dev;
            if (lru->dev != cur && cudaSetDevice(lru->dev) != cudaSuccess) return nullptr;
            cudaDeviceSynchronize();
            if (lru->dev != cur) { cudaFree(lru->buf); lru->buf = nullptr; cudaSetDevice(cur); }
        }
        if (lru->buf == nullptr && cudaMalloc(&lru->buf, (size_t)(CMAP_HDR_WORDS + CMAP_WORDS) * 4) != cudaSuccess) {
            cudaGetLastError();
            lru->buf = nullptr; lru->dev = -1;
            return nullptr;
        }
        if (cudaMemsetAsync(lru->buf, 0, CMAP_HDR_WORDS * 4, s) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        lru->dev = dev; lru->bits = G.bits; lru->min_x = G.min_x; lru->S = G.S;
        std::memcpy(lru->par, par, sizeof(par));
        hit = lru;
    }
    hit->last_use = ++g_cmap_clock;
    return hit->buf;
}
}  // namespace

bool cspace_map_applies(const GridDev &G, int32_t max_occupied) {
    return G.stage && G.n_grids == 1 && G.S <= 32 && max_occupied >= 0 && max_occupied <= AG_LIST_MAX;
}

ag_status cspace_map_for_launch(const ag_params &P, const GridDev &G, cudaStream_t s, const uint32_t **map) {
    *map = nullptr;
    uint32_t *buf = cmap_buffer(P, G, s);
    if (buf == nullptr) return AG_OK;
    static std::atomic<unsigned> next_build{0};
    k_cspace_build<<<CMAP_BUILD_BLOCKS, 256, 0, s>>>(P, G, buf, next_build.fetch_add(1, std::memory_order_relaxed) % CMAP_SLOTS);
    ag_note_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (ag_status)e;
    *map = buf + CMAP_HDR_WORDS;
    return AG_OK;
}

int64_t cspace_map_words(int32_t *b1, int32_t *b2) {
    if (b1) *b1 = CB1;
    if (b2) *b2 = CB2;
    return CMAP_WORDS;
}

// the map alone, into a caller's buffer (ag_cspace_map): built in a scratch buffer with the header in front
ag_status launch_cspace_map(const ag_params &P, const GridDev &G, uint32_t *map, cudaStream_t s) {
    uint32_t *buf = nullptr;
    cudaError_t e = cudaMallocAsync(&buf, (size_t)(CMAP_HDR_WORDS + CMAP_WORDS) * 4, s);
    if (e != cudaSuccess) return (ag_status)e;
    e = cudaMemsetAsync(buf, 0, CMAP_HDR_WORDS * 4, s);
    if (e == cudaSuccess) {
        k_cspace_build<<<CMAP_BUILD_BLOCKS, 256, 0, s>>>(P, G, buf, 0);
        ag_note_launch();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(map, buf + CMAP_HDR_WORDS, (size_t)CMAP_WORDS * 4, cudaMemcpyDeviceToDevice, s);
    cudaFreeAsync(buf, s);
    return (ag_status)e;
}

ag_status launch_rollout_lut(const ag_params &P, const GridDev &G, const RolloutDev &A, size_t smem_grid, cudaStream_t s) {
    LutConst L;
    L.phase_scale = 4294967296.0 / TWO_PI;
    L.thr_c = (float)P.reach_eps + (AG_DELTA_P + 2.0e-7f);
    L.n_tiles = (A.n + 31) / 32;
    static std::atomic<unsigned> next_slot{0};
    L.slot = next_slot.fetch_add(1, std::memory_order_relaxed) % AG_TILE_SLOTS;
    L.ss_off = (uint32_t)((smem_grid + 15) & ~(size_t)15);
    size_t smem = (size_t)L.ss_off + sizeof(SlowShared);
    const bool ha = A.actions != nullptr, rec = A.rec_j1 != nullptr;
    // the unrolled form tests three squares (scene_0's map); fewer are padded with far-away ones in the kernel
    const bool m3 = A.max_occupied >= 0 && A.max_occupied <= 3;
    // The map form: scene-wide target only (the map holds the target box), |link| small enough for the build's margins
    static const bool no_cmap = std::getenv("AG_ROLLOUT_NO_CMAP") != nullptr;
    L.cmap = nullptr; L.cmap_off = 0;
    if (!no_cmap && A.targets == nullptr) {
        const ag_status st = cspace_map_for_launch(P, G, s, &L.cmap);
        if (st != AG_OK) return st;
        if (L.cmap != nullptr) {
            L.cmap_off = (uint32_t)((smem + 15) & ~(size_t)15);
            smem = (size_t)L.cmap_off + (size_t)CMAP_WORDS * 4;
        }
    }
#define AG_LUT(HA, REC) (L.cmap ? launch_t<HA, REC, false, true>(P, G, A, L, smem, s) \
                                : (m3 ? launch_t<HA, REC, true, false>(P, G, A, L, smem, s) : launch_t<HA, REC, false, false>(P, G, A, L, smem, s)))
    if (ha) return rec ? AG_LUT(true, true) : AG_LUT(true, false);
    return rec ? AG_LUT(false, true) : AG_LUT(false, false);
#undef AG_LUT
}
