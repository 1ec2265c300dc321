/*
 * abstract_gym_b200.h -- C ABI of the B200-native batched scene_0 simulator.
 *
 * The reference (tualatint/abstract_gym) is pure Python and has no FFI of its own; the boundary it
 * offers is its class API.  Each entry point below names the reference method it replaces
 * (file:line relative to the reference root).  The Python host package (abstract_gym_b200/) keeps
 * the reference's class names/signatures and calls these symbols through ctypes; INTEGRATION.md
 * shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns ag_status (0 = ok, <0 = argument/shape error, >0 = cudaError_t);
 *     nothing throws across the boundary; no hidden global state;
 *   - unless a name ends in _host, every pointer is a DEVICE pointer owned by the caller and all
 *     work is enqueued on `stream` (a cudaStream_t passed as void*); calls are stream-ordered,
 *     re-entrant and never synchronise -- except ag_cspace_distance, which synchronises with its stream to
 *     detect convergence (and so cannot be captured in a CUDA graph);
 *   - *_host entry points take HOST pointers, do their own H2D/D2H copies and return after the
 *     results are in the host buffers;
 *   - there is no CPU implementation behind any of these symbols: without a CUDA device they
 *     return cudaErrorNoDevice / cudaErrorInsufficientDriver.
 */
#ifndef ABSTRACT_GYM_B200_H
#define ABSTRACT_GYM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AG_ABI_VERSION 9

#if defined(__GNUC__)
#define AG_API __attribute__((visibility("default")))
#else
#define AG_API
#endif

typedef int32_t ag_status;
enum {
    AG_OK = 0,
    AG_ERR_NULL = -1,        /* a required pointer is NULL */
    AG_ERR_SHAPE = -2,       /* n < 0, K < 1, S < 2, bad strides ... */
    AG_ERR_MODE = -3,        /* unknown mode / unsupported combination */
    AG_ERR_ALIGN = -4,       /* pointer not aligned as documented */
    AG_ERR_NOT_SQUARE = -5   /* occupancy matrix is not square (occupancy_grid.py:80-82) */
};

/* Scene constants: the literals of scenario/scene_0.py:17,30-31,78,96,99,122,
 * utils/collision_checker.py:81 and robot/two_joint_robot.py:12-13 (ag_default_params fills
 * them).  Passed by pointer from HOST memory; copied into the launch. */
typedef struct ag_params {
    double link_1, link_2;
    double target_x, target_y;       /* Scene.target_c */
    double target_j1, target_j2;     /* Scene.target_j */
    double reach_eps;                /* check_target_reached epsilon */
    double section_eps;              /* check_sections epsilon */
    double reward_collision;
    double reward_reach;
    double action_scale;             /* sample_action scale_factor */
    int32_t choose_j_tar;            /* Scene.choose_j_tar */
    int32_t max_reset_tries;         /* bound on random_valid_pose's loop (unbounded in the reference) */
} ag_params;

/* Bit-packed occupancy grid(s) + the float64 cell-corner tables (environment/occupancy_grid.py:
 * 28,59-67).  Bit c%32 of word bits[g*grid_stride_words + r*words_per_row + c/32] is cell
 * (row r, col c) of grid g; row 0 is the TOP row (y flipped), exactly the reference's `occ` matrix.
 * min_x[c], min_y[r] hold the reference's rounded corner values; max = min + side.
 * Env with global id e uses grid (e / envs_per_grid) % n_grids.  Passed from HOST memory; the
 * pointers inside are DEVICE pointers. */
typedef struct ag_grid {
    const uint32_t *bits;
    const double *min_x;             /* [S] */
    const double *min_y;             /* [S] */
    double side;                     /* E / (S-1) */
    double env_size;                 /* E */
    int32_t S;
    int32_t words_per_row;           /* ceil(S/32) */
    int32_t n_grids;
    int32_t max_occupied;            /* upper bound on occupied cells of any grid; < 0 = unknown (hint only) */
    int64_t grid_stride_words;       /* >= S*words_per_row, multiple of 4 (16-byte rows for bulk copies) */
    int64_t envs_per_grid;
    const uint32_t *bits_t;          /* optional transposed copy (same strides): bit r%32 of word
                                      * bits_t[g*grid_stride_words + c*words_per_row + r/32] is cell (row r, col c), i.e.
                                      * ag_grid_pack of the transposed matrices; NULL = none.  With it the FAST engine walks
                                      * a link along its minor axis (columns for shallow links) instead of always by rows. */
    const void *hier;                /* optional two-level form of the same bits, ag_grid_hier_bytes(S) bytes per grid, written
                                      * by ag_grid_pack_hier (NULL = none).  With T = ceil(S/8): first T*T uint64 "tiles" (padded
                                      * to an even count), tile (R, C) holding the 8x8 block of cells with bit (r%8)*8 + c%8 for
                                      * cell (8R + r%8, 8C + c%8); then a T x T summary bitmap, ceil(T/32) words per row (padded
                                      * to a multiple of 4 words), bit C%32 of word R*ceil(T/32) + C/32 set iff tile (R, C) has
                                      * an occupied cell; then the same bitmap transposed (bit R%32 of word C*ceil(T/32) + R/32).
                                      * With it the FAST engine walks a link over the summary along its minor axis (8x fewer,
                                      * at most T/sqrt(2) lines) and looks at the cells of occupied tiles only. */
} ag_grid;

/* Collision engine selection. All three return identical flags (tests/test_gpu_parity.py):
 *   EXACT : float64, reference operation order, conservative cell traversal of the bit grid;
 *   FAST  : float32 interval filter, float64 EXACT re-evaluation of every undecided lane;
 *   BRUTE : float64, every occupied cell of the grid (the reference's O(#obstacles) loop,
 *           scenario/scene_0.py:67) -- the on-device cross-check of the traversal. */
enum { AG_ENGINE_EXACT = 0, AG_ENGINE_FAST = 1, AG_ENGINE_BRUTE = 2 };

/* sticky flag bits (Scene.collision_status / Scene.done, scenario/scene_0.py:33-40) */
enum { AG_FLAG_COLLISION = 1, AG_FLAG_DONE = 2 };

/* episode statistics, int64 counters (the reference prints "records:"/"succ:" experiment_0.py:35-36) */
enum {
    AG_ST_EPISODES = 0,      /* terminal steps (done or collision) */
    AG_ST_COLLISIONS,        /* episodes that ended with collision_status set */
    AG_ST_SUCCESSES,         /* episodes that ended with done set */
    AG_ST_ENV_STEPS,
    AG_ST_EP_LEN_SUM,
    AG_ST_RETURN_MILLI,      /* sum of terminal rewards / 1000 (-1 or +10 each) */
    AG_ST_STUCK_RESETS,      /* resets that exhausted max_reset_tries / the candidate list */
    AG_ST_AXIS_ALIGNED,      /* check_sections a==0/b==0 evaluations (AttributeError in the reference) */
    AG_ST_COUNT
};

/* FAST-engine diagnostics of ag_rollout (not part of the reference's semantics; ag_rollout_args.diag) */
enum {
    AG_DIAG_EXACT_STEPS = 0, /* env-steps whose float32 filter was undecided and that were re-evaluated in float64 */
    AG_DIAG_COLD_CALLS,      /* lane visits of the out-of-line section (undecided steps + episode ends) */
    AG_DIAG_WARP_EXITS,      /* times a warp left the call-free inner loop */
    AG_DIAG_COUNT
};

/* ---- host-only helpers (no device needed) ------------------------------------------------- */

AG_API int32_t ag_abi_version(void);
AG_API const char *ag_status_string(ag_status s);
AG_API void ag_default_params(ag_params *p);
AG_API int32_t ag_grid_words_per_row(int32_t S);
AG_API int64_t ag_grid_stride_words(int32_t S);
AG_API int64_t ag_grid_hier_bytes(int32_t S);    /* size of ag_grid.hier per grid (a multiple of 16) */

/* OccupancyGrid.__init__/load_from_matrix -> packed bits (occupancy_grid.py:25-50,73-93).
 * occ: rows x cols uint8 host matrix (non-zero = occupied); bits_out: ag_grid_stride_words(S) words. */
AG_API ag_status ag_grid_pack_host(const uint8_t *occ, int32_t rows, int32_t cols, uint32_t *bits_out);
/* OccupancyGrid.transform_frame corner arithmetic (occupancy_grid.py:28,59-67), host float64. */
AG_API ag_status ag_grid_tables_host(int32_t S, double env_size, double *min_x, double *min_y, double *side);

/* ---- device entry points ------------------------------------------------------------------- */

/* K5: pack n_grids S x S uint8 occupancy matrices (device) into bits (device). */
AG_API ag_status ag_grid_pack(const uint8_t *occ, int32_t S, int32_t n_grids, uint32_t *bits,
                       int64_t grid_stride_words, void *stream);
/* the two-level form (ag_grid.hier) of n_grids packed grids: bits (device) -> hier (device, 16-byte aligned,
 * n_grids * ag_grid_hier_bytes(S) bytes) */
AG_API ag_status ag_grid_pack_hier(const uint32_t *bits, int32_t S, int32_t n_grids, int64_t grid_stride_words, void *hier,
                            void *stream);

/* utils/geometry.py:14-32 Line.compute_line_function() and utils/collision_checker.py:12-46
 * CollisionChecker(line, square).compute_corner_line_value()/.collision_check() over arrays.
 * seg: [n][4] (p0x,p0y,p1x,p1y); sq: [n][4] (min_x,min_y,max_x,max_y); hit: [n] uint8.
 * Optional: abc [n][3] line coefficients; corner_values [n][4] (v1..v4 before np.sign);
 * axis_aligned int64[1] counter (accumulated). */
AG_API ag_status ag_segment_square(const double *seg, const double *sq, double section_eps, uint8_t *hit,
                            double *abc, double *corner_values, int64_t *axis_aligned, int64_t n,
                            void *stream);

/* robot/two_joint_robot.py:31-47  elbow_point()/end_effector() over arrays.
 * out: [n][4] (elbow_x, elbow_y, ee_x, ee_y). */
AG_API ag_status ag_forward_kinematics(const ag_params *p, const double *j1, const double *j2, double *out,
                                int64_t n, void *stream);

/* robot/two_joint_robot.py:74-113  cart_target_valid_check() + inverse_kinematic() over arrays (off the step/reset
 * path).  target: [n][2]; sol: [n][4] = (j1_1, j2_1, j1_2, j2_2), zeros where valid[i] == 0 (target outside the
 * annulus |l1-l2| < r <= l1+l2: the reference prints "Target out of reach." and returns None).
 * corrected != 0: alpha = atan2(y, x) instead of the reference's arccos(x/r), which drops the sign of y. */
AG_API ag_status ag_inverse_kinematics(const ag_params *p, const double *target, double *sol, uint8_t *valid,
                                int32_t corrected, int64_t n, void *stream);

/* robot/two_joint_robot.py:49-62  move_to_joint_pose(target_j1, target_j2, steps): target [n][2]; j1, j2 in/out. */
AG_API ag_status ag_move_to_joint_pose(double *j1, double *j2, const double *target, int32_t steps, int64_t n,
                                void *stream);

/* K2: scenario/scene_0.py:60-76  Scene.collision_check().  hit: [n] uint8; first_hit: optional
 * [n] int32 = min(row*S+col) over all cells hit by either link, -1 if none. */
AG_API ag_status ag_collision_check(const ag_params *p, const ag_grid *g, const double *j1, const double *j2,
                             uint8_t *hit, int32_t *first_hit, int64_t n, int64_t env_id0,
                             int32_t engine, void *stream);

/* Motion checking: robot/two_joint_robot.py:49-62 move_to_joint_pose() with scenario/scene_0.py:60-76
 * Scene.collision_check() at every intermediate pose (the reference checks none of them).  Motion i starts at
 * (j1[i], j2[i]) and goes to goal[i] = (g1, g2) in n = steps[i] increments: alpha = 1.0 / n, inc = alpha * (g - start),
 * pose_k = pose_{k-1} + inc for k = 1 .. n, pose_0 = start -- float64, one rounding per operation, the k-fold SEQUENTIAL
 * sum (not start + k * inc), so a free motion ends exactly where ag_move_to_joint_pose(start, goal, n) does.  The start
 * pose is not checked (the arm is already there; Scene.step, too, checks only after the move); poses 1 .. n are, and a
 * pose collides exactly when ag_collision_check with the same engine says so.  Motion i uses grid
 * ((env_id0 + i) / envs_per_grid) % n_grids.  A motion stops at its first colliding pose.
 * goal, last_free: [m][2] float64 (16-byte aligned); steps: [m] int32; all device arrays.  Outputs:
 *   first_collision [m] int32: the smallest colliding k, -1 if the motion is free, -2 if steps[i] < 1 (nothing is
 *                   checked; the reference divides by zero there);
 *   first_hit       optional [m] int32: min(row*S+col) over the cells hit at pose first_collision (as K2 reports it),
 *                   -1 if none;
 *   last_free       optional [m][2] float64: the last pose before the first collision -- the start when it is pose 1
 *                   or when steps[i] < 1, pose n when the motion is free. */
AG_API ag_status ag_check_motion(const ag_params *p, const ag_grid *g, const double *j1, const double *j2, const double *goal,
                                 const int32_t *steps, int32_t *first_collision, int32_t *first_hit, double *last_free,
                                 int64_t m, int64_t env_id0, int32_t engine, void *stream);

/* Configuration-space occupancy: scenario/scene_0.py:60-76 Scene.collision_check() at every pose of a b1 x b2 lattice of
 * joint angles, for every grid g = 0 .. n_grids-1 -- the obstacle image of the configuration-space torus, exact (unlike
 * ag_cspace_map's conservative bins).  Pose (i, j) = (lo1 + (double)i * step1, lo2 + (double)j * step2): float64, one
 * rounding per operation, never contracted to an FMA.  Its bit is 1 exactly when ag_collision_check with the same engine
 * says that pose collides on grid g (a grid's staging and broad phase are those of K2 launched on that grid's own envs
 * from an env_id0 that is a multiple of 256).
 * bits: [n_grids][b1][W] uint32 (device), W = ceil(b2 / 32); pose (i, j) is bit j % 32 of word j / 32 of row i; the
 *       padding bits of a row's last word are 0.  With b2 a multiple of 32 this is ag_cspace_map's bit order.
 * free_count: optional [n_grids] int64 (device, 8-byte aligned): the collision-free poses of each grid, written (not
 *       accumulated).
 * Errors, before anything touches the device: b1 < 1 or b2 < 1, a non-finite lo or step, or n_grids * b1 * W beyond
 * int64 -> AG_ERR_SHAPE; the grid checks of ag_collision_check; bits NULL -> AG_ERR_NULL; an unknown engine ->
 * AG_ERR_MODE.  Stream-ordered (the free counts are zeroed by a memset on `stream`) and capturable in a CUDA graph. */
AG_API ag_status ag_cspace_occupancy(const ag_params *p, const ag_grid *g, double lo1, double step1, int32_t b1, double lo2,
                                     double step2, int32_t b2, uint32_t *bits, int64_t *free_count, int32_t engine,
                                     void *stream);

/* Free-space components: the connected components of the free poses (bit 0) of an occupancy image in the layout
 * ag_cspace_occupancy writes, per grid g = 0 .. n_grids-1.  No grid or params: this is image work on the words alone.
 * bits: [n_grids][b1][W] uint32 (device, 4-byte aligned), W = ceil(b2 / 32); pose (i, j) is bit j % 32 of word j / 32 of
 *       row i, 1 = colliding.  Padding bits (j >= b2) are ignored: those poses do not exist.
 * Free poses (i, j) and (i+-1, j), (i, j+-1) are adjacent (4-neighbour: a diagonal step would pass a blocked corner).
 * wrap bit 0: row b1-1 is adjacent to row 0 (joint_1 wraps); bit 1: column b2-1 to column 0 (joint_2 wraps); both: the
 * torus.  A pose is never its own neighbour (b = 1 adds no edge).  Grids never connect to each other.
 * labels: [n_grids][b1][b2] int32 (device, 4-byte aligned, no padding): -1 for a colliding pose, else the smallest
 *       row-major index i * b2 + j (local to the grid) of any pose of its component -- canonical, so the result does not
 *       depend on scheduling.
 * n_components: optional [n_grids] int64 (device, 8-byte aligned): the components of each grid, written (not
 *       accumulated).
 * This is connectivity of the LATTICE image: two adjacent free poses may have a colliding pose between them when the
 * lattice is coarse for the grid's cells.  Nothing here checks the motion between them (ag_check_motion does).
 * Errors, in this order, before anything touches the device: n_grids < 0, b1 < 1 or b2 < 1, b1 * b2 > INT32_MAX or
 * n_grids * b1 * b2 beyond int64 -> AG_ERR_SHAPE; wrap & ~3 -> AG_ERR_MODE; n_grids == 0 -> AG_OK (nothing launched);
 * bits or labels NULL -> AG_ERR_NULL; a misaligned pointer -> AG_ERR_ALIGN.  Stream-ordered, no scratch memory, no host
 * synchronisation (the counts are zeroed by a memset on `stream`): capturable in a CUDA graph. */
AG_API ag_status ag_cspace_components(const uint32_t *bits, int64_t n_grids, int32_t b1, int32_t b2, int32_t wrap,
                                      int32_t *labels, int64_t *n_components, void *stream);

/* Free-space distance: the fewest 4-neighbour steps through free poses from every pose of an occupancy image to a goal
 * pose, per grid g = 0 .. n_grids-1 (a multi-source BFS on the lattice).  No grid or params: image work on the words.
 * bits, goals: [n_grids][b1][W] uint32 (device, 4-byte aligned), W = ceil(b2 / 32), the layout ag_cspace_occupancy writes:
 *       pose (i, j) is bit j % 32 of word j / 32 of row i; bits: 1 = colliding; goals: 1 = goal.  Padding bits (j >= b2)
 *       are ignored, and so are goal bits on colliding poses: neither seeds anything.
 * Adjacency is that of ag_cspace_components: 4 neighbours, wrap bit 0 joins row b1-1 to row 0, bit 1 column b2-1 to
 * column 0, a pose is never its own neighbour and grids never connect.
 * dist: [n_grids][b1][b2] int32 (device, 4-byte aligned, no padding): -1 for a colliding pose; -2 for a free pose whose
 *       component holds no free goal; else the fewest steps to a free goal (0 at a free goal).  This distance is unique,
 *       so the result does not depend on scheduling.
 * max_dist: optional [n_grids] int32 (device, 4-byte aligned): the largest distance of each grid, -1 if no pose reaches a
 *       goal; written (not accumulated).
 * Like ag_cspace_components this is the LATTICE image: a step between adjacent free poses may cross a colliding pose in
 * continuous joint space when the lattice is coarse (ag_check_motion checks such a step).
 * Errors, in this order, before anything touches the device: n_grids < 0, b1 < 1 or b2 < 1, b1 * b2 > INT32_MAX - 1 or
 * n_grids * b1 * b2 beyond int64 -> AG_ERR_SHAPE; wrap & ~3 -> AG_ERR_MODE; n_grids == 0 -> AG_OK (nothing launched);
 * bits, goals or dist NULL -> AG_ERR_NULL; a misaligned pointer -> AG_ERR_ALIGN.
 * THE ONE EXCEPTION to "never synchronise": this call synchronises with `stream` every few relaxation passes to learn
 * whether the field has converged.  It returns once it has; the final pass (the -2 marks and max_dist) is enqueued on
 * `stream` after the last synchronisation, so the results are stream-ordered like those of every other call.  On a stream
 * that is capturing a CUDA graph it returns cudaErrorStreamCaptureUnsupported before it enqueues anything, and the
 * capture stays intact.  Scratch memory (tile stamps, change counters) comes from cudaMallocAsync on `stream`. */
AG_API ag_status ag_cspace_distance(const uint32_t *bits, const uint32_t *goals, int64_t n_grids, int32_t b1, int32_t b2,
                                    int32_t wrap, int32_t *dist, int32_t *max_dist, void *stream);

/* Lattice descent: m paths down a distance field of ag_cspace_distance (same n_grids, b1, b2, wrap).  Query q starts at
 * the grid-local row-major index start[q] = i * b2 + j on grid grid[q].  path[q][0] = start; from a pose at distance
 * d > 0 the next pose is the FIRST neighbour in the order (i+1, j), (i-1, j), (i, j+1), (i, j-1) that exists (across a
 * seam only where that axis wraps) and has distance d - 1, so the path is canonical.  The walk stops at distance 0 or
 * after max_len poses.
 * dist: [n_grids][b1][b2] int32; start: [m] int32; grid: [m] int64 (8-byte aligned); path: [m][max_len] int32;
 * length: [m] int32 -- all device arrays.  length[q] = min(dist(start) + 1, max_len), and 0 when start is outside
 * [0, b1 * b2), grid[q] outside [0, n_grids), or the start pose is colliding or unreachable (dist < 0): these are device
 * data, not errors.  path[q][k] = -1 for k >= length[q].
 * Errors, in this order, before anything touches the device: n_grids < 0, b1 < 1 or b2 < 1, b1 * b2 > INT32_MAX - 1 or
 * n_grids * b1 * b2 beyond int64, m < 0, max_len < 1 or m * max_len beyond int64 -> AG_ERR_SHAPE; wrap & ~3 ->
 * AG_ERR_MODE; m == 0 -> AG_OK (nothing launched); dist, start, grid, path or length NULL -> AG_ERR_NULL; a misaligned
 * pointer -> AG_ERR_ALIGN.  Stream-ordered, never synchronises: capturable in a CUDA graph. */
AG_API ag_status ag_cspace_descend(const int32_t *dist, int64_t n_grids, int32_t b1, int32_t b2, int32_t wrap,
                                   const int32_t *start, const int64_t *grid, int64_t m, int32_t max_len, int32_t *path,
                                   int32_t *length, void *stream);

/* K1: scenario/scene_0.py:88-103  Scene.step(action).  j1,j2,reward,flags are in/out (sticky
 * semantics).  actions: [n][2] float64 (actions_f32 == 0) or float32.  Optional outputs:
 * ee [n][2] float64 end effector, dist [n][2] float64 (|tx-EEx|, |ty-EEy|), first_hit [n] int32.
 * targets: optional [n][2] float64 per-env cartesian targets replacing Scene.target_c (NULL = p->target_x/y;
 * ignored in joint-target mode). */
AG_API ag_status ag_step(const ag_params *p, const ag_grid *g, double *j1, double *j2, const void *actions,
                  int32_t actions_f32, float *reward, uint8_t *flags, double *ee, double *dist,
                  int32_t *first_hit, int64_t *stats, const double *targets, int64_t n, int64_t env_id0,
                  int32_t engine, void *stream);

/* K3: scenario/scene_0.py:105-113,174-181  Scene.reset() / random_valid_pose() for envs with
 * mask[e] != 0 (mask == NULL: all).  Candidates come from reset_u [n][R][2] float64 uniforms
 * (consumed from reset_ctr[e]) or, when reset_u == NULL, from Philox stream 1 keyed by
 * (seed, env_id0+e).  clear_flags != 0 -> reset() (clears reward/flags); 0 -> random_valid_pose(). */
AG_API ag_status ag_reset(const ag_params *p, const ag_grid *g, double *j1, double *j2, float *reward,
                   uint8_t *flags, uint32_t *reset_ctr, const uint8_t *mask, const double *reset_u,
                   int32_t R, uint64_t seed, int32_t clear_flags, int64_t *stats, int64_t n,
                   int64_t env_id0, int32_t engine, void *stream);

/* K6: the gym-style step of an RL training loop (the caller of Scene.step / Scene.reset, scenario/scene_0.py:88-113,
 * restarted the way experiment/experiment_0.py:30-34 does) in one launch: step, terminal observation, episode
 * statistics, Scene.reset() of terminated envs (auto_reset != 0; Philox stream 1 candidates keyed by (seed, env_id0+e),
 * consumed from reset_ctr) and the observation the env continues from.
 * reward / flags: the sticky Scene.step_reward / flags, in/out (cleared by the auto-reset).
 * obs, final_obs (optional): [n][AG_OBS_DIM] float64 = (joint_1, joint_2, EE_x, EE_y, |target_x-EE_x|, |target_y-EE_y|) --
 * the last two are the quantities check_target_reached thresholds (scene_0.py:129-130).  reward_out / terminated /
 * collision: this step's (joint_1, joint_2, step_reward, done|collision, collision_status) return values.
 * crop (optional): [n][crop_size][crop_size] uint8 occupancy of the cells centred on the end effector's cell
 * (1 occupied, 2 outside the grid; row 0 = top); crop_size odd, <= 63. */
#define AG_OBS_DIM 6
AG_API ag_status ag_step_obs(const ag_params *p, const ag_grid *g, double *j1, double *j2, const void *actions,
                      int32_t actions_f32, float *reward, uint8_t *flags, uint32_t *reset_ctr, uint32_t *ep_len,
                      const double *targets, double *obs, float *reward_out, uint8_t *terminated, uint8_t *collision,
                      double *final_obs, uint8_t *crop, int32_t crop_size, int64_t *stats, uint64_t seed,
                      int32_t auto_reset, int64_t n, int64_t env_id0, int32_t engine, void *stream);

/* K4: the rollout loop experiment/experiment_0.py:20-34 fused over K steps:
 *   action -> step -> record -> if done|collision: reset.
 * actions: [K][n][2] float32, or NULL = Philox stream 0 (float64 (u-0.5)*action_scale).
 * reset_u: as ag_reset.  rec_*: [K][n]; all four, or rec_j1 + rec_j2 only (with or without the event sink), or all
 * NULL (statistics only).
 * stats: int64[AG_ST_COUNT], accumulated with one atomic per block per slot. */
typedef struct ag_rollout_args {
    int64_t n;
    int64_t env_id0;
    int32_t K;               /* steps fused in this launch, 1 .. 65536 */
    int32_t engine;
    uint64_t seed;
    const float *actions;
    const double *reset_u;
    int32_t R;
    int32_t reserved;
    double *j1, *j2;
    float *reward;
    uint8_t *flags;
    uint32_t *step_ctr, *reset_ctr, *ep_len;
    float *rec_j1, *rec_j2, *rec_reward;
    uint8_t *rec_flags;
    int64_t *stats;
    int64_t *diag;           /* optional int64[AG_DIAG_COUNT] filter diagnostics (accumulated), or NULL */
    const double *targets;   /* optional [n][2] float64 per-env cartesian targets replacing Scene.target_c in the reach
                              * test (scenario/scene_0.py:129-130), or NULL = p->target_x/y; ignored in joint-target mode */
    /* Event sink (optional).  In a rollout record reward and flags are zero for all but the terminal steps (~0.1 % of
     * the env-steps on scene_0), so a caller may leave rec_reward / rec_flags NULL (rec_j1 / rec_j2 only) and collect
     * the eventful steps here instead: events[3*i] = local env index, events[3*i+1] = (step << 8) | flags with
     * step = event_step0 + step within this launch, events[3*i+2] = the float32 bits of step_reward.  *event_count is
     * advanced by one per event (atomically, in no particular order); events beyond event_capacity are counted but
     * not stored. */
    uint32_t *events;
    int64_t *event_count;
    int64_t event_capacity;
    int32_t event_step0;
    int32_t reserved2;
} ag_rollout_args;

AG_API ag_status ag_rollout(const ag_params *p, const ag_grid *g, const ag_rollout_args *a, void *stream);

/* The configuration-space map ag_rollout consults for scene_0-class grids (one staged grid of at most 8 occupied
 * cells, S <= 32, FAST engine, scene-wide cartesian target): one bit per bin of (joint_1, joint_2) mod 2 pi,
 * 2^*b1 x 2^*b2 bins; bit (i1 << *b2 | i2) is bit (i & 31) of word i >> 5.  CLEAR means: for every pose of the bin,
 * Scene.collision_check() is False and check_target_reached() is False (scenario/scene_0.py:60-76,129-130), so a step
 * that lands there is uneventful; SET means "evaluate".  ag_rollout builds and caches the map itself (validated against
 * the current grid and parameters at every launch); this entry point builds it into a caller's device buffer of
 * ag_cspace_map_words() uint32 words -- it exists for inspection and for tests/test_gpu_parity.py, which checks the
 * CLEAR guarantee against the BRUTE engine. */
AG_API int64_t ag_cspace_map_words(int32_t *b1, int32_t *b2);
AG_API ag_status ag_cspace_map(const ag_params *p, const ag_grid *g, uint32_t *map, void *stream);

/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
AG_API int64_t ag_launch_count(void);

/* ---- host-buffer entry points (end-to-end path) -------------------------------------------- */

/* Opaque pipelined executor: owns device staging buffers and streams for chunked
 * H2D(actions) -> K4 -> D2H(records) with copies overlapping compute. */
typedef struct ag_pipeline ag_pipeline;

/* n envs resident on `device`, K steps per call, records enabled or not.  chunk_steps > 0: the rollout is
 * sliced over steps (all envs, chunk_steps steps per stage; contiguous copies -- the faster form); otherwise over
 * envs (chunk_envs envs per stage, all K steps: one kernel launch per env slice). */
AG_API ag_status ag_pipeline_create(ag_pipeline **out, int32_t device, int64_t n, int32_t K,
                             int64_t chunk_envs, int32_t chunk_steps, int32_t record, int64_t event_capacity);
AG_API void ag_pipeline_destroy(ag_pipeline *pl);
/* Same as ag_rollout but actions / rec_* / stats_host are HOST pointers (pinned for full speed);
 * env state pointers inside `a` stay DEVICE pointers (the state lives in HBM between calls).
 * a->rec_reward may be NULL while the other three record pointers are set ("compact records": the reward of a
 * rollout record is a function of its flags -- reward_reach if done, else reward_collision if collision, else 0 --
 * so it need not cross PCIe).  a->actions == NULL: the actions are drawn in the kernel (Philox stream 0), nothing is
 * copied to the device.  a->events / a->event_count: HOST pointers here (the pipeline was created with
 * event_capacity > 0); the events of the whole call are appended from index 0, *event_count is SET to their number.
 * stats_host (int64[AG_ST_COUNT], may be NULL) is ACCUMULATED into: zero it to get this call's counters.
 * Returns after all records, events and stats are on the host; on failure every stream of the pipeline has been
 * synchronised, so no copy is still writing the caller's buffers.  The caller's current device is preserved. */
AG_API ag_status ag_rollout_host(ag_pipeline *pl, const ag_params *p, const ag_grid *g,
                          const ag_rollout_args *a, int64_t *stats_host);

#ifdef __cplusplus
}
#endif
#endif
