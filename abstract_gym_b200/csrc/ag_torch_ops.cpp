// ag_torch_ops.cpp -- torch.ops.abstract_gym_b200.*: a compiled custom-op library over the C ABI.
//
// Thin by design (BASELINE.json north_star: "a thin C-ABI PyTorch custom-op extension"): every op checks device /
// dtype / contiguity / shapes, takes the current CUDA stream of the tensors' device and calls the extern "C" entry
// point of include/abstract_gym_b200.h in libabstract_gym_b200.so.  There is no CPU dispatch key: the ops are
// registered for CUDA only, so CPU tensors raise NotImplementedError.  State tensors are mutated in place
// (declared in the schemas), nothing is allocated and nothing synchronises, so the ops can sit inside CUDA-graph
// captures next to a policy network -- except cspace_distance, which synchronises with its stream to detect convergence
// (ag_cspace_distance) and fails inside a capture.
//
// Scene constants travel as a float64[13] CPU tensor (ag_params order, see pack_params in ops.py) that is read in
// place; the grid as its device tensors plus six scalars.  The reference methods each op replaces are cited in the
// header next to the entry point it forwards to.
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <cstdint>

#include "../../include/abstract_gym_b200.h"

namespace {

using at::Tensor;
using OptTensor = std::optional<Tensor>;

const char *status_text(ag_status s) { return ag_status_string(s); }

void check_status(ag_status s, const char *what) {
    TORCH_CHECK(s == AG_OK, what, " failed: status ", (int)s, " (", status_text(s), ")");
}

void need(const Tensor &t, at::ScalarType dt, const char *name, c10::Device dev) {
    TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (no CPU dispatch)");
    TORCH_CHECK(t.device() == dev, name, " is on ", t.device(), ", expected ", dev);
    TORCH_CHECK(t.scalar_type() == dt, name, " must be ", dt, ", got ", t.scalar_type());
    TORCH_CHECK(t.is_contiguous(), name, " must be contiguous");
}

// element counts are checked before anything launches: an undersized tensor would be read or written out of bounds
void need_numel(const Tensor &t, int64_t count, const char *name) {
    TORCH_CHECK(t.numel() == count, name, " must have ", count, " elements, got ", t.numel());
}

void opt_numel(const OptTensor &t, int64_t count, const char *name) {
    if (t.has_value() && t->defined()) need_numel(*t, count, name);
}

template <typename T>
T *opt_ptr(const OptTensor &t, at::ScalarType dt, const char *name, c10::Device dev) {
    if (!t.has_value() || !t->defined()) return nullptr;
    need(*t, dt, name, dev);
    return reinterpret_cast<T *>(t->data_ptr());
}

ag_params unpack_params(const Tensor &p) {
    TORCH_CHECK(p.device().is_cpu() && p.scalar_type() == at::kDouble && p.numel() == 13 && p.is_contiguous(),
                "params must be a contiguous float64[13] CPU tensor (ops.pack_params)");
    const double *v = p.data_ptr<double>();
    ag_params q;
    q.link_1 = v[0]; q.link_2 = v[1]; q.target_x = v[2]; q.target_y = v[3]; q.target_j1 = v[4]; q.target_j2 = v[5];
    q.reach_eps = v[6]; q.section_eps = v[7]; q.reward_collision = v[8]; q.reward_reach = v[9]; q.action_scale = v[10];
    q.choose_j_tar = (int32_t)v[11]; q.max_reset_tries = (int32_t)v[12];
    return q;
}

ag_grid make_grid(const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x, const Tensor &min_y, double side,
                  double env_size, int64_t S, int64_t n_grids, int64_t max_occupied, int64_t envs_per_grid, c10::Device dev) {
    need(bits, at::kInt, "grid_bits", dev);
    need(min_x, at::kDouble, "min_x", dev);
    need(min_y, at::kDouble, "min_y", dev);
    TORCH_CHECK(min_x.numel() >= S && min_y.numel() >= S, "corner tables shorter than S");
    ag_grid g;
    g.bits = reinterpret_cast<const uint32_t *>(bits.data_ptr());
    g.bits_t = opt_ptr<const uint32_t>(bits_t, at::kInt, "grid_bits_t", dev);
    g.hier = opt_ptr<const void>(hier, at::kByte, "grid_hier", dev);
    TORCH_CHECK(g.hier == nullptr || hier->numel() == n_grids * ag_grid_hier_bytes((int32_t)S),
                "grid_hier must hold n_grids * ag_grid_hier_bytes(S) bytes (ag_grid_pack_hier)");
    g.min_x = min_x.data_ptr<double>(); g.min_y = min_y.data_ptr<double>();
    g.side = side; g.env_size = env_size;
    g.S = (int32_t)S; g.words_per_row = ag_grid_words_per_row((int32_t)S);
    g.n_grids = (int32_t)n_grids; g.max_occupied = (int32_t)max_occupied;
    g.grid_stride_words = ag_grid_stride_words((int32_t)S);
    g.envs_per_grid = envs_per_grid;
    TORCH_CHECK(bits.numel() == n_grids * g.grid_stride_words, "grid_bits must hold n_grids * ag_grid_stride_words(S) words");
    return g;
}

void *stream_of(c10::Device dev) { return c10::cuda::getCurrentCUDAStream(dev.index()).stream(); }

// Scene.collision_check (scenario/scene_0.py:60-76) -> ag_collision_check
void collision_check(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x, const Tensor &min_y,
                     double side, double env_size, int64_t S, int64_t n_grids, int64_t max_occupied, int64_t envs_per_grid,
                     const Tensor &j1, const Tensor &j2, Tensor hit, OptTensor first_hit, int64_t env_id0, int64_t engine) {
    const c10::Device dev = j1.device();
    c10::cuda::CUDAGuard guard(dev);
    need(j1, at::kDouble, "j1", dev); need(j2, at::kDouble, "j2", dev); need(hit, at::kByte, "hit", dev);
    TORCH_CHECK(j2.numel() == j1.numel() && hit.numel() == j1.numel(), "j1, j2, hit must have one element per env");
    opt_numel(first_hit, j1.numel(), "first_hit");
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_collision_check(&p, &g, j1.data_ptr<double>(), j2.data_ptr<double>(), hit.data_ptr<uint8_t>(),
                                    opt_ptr<int32_t>(first_hit, at::kInt, "first_hit", dev), j1.numel(), env_id0,
                                    (int32_t)engine, stream_of(dev)), "ag_collision_check");
}

// move_to_joint_pose with a collision check at every pose (two_joint_robot.py:49-62, scene_0.py:60-76) -> ag_check_motion
void check_motion(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x,
                  const Tensor &min_y, double side, double env_size, int64_t S, int64_t n_grids, int64_t max_occupied,
                  int64_t envs_per_grid, const Tensor &j1, const Tensor &j2, const Tensor &goal, const Tensor &steps,
                  Tensor first_collision, OptTensor first_hit, OptTensor last_free, int64_t env_id0, int64_t engine) {
    const c10::Device dev = j1.device();
    c10::cuda::CUDAGuard guard(dev);
    need(j1, at::kDouble, "j1", dev); need(j2, at::kDouble, "j2", dev); need(goal, at::kDouble, "goal", dev);
    need(steps, at::kInt, "steps", dev); need(first_collision, at::kInt, "first_collision", dev);
    const int64_t m = j1.numel();
    TORCH_CHECK(j2.numel() == m && steps.numel() == m && first_collision.numel() == m, "j1, j2, steps, first_collision must have one element per motion");
    TORCH_CHECK(goal.numel() == 2 * m, "goal must be [M,2]");
    if (first_hit.has_value() && first_hit->defined()) TORCH_CHECK(first_hit->numel() == m, "first_hit must be [M]");
    if (last_free.has_value() && last_free->defined()) TORCH_CHECK(last_free->numel() == 2 * m, "last_free must be [M,2]");
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_check_motion(&p, &g, j1.data_ptr<double>(), j2.data_ptr<double>(), goal.data_ptr<double>(),
                                 steps.data_ptr<int32_t>(), first_collision.data_ptr<int32_t>(),
                                 opt_ptr<int32_t>(first_hit, at::kInt, "first_hit", dev), opt_ptr<double>(last_free, at::kDouble, "last_free", dev),
                                 m, env_id0, (int32_t)engine, stream_of(dev)),
                 "ag_check_motion");
}

// collision_check (scene_0.py:60-76) at every pose of a joint-angle lattice, per grid -> ag_cspace_occupancy
void cspace_occupancy(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x,
                      const Tensor &min_y, double side, double env_size, int64_t S, int64_t n_grids, int64_t max_occupied,
                      int64_t envs_per_grid, double lo1, double step1, int64_t b1, double lo2, double step2, int64_t b2,
                      Tensor occupancy, OptTensor free_count, int64_t engine) {
    const c10::Device dev = occupancy.device();
    c10::cuda::CUDAGuard guard(dev);
    need(occupancy, at::kInt, "occupancy", dev);
    TORCH_CHECK(b1 >= 1 && b2 >= 1 && b1 <= INT32_MAX && b2 <= INT32_MAX, "b1 and b2 must be in [1, 2^31)");
    const int64_t grid_words = b1 * ((b2 + 31) / 32);
    TORCH_CHECK(n_grids >= 1 && grid_words <= INT64_MAX / n_grids && occupancy.numel() == n_grids * grid_words,
                "occupancy must be [n_grids, b1, ceil(b2/32)] int32 words");
    if (free_count.has_value() && free_count->defined()) TORCH_CHECK(free_count->numel() == n_grids, "free_count must be [n_grids]");
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_cspace_occupancy(&p, &g, lo1, step1, (int32_t)b1, lo2, step2, (int32_t)b2,
                                     reinterpret_cast<uint32_t *>(occupancy.data_ptr()),
                                     opt_ptr<int64_t>(free_count, at::kLong, "free_count", dev), (int32_t)engine, stream_of(dev)),
                 "ag_cspace_occupancy");
}

// connected components of the free poses of cspace_occupancy's words, per grid -> ag_cspace_components
void cspace_components(const Tensor &occupancy, int64_t b1, int64_t b2, int64_t wrap, Tensor labels, OptTensor n_components) {
    const c10::Device dev = labels.device();
    c10::cuda::CUDAGuard guard(dev);
    need(occupancy, at::kInt, "occupancy", dev);
    need(labels, at::kInt, "labels", dev);
    TORCH_CHECK(b1 >= 1 && b2 >= 1 && b1 <= INT32_MAX && b2 <= INT32_MAX && b1 * b2 <= INT32_MAX,
                "b1 and b2 must be >= 1 with b1 * b2 < 2^31");
    const int64_t grid_words = b1 * ((b2 + 31) / 32);
    TORCH_CHECK(occupancy.numel() % grid_words == 0, "occupancy must be [n_grids, b1, ceil(b2/32)] int32 words");
    const int64_t n_grids = occupancy.numel() / grid_words;
    TORCH_CHECK(labels.numel() == n_grids * b1 * b2, "labels must be [n_grids, b1, b2] int32");
    if (n_components.has_value() && n_components->defined())
        TORCH_CHECK(n_components->numel() == n_grids, "n_components must be [n_grids]");
    check_status(ag_cspace_components(reinterpret_cast<const uint32_t *>(occupancy.data_ptr()), n_grids, (int32_t)b1,
                                      (int32_t)b2, (int32_t)wrap, labels.data_ptr<int32_t>(),
                                      opt_ptr<int64_t>(n_components, at::kLong, "n_components", dev), stream_of(dev)),
                 "ag_cspace_components");
}

// steps from every free pose of cspace_occupancy's words to a goal image in the same layout, per grid -> ag_cspace_distance
void cspace_distance(const Tensor &occupancy, const Tensor &goals, int64_t b1, int64_t b2, int64_t wrap, Tensor dist,
                     OptTensor max_dist) {
    const c10::Device dev = dist.device();
    c10::cuda::CUDAGuard guard(dev);
    need(occupancy, at::kInt, "occupancy", dev);
    need(goals, at::kInt, "goals", dev);
    need(dist, at::kInt, "dist", dev);
    TORCH_CHECK(b1 >= 1 && b2 >= 1 && b1 <= INT32_MAX && b2 <= INT32_MAX && b1 * b2 < INT32_MAX,
                "b1 and b2 must be >= 1 with b1 * b2 < 2^31 - 1");
    const int64_t grid_words = b1 * ((b2 + 31) / 32);
    TORCH_CHECK(occupancy.numel() % grid_words == 0, "occupancy must be [n_grids, b1, ceil(b2/32)] int32 words");
    const int64_t n_grids = occupancy.numel() / grid_words;
    TORCH_CHECK(goals.numel() == occupancy.numel(), "goals must have the layout of occupancy");
    TORCH_CHECK(dist.numel() == n_grids * b1 * b2, "dist must be [n_grids, b1, b2] int32");
    if (max_dist.has_value() && max_dist->defined()) TORCH_CHECK(max_dist->numel() == n_grids, "max_dist must be [n_grids]");
    check_status(ag_cspace_distance(reinterpret_cast<const uint32_t *>(occupancy.data_ptr()),
                                    reinterpret_cast<const uint32_t *>(goals.data_ptr()), n_grids, (int32_t)b1, (int32_t)b2,
                                    (int32_t)wrap, dist.data_ptr<int32_t>(),
                                    opt_ptr<int32_t>(max_dist, at::kInt, "max_dist", dev), stream_of(dev)),
                 "ag_cspace_distance");
}

// lattice paths down a cspace_distance field -> ag_cspace_descend
void cspace_descend(const Tensor &dist, int64_t b1, int64_t b2, int64_t wrap, const Tensor &start, const Tensor &grid,
                    int64_t max_len, Tensor path, Tensor length) {
    const c10::Device dev = path.device();
    c10::cuda::CUDAGuard guard(dev);
    need(dist, at::kInt, "dist", dev);
    need(start, at::kInt, "start", dev);
    need(grid, at::kLong, "grid", dev);
    need(path, at::kInt, "path", dev);
    need(length, at::kInt, "length", dev);
    TORCH_CHECK(b1 >= 1 && b2 >= 1 && b1 <= INT32_MAX && b2 <= INT32_MAX && b1 * b2 < INT32_MAX,
                "b1 and b2 must be >= 1 with b1 * b2 < 2^31 - 1");
    TORCH_CHECK(dist.numel() % (b1 * b2) == 0, "dist must be [n_grids, b1, b2] int32");
    TORCH_CHECK(max_len >= 1 && max_len <= INT32_MAX, "max_len must be in [1, 2^31)");
    const int64_t m = start.numel();
    TORCH_CHECK(grid.numel() == m && length.numel() == m, "start, grid, length must have one element per query");
    TORCH_CHECK(path.numel() == m * max_len, "path must be [M, max_len] int32");
    check_status(ag_cspace_descend(dist.data_ptr<int32_t>(), dist.numel() / (b1 * b2), (int32_t)b1, (int32_t)b2,
                                   (int32_t)wrap, start.data_ptr<int32_t>(), grid.data_ptr<int64_t>(), m, (int32_t)max_len,
                                   path.data_ptr<int32_t>(), length.data_ptr<int32_t>(), stream_of(dev)),
                 "ag_cspace_descend");
}

// Scene.step (scenario/scene_0.py:88-103) -> ag_step
void step(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x, const Tensor &min_y, double side,
          double env_size, int64_t S, int64_t n_grids, int64_t max_occupied, int64_t envs_per_grid, Tensor j1, Tensor j2,
          const Tensor &actions, Tensor reward, Tensor flags, OptTensor ee, OptTensor dist, OptTensor first_hit, OptTensor stats,
          const OptTensor &targets, int64_t env_id0, int64_t engine) {
    const c10::Device dev = j1.device();
    c10::cuda::CUDAGuard guard(dev);
    need(j1, at::kDouble, "j1", dev); need(j2, at::kDouble, "j2", dev);
    need(reward, at::kFloat, "reward", dev); need(flags, at::kByte, "flags", dev);
    const int64_t n = j1.numel();
    TORCH_CHECK(actions.is_cuda() && actions.is_contiguous() && actions.numel() == 2 * n &&
                (actions.scalar_type() == at::kFloat || actions.scalar_type() == at::kDouble),
                "actions must be a contiguous CUDA [N,2] float32 or float64 tensor");
    need_numel(j2, n, "j2"); need_numel(reward, n, "reward"); need_numel(flags, n, "flags");
    opt_numel(ee, 2 * n, "ee"); opt_numel(dist, 2 * n, "dist"); opt_numel(first_hit, n, "first_hit");
    opt_numel(stats, AG_ST_COUNT, "stats"); opt_numel(targets, 2 * n, "targets");
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_step(&p, &g, j1.data_ptr<double>(), j2.data_ptr<double>(), actions.data_ptr(),
                         actions.scalar_type() == at::kFloat ? 1 : 0, reward.data_ptr<float>(), flags.data_ptr<uint8_t>(),
                         opt_ptr<double>(ee, at::kDouble, "ee", dev), opt_ptr<double>(dist, at::kDouble, "dist", dev),
                         opt_ptr<int32_t>(first_hit, at::kInt, "first_hit", dev), opt_ptr<int64_t>(stats, at::kLong, "stats", dev),
                         opt_ptr<const double>(targets, at::kDouble, "targets", dev), n, env_id0, (int32_t)engine, stream_of(dev)),
                 "ag_step");
}

// Scene.reset / random_valid_pose (scenario/scene_0.py:105-113,174-181) -> ag_reset
void reset(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x, const Tensor &min_y, double side,
           double env_size, int64_t S, int64_t n_grids, int64_t max_occupied, int64_t envs_per_grid, Tensor j1, Tensor j2,
           Tensor reward, Tensor flags, Tensor reset_ctr, const OptTensor &mask, const OptTensor &reset_u, OptTensor stats,
           int64_t seed, bool clear_flags, int64_t env_id0, int64_t engine) {
    const c10::Device dev = j1.device();
    c10::cuda::CUDAGuard guard(dev);
    need(j1, at::kDouble, "j1", dev); need(j2, at::kDouble, "j2", dev);
    need(reward, at::kFloat, "reward", dev); need(flags, at::kByte, "flags", dev); need(reset_ctr, at::kInt, "reset_ctr", dev);
    const int64_t n = j1.numel();
    int32_t R = 0;
    if (reset_u.has_value() && reset_u->defined()) {
        TORCH_CHECK(reset_u->dim() == 3 && reset_u->size(0) == n && reset_u->size(2) == 2, "reset_u must be [N,R,2]");
        R = (int32_t)reset_u->size(1);
    }
    need_numel(j2, n, "j2"); need_numel(reward, n, "reward"); need_numel(flags, n, "flags"); need_numel(reset_ctr, n, "reset_ctr");
    opt_numel(mask, n, "mask"); opt_numel(stats, AG_ST_COUNT, "stats");
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_reset(&p, &g, j1.data_ptr<double>(), j2.data_ptr<double>(), reward.data_ptr<float>(), flags.data_ptr<uint8_t>(),
                          reinterpret_cast<uint32_t *>(reset_ctr.data_ptr()), opt_ptr<const uint8_t>(mask, at::kByte, "mask", dev),
                          opt_ptr<const double>(reset_u, at::kDouble, "reset_u", dev), R, (uint64_t)seed, clear_flags ? 1 : 0,
                          opt_ptr<int64_t>(stats, at::kLong, "stats", dev), n, env_id0, (int32_t)engine, stream_of(dev)),
                 "ag_reset");
}

// the loop body of experiment/experiment_0.py:20-34 fused over K steps -> ag_rollout
void rollout(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x, const Tensor &min_y, double side,
             double env_size, int64_t S, int64_t n_grids, int64_t max_occupied, int64_t envs_per_grid, Tensor j1, Tensor j2,
             Tensor reward, Tensor flags, Tensor step_ctr, Tensor reset_ctr, Tensor ep_len, const OptTensor &actions,
             const OptTensor &reset_u, const OptTensor &targets, OptTensor rec_j1, OptTensor rec_j2, OptTensor rec_reward,
             OptTensor rec_flags, Tensor stats, OptTensor diag, OptTensor events, OptTensor event_count, int64_t K, int64_t seed,
             int64_t env_id0, int64_t engine) {
    const c10::Device dev = j1.device();
    c10::cuda::CUDAGuard guard(dev);
    need(j1, at::kDouble, "j1", dev); need(j2, at::kDouble, "j2", dev);
    need(reward, at::kFloat, "reward", dev); need(flags, at::kByte, "flags", dev);
    need(step_ctr, at::kInt, "step_ctr", dev); need(reset_ctr, at::kInt, "reset_ctr", dev); need(ep_len, at::kInt, "ep_len", dev);
    need(stats, at::kLong, "stats", dev);
    const int64_t n = j1.numel();
    need_numel(j2, n, "j2"); need_numel(reward, n, "reward"); need_numel(flags, n, "flags");
    need_numel(step_ctr, n, "step_ctr"); need_numel(reset_ctr, n, "reset_ctr"); need_numel(ep_len, n, "ep_len");
    need_numel(stats, AG_ST_COUNT, "stats"); opt_numel(diag, AG_DIAG_COUNT, "diag"); opt_numel(targets, 2 * n, "targets");
    opt_numel(event_count, 1, "event_count");
    ag_rollout_args a = {};
    a.n = n; a.env_id0 = env_id0; a.K = (int32_t)K; a.engine = (int32_t)engine; a.seed = (uint64_t)seed;
    if (actions.has_value() && actions->defined())
        TORCH_CHECK(actions->dim() == 3 && actions->size(0) == K && actions->size(1) == n && actions->size(2) == 2, "actions must be [K,N,2]");
    a.actions = opt_ptr<const float>(actions, at::kFloat, "actions", dev);
    if (reset_u.has_value() && reset_u->defined()) {
        TORCH_CHECK(reset_u->dim() == 3 && reset_u->size(0) == n && reset_u->size(2) == 2, "reset_u must be [N,R,2]");
        a.R = (int32_t)reset_u->size(1);
    }
    a.reset_u = opt_ptr<const double>(reset_u, at::kDouble, "reset_u", dev);
    a.targets = opt_ptr<const double>(targets, at::kDouble, "targets", dev);
    a.j1 = j1.data_ptr<double>(); a.j2 = j2.data_ptr<double>(); a.reward = reward.data_ptr<float>(); a.flags = flags.data_ptr<uint8_t>();
    a.step_ctr = reinterpret_cast<uint32_t *>(step_ctr.data_ptr()); a.reset_ctr = reinterpret_cast<uint32_t *>(reset_ctr.data_ptr());
    a.ep_len = reinterpret_cast<uint32_t *>(ep_len.data_ptr());
    for (const OptTensor *r : {&rec_j1, &rec_j2, &rec_reward, &rec_flags})
        if (r->has_value() && (*r)->defined()) TORCH_CHECK((*r)->numel() == K * n, "record planes must be [K,N]");
    a.rec_j1 = opt_ptr<float>(rec_j1, at::kFloat, "rec_j1", dev); a.rec_j2 = opt_ptr<float>(rec_j2, at::kFloat, "rec_j2", dev);
    a.rec_reward = opt_ptr<float>(rec_reward, at::kFloat, "rec_reward", dev);
    a.rec_flags = opt_ptr<uint8_t>(rec_flags, at::kByte, "rec_flags", dev);
    a.stats = stats.data_ptr<int64_t>();
    a.diag = opt_ptr<int64_t>(diag, at::kLong, "diag", dev);
    a.events = opt_ptr<uint32_t>(events, at::kInt, "events", dev);
    a.event_count = opt_ptr<int64_t>(event_count, at::kLong, "event_count", dev);
    if (a.events) a.event_capacity = events->numel() / 3;
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_rollout(&p, &g, &a, stream_of(dev)), "ag_rollout");
}

// fused gym-style step (scenario/vector_env.py): Scene.step + same-step auto-reset + observations -> ag_step_obs
void step_obs(const Tensor &params, const Tensor &bits, const OptTensor &bits_t, const OptTensor &hier, const Tensor &min_x, const Tensor &min_y, double side,
              double env_size, int64_t S, int64_t n_grids, int64_t max_occupied, int64_t envs_per_grid, Tensor j1, Tensor j2,
              const Tensor &actions, Tensor reward, Tensor flags, Tensor reset_ctr, Tensor ep_len, const OptTensor &targets, Tensor obs,
              Tensor reward_out, Tensor terminated, Tensor collision, OptTensor final_obs, OptTensor crop, Tensor stats, int64_t seed,
              bool auto_reset, int64_t env_id0, int64_t engine) {
    const c10::Device dev = j1.device();
    c10::cuda::CUDAGuard guard(dev);
    need(j1, at::kDouble, "j1", dev); need(j2, at::kDouble, "j2", dev);
    need(reward, at::kFloat, "reward", dev); need(flags, at::kByte, "flags", dev);
    need(reset_ctr, at::kInt, "reset_ctr", dev); need(ep_len, at::kInt, "ep_len", dev);
    need(obs, at::kDouble, "obs", dev); need(reward_out, at::kFloat, "reward_out", dev);
    need(terminated, at::kByte, "terminated", dev); need(collision, at::kByte, "collision", dev); need(stats, at::kLong, "stats", dev);
    const int64_t n = j1.numel();
    TORCH_CHECK(actions.is_cuda() && actions.is_contiguous() && actions.numel() == 2 * n &&
                (actions.scalar_type() == at::kFloat || actions.scalar_type() == at::kDouble),
                "actions must be a contiguous CUDA [N,2] float32 or float64 tensor");
    TORCH_CHECK(obs.numel() == n * AG_OBS_DIM, "obs must be [N,", AG_OBS_DIM, "]");
    for (const auto &[t, name] : {std::pair<const Tensor *, const char *>{&j2, "j2"}, {&reward, "reward"}, {&flags, "flags"},
                                  {&reset_ctr, "reset_ctr"}, {&ep_len, "ep_len"}, {&reward_out, "reward_out"},
                                  {&terminated, "terminated"}, {&collision, "collision"}})
        TORCH_CHECK(t->numel() == n, name, " must have one element per env (", n, "), got ", t->numel());
    TORCH_CHECK(stats.numel() == AG_ST_COUNT, "stats must be int64[", AG_ST_COUNT, "], got ", stats.numel(), " elements");
    if (targets.has_value() && targets->defined()) TORCH_CHECK(targets->numel() == 2 * n, "targets must be [N,2]");
    if (final_obs.has_value() && final_obs->defined())
        TORCH_CHECK(final_obs->numel() == n * AG_OBS_DIM, "final_obs must be [N,", AG_OBS_DIM, "]");
    int32_t crop_size = 0;
    if (crop.has_value() && crop->defined()) {
        TORCH_CHECK(crop->dim() == 3 && crop->size(0) == n && crop->size(1) == crop->size(2), "crop must be [N,c,c]");
        crop_size = (int32_t)crop->size(1);
    }
    const ag_params p = unpack_params(params);
    const ag_grid g = make_grid(bits, bits_t, hier, min_x, min_y, side, env_size, S, n_grids, max_occupied, envs_per_grid, dev);
    check_status(ag_step_obs(&p, &g, j1.data_ptr<double>(), j2.data_ptr<double>(), actions.data_ptr(),
                             actions.scalar_type() == at::kFloat ? 1 : 0, reward.data_ptr<float>(), flags.data_ptr<uint8_t>(),
                             reinterpret_cast<uint32_t *>(reset_ctr.data_ptr()), reinterpret_cast<uint32_t *>(ep_len.data_ptr()),
                             opt_ptr<const double>(targets, at::kDouble, "targets", dev), obs.data_ptr<double>(),
                             reward_out.data_ptr<float>(), terminated.data_ptr<uint8_t>(), collision.data_ptr<uint8_t>(),
                             opt_ptr<double>(final_obs, at::kDouble, "final_obs", dev), opt_ptr<uint8_t>(crop, at::kByte, "crop", dev),
                             crop_size, stats.data_ptr<int64_t>(), (uint64_t)seed, auto_reset ? 1 : 0, n, env_id0, (int32_t)engine,
                             stream_of(dev)),
                 "ag_step_obs");
}

#define AG_GRID_SCHEMA "Tensor params, Tensor grid_bits, Tensor? grid_bits_t, Tensor? grid_hier, Tensor min_x, Tensor min_y, float side, float env_size, " \
                       "int S, int n_grids, int max_occupied, int envs_per_grid, "

}  // namespace

TORCH_LIBRARY(abstract_gym_b200, m) {
    m.def("collision_check(" AG_GRID_SCHEMA "Tensor j1, Tensor j2, Tensor(a!) hit, Tensor(b!)? first_hit, int env_id0, int engine) -> ()");
    m.def("check_motion(" AG_GRID_SCHEMA "Tensor j1, Tensor j2, Tensor goal, Tensor steps, Tensor(a!) first_collision, "
          "Tensor(b!)? first_hit, Tensor(c!)? last_free, int env_id0, int engine) -> ()");
    m.def("cspace_occupancy(" AG_GRID_SCHEMA "float lo1, float step1, int b1, float lo2, float step2, int b2, "
          "Tensor(a!) occupancy, Tensor(b!)? free_count, int engine) -> ()");
    m.def("cspace_components(Tensor occupancy, int b1, int b2, int wrap, Tensor(a!) labels, Tensor(b!)? n_components) -> ()");
    m.def("cspace_distance(Tensor occupancy, Tensor goals, int b1, int b2, int wrap, Tensor(a!) dist, Tensor(b!)? max_dist) -> ()");
    m.def("cspace_descend(Tensor dist, int b1, int b2, int wrap, Tensor start, Tensor grid, int max_len, Tensor(a!) path, "
          "Tensor(b!) length) -> ()");
    m.def("step(" AG_GRID_SCHEMA "Tensor(a!) j1, Tensor(b!) j2, Tensor actions, Tensor(c!) reward, Tensor(d!) flags, Tensor(e!)? ee, "
          "Tensor(f!)? dist, Tensor(g!)? first_hit, Tensor(h!)? stats, Tensor? targets, int env_id0, int engine) -> ()");
    m.def("reset(" AG_GRID_SCHEMA "Tensor(a!) j1, Tensor(b!) j2, Tensor(c!) reward, Tensor(d!) flags, Tensor(e!) reset_ctr, Tensor? mask, "
          "Tensor? reset_u, Tensor(f!)? stats, int seed, bool clear_flags, int env_id0, int engine) -> ()");
    m.def("rollout(" AG_GRID_SCHEMA "Tensor(a!) j1, Tensor(b!) j2, Tensor(c!) reward, Tensor(d!) flags, Tensor(e!) step_ctr, "
          "Tensor(f!) reset_ctr, Tensor(g!) ep_len, Tensor? actions, Tensor? reset_u, Tensor? targets, Tensor(h!)? rec_j1, "
          "Tensor(i!)? rec_j2, Tensor(j!)? rec_reward, Tensor(k!)? rec_flags, Tensor(l!) stats, Tensor(m!)? diag, Tensor(n!)? events, "
          "Tensor(o!)? event_count, int K, int seed, int env_id0, int engine) -> ()");
    m.def("step_obs(" AG_GRID_SCHEMA "Tensor(a!) j1, Tensor(b!) j2, Tensor actions, Tensor(c!) reward, Tensor(d!) flags, "
          "Tensor(e!) reset_ctr, Tensor(f!) ep_len, Tensor? targets, Tensor(g!) obs, Tensor(h!) reward_out, Tensor(i!) terminated, "
          "Tensor(j!) collision, Tensor(k!)? final_obs, Tensor(l!)? crop, Tensor(m!) stats, int seed, bool auto_reset, int env_id0, "
          "int engine) -> ()");
}

TORCH_LIBRARY_IMPL(abstract_gym_b200, CUDA, m) {
    m.impl("collision_check", &collision_check);
    m.impl("check_motion", &check_motion);
    m.impl("cspace_occupancy", &cspace_occupancy);
    m.impl("cspace_components", &cspace_components);
    m.impl("cspace_distance", &cspace_distance);
    m.impl("cspace_descend", &cspace_descend);
    m.impl("step", &step);
    m.impl("reset", &reset);
    m.impl("rollout", &rollout);
    m.impl("step_obs", &step_obs);
}
