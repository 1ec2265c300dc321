"""torch custom ops over the C ABI: `torch.ops.abstract_gym_b200.{collision_check, check_motion, cspace_occupancy,
cspace_components, cspace_distance, cspace_descend, step, reset, rollout, step_obs}`.

The ops live in a COMPILED library, libabstract_gym_b200_ops.so (csrc/ag_torch_ops.cpp: TORCH_LIBRARY schemas, CUDA-only
registration), which validates device / dtype / contiguity / shapes, takes the current CUDA stream and calls the
`extern "C"` symbols of include/abstract_gym_b200.h.  This module loads that library and offers the two packing helpers
the schemas need.  There is no CPU dispatch: a CPU tensor raises NotImplementedError.  The ops mutate their state
tensors in place (declared in the schemas) and return nothing, so they can sit inside captured graphs next to a policy
network.  The one exception is cspace_distance: it synchronises with its stream to detect convergence, so it cannot be
captured (inside a capture it raises and the capture stays intact).

The image ops take no scene: cspace_components(occupancy, b1, b2, wrap, labels, n_components?),
cspace_distance(occupancy, goals, b1, b2, wrap, dist, max_dist?) and cspace_descend(dist, b1, b2, wrap, start, grid,
max_len, path, length) (include/abstract_gym_b200.h).  Every other op starts with the same eleven scene / grid arguments:
    params        float64[13] CPU tensor  = pack_params(scene.params())      (ag_params)
    grid_bits     int32 [n_grids * stride] CUDA, grid_bits_t (optional transposed planes), grid_hier (optional two-level form, uint8), min_x, min_y float64 [>= S]
    side, env_size, S, n_grids, max_occupied, envs_per_grid                   = grid_args(device_grid)
The object API (`BatchedScene`, `VectorEnv`) is the convenient front end; these ops are the functional one.
"""
import torch

from . import _lib
from . import build as _build

NS = "abstract_gym_b200"
_loaded = False


def load():
    """Load (building in-tree if needed) the compiled op library.  Raises if that is impossible."""
    global _loaded
    if _loaded:
        return
    _lib.load()                                   # libabstract_gym_b200.so first: the op library links against it
    if _build.ops_needs_build():
        try:
            _build.build_ops()
        except Exception as e:
            raise ImportError("abstract_gym_b200: the torch op library %s is stale or missing and could not be built (%s)"
                              % (_build.OPS_LIB, e)) from e
    torch.ops.load_library(_build.OPS_LIB)
    _loaded = True


def pack_params(p: _lib.Params) -> torch.Tensor:
    return torch.tensor([p.link_1, p.link_2, p.target_x, p.target_y, p.target_j1, p.target_j2, p.reach_eps,
                         p.section_eps, p.reward_collision, p.reward_reach, p.action_scale, float(p.choose_j_tar),
                         float(p.max_reset_tries)], dtype=torch.float64)


def grid_args(dg):
    """dg: abstract_gym_b200.DeviceGrid -> the eleven grid arguments every op takes after `params`"""
    return (dg.bits, dg.bits_t, dg.hier, dg.min_x, dg.min_y, float(dg.side), float(dg.environment_size), int(dg.S), int(dg.n_grids),
            int(dg.max_occupied), int(dg.envs_per_grid))


load()
collision_check = torch.ops.abstract_gym_b200.collision_check
check_motion = torch.ops.abstract_gym_b200.check_motion
cspace_occupancy = torch.ops.abstract_gym_b200.cspace_occupancy
cspace_components = torch.ops.abstract_gym_b200.cspace_components
cspace_distance = torch.ops.abstract_gym_b200.cspace_distance
cspace_descend = torch.ops.abstract_gym_b200.cspace_descend
step = torch.ops.abstract_gym_b200.step
reset = torch.ops.abstract_gym_b200.reset
rollout = torch.ops.abstract_gym_b200.rollout
step_obs = torch.ops.abstract_gym_b200.step_obs
