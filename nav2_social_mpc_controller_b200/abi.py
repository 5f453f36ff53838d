"""ctypes mirror of include/smpc.h (the C-ABI of libsmpc.so).

The structures here are byte-for-byte the PODs declared in include/smpc.h; they are
also what the CPU oracle (test infrastructure under oracle/) consumes, so parity tests hand the
same buffers to both. Nothing in this module computes anything.
"""
from __future__ import annotations

import ctypes as C
import numpy as np

SMPC_ABI_VERSION = 4
SMPC_MAX_BLOCKS = 18

# enum smpc_termination
CONVERGENCE_GRADIENT = 0
CONVERGENCE_PARAMETER = 1
CONVERGENCE_FUNCTION = 2
CONVERGENCE_RADIUS = 3
NO_CONVERGENCE = 4
FAILURE_INVALID_STEPS = 5
FAILURE_EVALUATION = 6
TERMINATION_NAMES = {
    0: "CONVERGENCE(gradient)", 1: "CONVERGENCE(parameter)", 2: "CONVERGENCE(function)",
    3: "CONVERGENCE(radius)", 4: "NO_CONVERGENCE", 5: "FAILURE(invalid steps)", 6: "FAILURE(evaluation)",
}


class SmpcParams(C.Structure):
    """struct smpc_params — mirrors OptimizerParams (reference optimizer.hpp:59-101)."""
    _fields_ = [
        ("linear_solver_type", C.c_char * 32),
        ("param_tol", C.c_double),
        ("fn_tol", C.c_double),
        ("gradient_tol", C.c_double),
        ("max_iterations", C.c_int),
        ("debug", C.c_int),
        ("control_horizon", C.c_int),
        ("parameter_block_length", C.c_int),
        ("discretization", C.c_int),
        ("distance_w", C.c_double),
        ("socialwork_w", C.c_double),
        ("velocity_w", C.c_double),
        ("angle_w", C.c_double),
        ("agent_angle_w", C.c_double),
        ("proxemics_w", C.c_double),
        ("velocity_feasibility_w", C.c_double),
        ("obstacle_w", C.c_double),
        ("goal_align_w", C.c_double),
        ("current_path_w", C.c_float),
        ("current_cmds_w", C.c_float),
        ("max_time", C.c_float),
        ("time_step", C.c_float),
        ("omnidirectional", C.c_int),
        ("traj_desired_linear_vel", C.c_double),
        ("lookahead_dist", C.c_double),
        ("max_angular_vel", C.c_double),
        ("transform_tolerance", C.c_double),
        ("base_frame", C.c_char * 64),
        ("desired_linear_vel", C.c_double),
        ("fov_angle", C.c_double),
        ("ceres_compat", C.c_int),
        ("max_evaluations", C.c_int),
        ("omni_solve", C.c_int),
    ]


class SmpcBatch(C.Structure):
    """struct smpc_batch — one batch of post-projection MPC problems."""
    _fields_ = [
        ("n_problems", C.c_int),
        ("n_steps", C.c_int),
        ("n_agents", C.c_int),
        ("n_costmaps", C.c_int),
        ("size_x", C.c_int),
        ("size_y", C.c_int),
        ("resolution", C.c_double),
        ("dt", C.c_double),
        ("pose0", C.c_void_p),
        ("u0", C.c_void_p),
        ("path_xy", C.c_void_p),
        ("goal_yaw", C.c_void_p),
        ("agents", C.c_void_p),
        ("has_people", C.c_void_p),
        ("costmaps", C.c_void_p),
        ("costmap_origin", C.c_void_p),
        ("costmap_index", C.c_void_p),
        ("n_steps_each", C.c_void_p),
        ("scenario_index", C.c_void_p),
        ("n_scenarios", C.c_int),
    ]


class SmpcResult(C.Structure):
    _fields_ = [
        ("u", C.c_void_p),
        ("cmds", C.c_void_p),
        ("path", C.c_void_p),
        ("cost_initial", C.c_void_p),
        ("cost_final", C.c_void_p),
        ("iterations", C.c_void_p),
        ("termination", C.c_void_p),
        ("usable", C.c_void_p),
        ("n_evals", C.c_void_p),
        ("trace", C.c_void_p),
        ("trace_rows", C.c_int),
    ]


class SmpcEvalOut(C.Structure):
    _fields_ = [
        ("cost", C.c_void_p),
        ("grad", C.c_void_p),
        ("hess", C.c_void_p),
        ("ok", C.c_void_p),
        ("cost_plain", C.c_void_p),
    ]


def problem_dims(control_horizon: int, block_length: int, n_steps: int):
    """ch, bl, n_blocks, n_bounded exactly as reference src/optimizer.cpp:248-249,254-261,373."""
    ch = min(int(control_horizon), int(n_steps))
    bl = min(int(block_length), ch)
    nb = (ch + bl - 1) // bl
    return ch, bl, nb, ch // bl


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    # torch tensor (device or host)
    return int(a.data_ptr())


BATCH_FIELDS = ("pose0", "u0", "path_xy", "goal_yaw", "agents", "has_people", "costmaps",
                "costmap_origin", "costmap_index", "n_steps_each", "scenario_index")
# with scenario_index these have one row per SCENE (n_scenarios), not per problem (include/smpc.h)
SCENE_FIELDS = ("pose0", "path_xy", "goal_yaw", "agents", "has_people", "costmap_index", "n_steps_each")
BATCH_DTYPES = {"pose0": np.float64, "u0": np.float64, "path_xy": np.float64, "goal_yaw": np.float64,
                "agents": np.float64, "has_people": np.uint8, "costmaps": np.uint8,
                "costmap_origin": np.float64, "costmap_index": np.int32, "n_steps_each": np.int32,
                "scenario_index": np.int32}


def make_batch_struct(arrays: dict, n_problems: int, n_steps: int, n_agents: int, n_costmaps: int,
                      size_x: int, size_y: int, resolution: float, dt: float) -> SmpcBatch:
    """Fill a smpc_batch from numpy arrays or torch tensors (the caller keeps them alive)."""
    b = SmpcBatch()
    b.n_problems, b.n_steps, b.n_agents, b.n_costmaps = n_problems, n_steps, n_agents, n_costmaps
    b.size_x, b.size_y, b.resolution, b.dt = size_x, size_y, float(resolution), float(dt)
    for f in BATCH_FIELDS:
        setattr(b, f, _ptr(arrays.get(f)))
    b.n_scenarios = int(arrays["pose0"].shape[0]) if arrays.get("scenario_index") is not None else 0
    return b


RESULT_FIELDS = ("u", "cmds", "path", "cost_initial", "cost_final", "iterations", "termination", "usable",
                 "n_evals")


def result_shapes(n_problems: int, n_steps: int, n_blocks: int, dof: int = 2):
    """dof = parameters per block: 2 = (v, w), 3 = omnidirectional (vx, vy, w) (smpc_params.omni_solve)."""
    return {
        "u": ((n_problems, n_blocks, dof), np.float64),
        "cmds": ((n_problems, n_steps + 1, dof), np.float64),
        "path": ((n_problems, n_steps + 1, 3), np.float64),
        "cost_initial": ((n_problems,), np.float64),
        "cost_final": ((n_problems,), np.float64),
        "iterations": ((n_problems,), np.int32),
        "termination": ((n_problems,), np.int32),
        "usable": ((n_problems,), np.uint8),
        "n_evals": ((n_problems, 2), np.int32),
    }


def make_result_struct(arrays: dict) -> SmpcResult:
    r = SmpcResult()
    for f in RESULT_FIELDS:
        setattr(r, f, _ptr(arrays.get(f)))
    tr = arrays.get("trace")
    r.trace = _ptr(tr)
    r.trace_rows = int(tr.shape[1]) if tr is not None else 0
    return r


class SmpcObstacleDistance(C.Structure):
    """struct smpc_obstacle_distance — obstacle_distance_msgs::msg::ObstacleDistance."""
    _fields_ = [
        ("width", C.c_uint32),
        ("height", C.c_uint32),
        ("resolution", C.c_float),
        ("origin_x", C.c_double),
        ("origin_y", C.c_double),
        ("distances", C.c_void_p),
        ("indexes", C.c_void_p),
    ]


class SmpcOptimizeIo(C.Structure):
    """struct smpc_optimize_io — arguments of the level-2 entry mirroring Optimizer::optimize."""
    _fields_ = [
        ("capacity", C.c_int),
        ("n_poses", C.c_int),
        ("poses", C.c_void_p),
        ("n_cmds", C.c_int),
        ("cmds", C.c_void_p),
        ("n_people", C.c_int),
        ("people", C.c_void_p),
        ("speed_v", C.c_double),
        ("speed_w", C.c_double),
        ("time_step", C.c_float),
        ("costmap", C.c_void_p),
        ("size_x", C.c_int),
        ("size_y", C.c_int),
        ("origin_x", C.c_double),
        ("origin_y", C.c_double),
        ("resolution", C.c_double),
        ("od", SmpcObstacleDistance),
        ("n_proj_steps", C.c_int),
        ("people_proj", C.c_void_p),
        ("optimized", C.c_int),
        ("termination", C.c_int),
        ("iterations", C.c_int),
        ("cost_initial", C.c_double),
        ("cost_final", C.c_double),
    ]


class SmpcProjectArgs(C.Structure):
    """struct smpc_project_args — batched project_people (SFM crowd projection)."""
    _fields_ = [
        ("n_problems", C.c_int),
        ("n_steps", C.c_int),
        ("n_agents", C.c_int),
        ("n_grids", C.c_int),
        ("od_width", C.c_uint32),
        ("od_height", C.c_uint32),
        ("od_resolution", C.c_float),
        ("max_time", C.c_float),
        ("time_step", C.c_float),
        ("od_origin", C.c_void_p),
        ("od_indexes", C.c_void_p),
        ("od_index", C.c_void_p),
        ("robot", C.c_void_p),
        ("people_init", C.c_void_p),
        ("agents", C.c_void_p),
        ("status", C.c_void_p),
        ("n_steps_each", C.c_void_p),
    ]


class SmpcFormatArgs(C.Structure):
    """struct smpc_format_args — batched format_to_optimize + unpacking."""
    _fields_ = [
        ("n_problems", C.c_int),
        ("n_poses", C.c_int),
        ("n_prev_poses", C.c_int),
        ("n_prev_cmds", C.c_int),
        ("n_blocks", C.c_int),
        ("time_step", C.c_float),
        ("current_path_w", C.c_float),
        ("current_cmds_w", C.c_float),
        ("poses", C.c_void_p),
        ("cmds", C.c_void_p),
        ("speed", C.c_void_p),
        ("prev_poses", C.c_void_p),
        ("prev_cmds", C.c_void_p),
        ("robot", C.c_void_p),
        ("pose0", C.c_void_p),
        ("u0", C.c_void_p),
        ("path_xy", C.c_void_p),
        ("goal_yaw", C.c_void_p),
        ("n_poses_each", C.c_void_p),
        ("n_prev_poses_each", C.c_void_p),
        ("n_prev_cmds_each", C.c_void_p),
        ("cmds_stride", C.c_int),
        ("has_people", C.c_void_p),
    ]


class SmpcTrajectorizeArgs(C.Structure):
    """struct smpc_trajectorize_args — batched PathTrajectorizer::trajectorize."""
    _fields_ = [
        ("n_problems", C.c_int),
        ("n_path", C.c_int),
        ("max_steps", C.c_int),
        ("omnidirectional", C.c_int),
        ("desired_linear_vel", C.c_double),
        ("lookahead_dist", C.c_double),
        ("max_angular_vel", C.c_double),
        ("time_step", C.c_double),
        ("global_path", C.c_void_p),
        ("path_index", C.c_void_p),
        ("pose", C.c_void_p),
        ("poses", C.c_void_p),
        ("cmds", C.c_void_p),
        ("n_steps", C.c_void_p),
    ]


class SmpcFleetIo(C.Structure):
    """struct smpc_fleet_io — one controller tick of a fleet (smpc_optimize_batch)."""
    _fields_ = [
        ("n_robots", C.c_int),
        ("max_poses", C.c_int),
        ("n_agents", C.c_int),
        ("time_step", C.c_float),
        ("n_poses", C.c_void_p),
        ("people", C.c_void_p),
        ("n_people", C.c_void_p),
        ("speed", C.c_void_p),
        ("costmaps", C.c_void_p),
        ("costmap_origin", C.c_void_p),
        ("costmap_index", C.c_void_p),
        ("n_costmaps", C.c_int),
        ("size_x", C.c_int),
        ("size_y", C.c_int),
        ("resolution", C.c_double),
        ("od_indexes", C.c_void_p),
        ("od_origin", C.c_void_p),
        ("od_index", C.c_void_p),
        ("n_od_grids", C.c_int),
        ("od_width", C.c_uint32),
        ("od_height", C.c_uint32),
        ("od_resolution", C.c_float),
        ("maps_version", C.c_longlong),
        ("poses", C.c_void_p),
        ("cmds", C.c_void_p),
        ("n_out", C.c_void_p),
        ("optimized", C.c_void_p),
        ("termination", C.c_void_p),
        ("iterations", C.c_void_p),
        ("cost_initial", C.c_void_p),
        ("cost_final", C.c_void_p),
        ("project_status", C.c_void_p),
        ("people_proj", C.c_void_p),
    ]


class SmpcFovArgs(C.Structure):
    """struct smpc_fov_args — batched FOV people filter of SocialMPCController::computeVelocityCommands."""
    _fields_ = [
        ("n_robots", C.c_int),
        ("n_in_max", C.c_int),
        ("n_out_max", C.c_int),
        ("n_costmaps", C.c_int),
        ("size_x", C.c_int),
        ("size_y", C.c_int),
        ("resolution", C.c_double),
        ("fov_angle", C.c_double),
        ("people_in", C.c_void_p),
        ("n_people_in", C.c_void_p),
        ("pose", C.c_void_p),
        ("costmap_origin", C.c_void_p),
        ("costmap_index", C.c_void_p),
        ("people_out", C.c_void_p),
        ("n_people_out", C.c_void_p),
    ]


class SmpcEpisodeIo(C.Structure):
    """struct smpc_episode_io — closed-loop episodes (smpc_run_episodes)."""
    _fields_ = [
        ("n_episodes", C.c_int),
        ("n_ticks", C.c_int),
        ("n_path", C.c_int),
        ("n_people", C.c_int),
        ("n_agents", C.c_int),
        ("control_period", C.c_double),
        ("goal_tolerance", C.c_double),
        ("global_path", C.c_void_p),
        ("pose", C.c_void_p),
        ("speed", C.c_void_p),
        ("people", C.c_void_p),
        ("n_people_each", C.c_void_p),
        ("costmaps", C.c_void_p),
        ("costmap_origin", C.c_void_p),
        ("costmap_index", C.c_void_p),
        ("n_costmaps", C.c_int),
        ("size_x", C.c_int),
        ("size_y", C.c_int),
        ("resolution", C.c_double),
        ("od_indexes", C.c_void_p),
        ("od_origin", C.c_void_p),
        ("od_index", C.c_void_p),
        ("n_od_grids", C.c_int),
        ("od_width", C.c_uint32),
        ("od_height", C.c_uint32),
        ("od_resolution", C.c_float),
        ("reached", C.c_void_p),
        ("ticks", C.c_void_p),
        ("path_length", C.c_void_p),
        ("min_person_dist", C.c_void_p),
        ("intimate_ticks", C.c_void_p),
        ("personal_ticks", C.c_void_p),
        ("collision_ticks", C.c_void_p),
        ("not_optimized_ticks", C.c_void_p),
        ("cmd_variation", C.c_void_p),
        ("pose_log", C.c_void_p),
        ("cmd_log", C.c_void_p),
        ("optimized_log", C.c_void_p),
    ]


class SmpcCrowdIo(C.Structure):
    """struct smpc_crowd_io — the reactive crowd of smpc_run_crowd_episodes."""
    _fields_ = [
        ("goals", C.c_void_p),
        ("desired_speed", C.c_void_p),
        ("substeps", C.c_int),
        ("people_disturbance", C.c_void_p),
        ("people_log", C.c_void_p),
    ]


class SmpcSceneIo(C.Structure):
    """struct smpc_scene_io — the shared scenes of smpc_run_shared_episodes."""
    _fields_ = [
        ("robots_per_scene", C.c_int),
        ("robot_min_dist", C.c_void_p),
        ("robot_intimate_ticks", C.c_void_p),
    ]
