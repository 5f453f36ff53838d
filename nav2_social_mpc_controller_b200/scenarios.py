"""Synthetic MPC scenarios for tests and benchmarks (SURVEY §8d), host side, numpy only.

Every batch is built the way the reference builds the Ceres problem input:
  global path + robot pose --(pure-pursuit seed, reference src/path_trajectorizer.cpp:120-288)-->
  seed poses + cmds --(cut + blend, reference src/optimizer.cpp:484-551)--> robot AgentTrajectory
  --> pose0 / u0 / path_xy / goal_yaw of include/smpc.h (u0 follows SURVEY Q1).
People are projected with a constant-velocity model here (the level-1 C-ABI takes post-projection
agents; the SFM projection of src/optimizer.cpp:554-671 is a separate pre-solve stage).

Random numbers: numpy Philox counter-based generator, seed = 20261018 + config id.
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np

from . import abi

SEED_BASE = 20261018

# FollowPath.optimizer / trajectorizer values of the reference parameter sets (values only):
#   readme        reference README.md:75-99 (BASELINE.json config 1 text)
#   params_yaml   reference params/params.yaml:25-55
#   obst_only     reference params/obst_only_parameters_in_benchmark.yaml:104-136
#   soc_work_obst reference params/soc_work_obst_parameters_in_benchmark.yaml:104-136
# Weights a yaml does not set keep the defaults of reference src/optimizer.cpp:57-75 (e.g. proxemics 90, SURVEY Q13).
_DEFAULT_W = dict(distance_w=3.0, socialwork_w=1.0, velocity_w=0.5, angle_w=0.0, agent_angle_w=0.5,
                  proxemics_w=90.0, velocity_feasibility_w=0.5, obstacle_w=0.0, goal_align_w=0.0)
PARAM_SETS = {
    "readme": dict(time_step=0.1, max_time=1.5, control_horizon=18, parameter_block_length=6, lookahead_dist=2.0,
                   current_cmds_w=0.5, distance_w=20.0, socialwork_w=120.0, velocity_w=10.0, angle_w=250.0,
                   agent_angle_w=40.0, velocity_feasibility_w=5.0, goal_align_w=10.0, obstacle_w=0.15,
                   proxemics_w=100.0),
    "params_yaml": dict(time_step=0.05, max_time=2.0, control_horizon=20, parameter_block_length=4,
                        lookahead_dist=1.0, discretization=2, transform_tolerance=0.3, current_cmds_w=0.5, distance_w=50.0, socialwork_w=700.0,
                        velocity_w=8.0, angle_w=180.0, agent_angle_w=0.0, velocity_feasibility_w=5.0,
                        goal_align_w=8.0, obstacle_w=0.2),
    "obst_only": dict(time_step=0.05, max_time=1.5, control_horizon=18, parameter_block_length=6,
                      lookahead_dist=2.0, current_cmds_w=0.5, distance_w=20.0, socialwork_w=0.0, velocity_w=10.0,
                      angle_w=250.0, agent_angle_w=0.0, velocity_feasibility_w=5.0, goal_align_w=10.0,
                      obstacle_w=0.13),
    "soc_work_obst": dict(time_step=0.05, max_time=1.5, control_horizon=18, parameter_block_length=6,
                          lookahead_dist=2.0, current_cmds_w=0.5, distance_w=20.0, socialwork_w=120.0,
                          velocity_w=10.0, angle_w=250.0, agent_angle_w=40.0, velocity_feasibility_w=5.0,
                          goal_align_w=10.0, obstacle_w=0.13),
}
_COMMON = dict(linear_solver_type="DENSE_SCHUR", param_tol=1e-9, fn_tol=1e-5, gradient_tol=1e-8,
               max_iterations=40, debug=0, discretization=1, current_path_w=1.0, omnidirectional=0,
               traj_desired_linear_vel=0.6, max_angular_vel=1.4, transform_tolerance=0.5,
               base_frame="base_link", desired_linear_vel=0.5, fov_angle=math.pi / 4, ceres_compat=200,
               max_evaluations=0, omni_solve=0)


def make_params(name: str, **overrides) -> abi.SmpcParams:
    """smpc_params for one of the reference parameter sets (see PARAM_SETS)."""
    vals = dict(_DEFAULT_W)
    vals.update(_COMMON)
    vals.update(PARAM_SETS[name])
    vals.update(overrides)
    p = abi.SmpcParams()
    for k, v in vals.items():
        if k in ("linear_solver_type", "base_frame"):
            setattr(p, k, v.encode())
        else:
            setattr(p, k, v)
    return p


def f32(x: float) -> float:
    """(double)(float)x — how time_step/max_time reach the functors (SURVEY Q15)."""
    return float(np.float32(x))


def yaw_roundtrip(yaw):
    """tf2 setRPY(0,0,yaw) -> getYaw (SURVEY Q14)."""
    h = np.asarray(yaw, dtype=np.float64) * 0.5
    qz, qw = np.sin(h), np.cos(h)
    return np.arctan2(2.0 * (qw * qz), qw * qw - qz * qz)


def seed_steps(p: abi.SmpcParams) -> int:
    """S = N_v for a full-length seed: trajectorizer emits max_steps+1 poses
    (reference src/path_trajectorizer.cpp:84,152), format_to_optimize keeps maxsize-1 of them
    (reference src/optimizer.cpp:492-497), one velocity is dropped (:237)."""
    max_steps = int(round(float(p.max_time) / float(p.time_step)))
    return max_steps - 2


def pure_pursuit_seed(path_xy: np.ndarray, pose: np.ndarray, p: abi.SmpcParams):
    """Vectorised restatement of PathTrajectorizer::trajectorize (diff-drive branch),
    reference src/path_trajectorizer.cpp:120-288. path_xy [B][N][2], pose [B][3].
    Returns poses [B][max_steps+1][3], cmds [B][max_steps][2]. The seed is integrated with the
    double time_step (SURVEY Q15). Early goal stop (goal_dist <= 0.2) is not modelled: callers
    place the goal farther than the horizon."""
    B = pose.shape[0]
    dt = round(float(p.time_step), 6)  # the trajectorizer holds time_step as the yaml DOUBLE (0.05), not 0.05f
    max_steps = int(round(float(p.max_time) / float(p.time_step)))
    L = float(p.lookahead_dist)
    v_des = float(p.traj_desired_linear_vel)
    w_max = float(p.max_angular_vel)
    rx, ry, rth = pose[:, 0].copy(), pose[:, 1].copy(), yaw_roundtrip(pose[:, 2])
    poses = np.empty((B, max_steps + 1, 3))
    cmds = np.empty((B, max_steps, 2))
    poses[:, 0, 0], poses[:, 0, 1], poses[:, 0, 2] = rx, ry, rth
    N = path_xy.shape[1]
    rev = np.arange(N)[::-1]
    for s in range(max_steps):
        d = np.sqrt((rx[:, None] - path_xy[:, :, 0]) ** 2 + (ry[:, None] - path_xy[:, :, 1]) ** 2)
        within = d <= L
        any_within = within.any(axis=1)
        last_within = N - 1 - np.argmax(within[:, ::-1], axis=1)
        nearest = rev[np.argmin(d[:, ::-1], axis=1)]
        wp = np.where(any_within, last_within, nearest)
        wpx = path_xy[np.arange(B), wp, 0]
        wpy = path_xy[np.arange(B), wp, 1]
        dx = (wpx - rx) * np.cos(rth) + (wpy - ry) * np.sin(rth)
        dy = -(wpx - rx) * np.sin(rth) + (wpy - ry) * np.cos(rth)
        dth = np.arctan2(dy, dx)
        d2 = dx * dx + dy * dy
        curv = np.where(d2 > 0.001, 2.0 * dy / np.where(d2 > 0.001, d2, 1.0), 0.0)
        rotate = np.abs(dth) > math.pi / 2.0
        vx = np.where(rotate, 0.0, v_des)
        wz = np.where(rotate, w_max * np.where(dth > 0, 1.0, -1.0), v_des * curv)
        rx = rx + (vx * np.cos(rth) + 0.0 * np.cos(math.pi / 2 + rth)) * dt
        ry = ry + (vx * np.sin(rth) + 0.0 * np.sin(math.pi / 2 + rth)) * dt
        rth = rth + wz * dt
        poses[:, s + 1, 0], poses[:, s + 1, 1], poses[:, s + 1, 2] = rx, ry, yaw_roundtrip(rth)
        cmds[:, s, 0], cmds[:, s, 1] = vx, wz
    return poses, cmds


def format_seed(poses: np.ndarray, cmds: np.ndarray, speed: np.ndarray, p: abi.SmpcParams,
                prev_poses: np.ndarray | None = None, prev_cmds: np.ndarray | None = None):
    """Restatement of Optimizer::format_to_optimize + the unpacking at reference src/optimizer.cpp:197-237,
    484-551 for a first call (previous == current when no memory is given).
    Returns dict(pose0 [B][3], u0 [B][NB][2], path_xy [B][2][S+1], goal_yaw [B]) and S."""
    B = poses.shape[0]
    maxsize = int(round(float(p.max_time) / float(p.time_step)))
    if poses.shape[1] > maxsize:
        poses = poses[:, : maxsize - 1]
    Pn = poses.shape[1]
    if prev_poses is None:
        prev_poses, prev_cmds = poses, cmds
    wpath = float(p.current_path_w)
    wcmd = float(p.current_cmds_w)
    n_prev = min(Pn, prev_poses.shape[1])
    robot = np.empty((B, Pn, 6))
    x = poses[:, :, 0].copy()
    y = poses[:, :, 1].copy()
    yaw = poses[:, :, 2].copy()
    x[:, :n_prev] = wpath * poses[:, :n_prev, 0] + (1.0 - wpath) * prev_poses[:, :n_prev, 0]
    y[:, :n_prev] = wpath * poses[:, :n_prev, 1] + (1.0 - wpath) * prev_poses[:, :n_prev, 1]
    yaw[:, :n_prev] = yaw_roundtrip(wpath * poses[:, :n_prev, 2] + (1.0 - wpath) * prev_poses[:, :n_prev, 2])
    robot[:, :, 0], robot[:, :, 1], robot[:, :, 2] = x, y, yaw
    robot[:, :, 3] = np.arange(Pn)[None, :] * f32(p.time_step)
    robot[:, 0, 4], robot[:, 0, 5] = speed[:, 0], speed[:, 1]
    # SURVEY Q11: previous_cmds[i-1] is read unguarded in the reference; missing entries fall back to the current cmd.
    pc = cmds[:, : Pn - 1].copy()
    k = min(Pn - 1, prev_cmds.shape[1])
    pc[:, :k] = prev_cmds[:, :k]
    robot[:, 1:, 4] = wcmd * cmds[:, : Pn - 1, 0] + (1.0 - wcmd) * pc[:, :, 0]
    robot[:, 1:, 5] = wcmd * cmds[:, : Pn - 1, 1] + (1.0 - wcmd) * pc[:, :, 1]
    S = Pn - 1
    ch, bl, nb, _ = abi.problem_dims(p.control_horizon, p.parameter_block_length, S)
    out = dict(
        pose0=np.ascontiguousarray(robot[:, 0, :3]),
        u0=np.ascontiguousarray(robot[:, :nb, 4:6]),  # block b starts at the seed velocity of time index b (Q1)
        path_xy=np.ascontiguousarray(np.stack([robot[:, :, 0], robot[:, :, 1]], axis=1)),
        goal_yaw=np.ascontiguousarray(robot[:, -1, 2]),
    )
    return out, S, robot


@dataclasses.dataclass
class Batch:
    """Host-side batch in the include/smpc.h layout."""
    params: abi.SmpcParams
    n_problems: int
    n_steps: int
    n_agents: int
    n_costmaps: int
    size_x: int
    size_y: int
    resolution: float
    dt: float
    arrays: dict

    @property
    def dims(self):
        return abi.problem_dims(self.params.control_horizon, self.params.parameter_block_length, self.n_steps)

    @property
    def n_blocks(self) -> int:
        return self.dims[2]

    @property
    def dof(self) -> int:
        """Parameters per block: 2 = (v, w); 3 = (vx, vy, w) when params.omni_solve is set (extension)."""
        return 3 if int(self.params.omni_solve) else 2

    def struct(self, arrays: dict | None = None) -> abi.SmpcBatch:
        return abi.make_batch_struct(arrays if arrays is not None else self.arrays, self.n_problems, self.n_steps,
                                     self.n_agents, self.n_costmaps, self.size_x, self.size_y, self.resolution,
                                     self.dt)

    def slice(self, lo: int, hi: int) -> "Batch":
        """Problems [lo, hi) as a new batch (costmaps are shared, indices kept)."""
        arr = {}
        shared = self.arrays.get("scenario_index") is not None  # per-scene arrays stay whole
        for k, v in self.arrays.items():
            if v is None:
                arr[k] = None
            elif k in ("costmaps", "costmap_origin") or (shared and k in abi.SCENE_FIELDS):
                arr[k] = v
            else:
                arr[k] = np.ascontiguousarray(v[lo:hi])
        if arr.get("costmap_index") is None and not shared:
            arr["costmap_index"] = (np.arange(lo, hi) % self.n_costmaps).astype(np.int32)
        return dataclasses.replace(self, n_problems=hi - lo, arrays=arr)

    def expanded(self) -> "Batch":
        """A scenario-sharing batch written out with one row per problem (what the oracle and older callers read)."""
        idx = self.arrays.get("scenario_index")
        if idx is None:
            return self
        arr = {}
        for k, v in self.arrays.items():
            if k == "scenario_index":
                continue
            arr[k] = np.ascontiguousarray(v[idx]) if (v is not None and k in abi.SCENE_FIELDS) else v
        if arr.get("costmap_index") is None:
            arr["costmap_index"] = (idx % self.n_costmaps).astype(np.int32)
        return dataclasses.replace(self, arrays=arr)

    def input_bytes(self) -> int:
        return int(sum(v.nbytes for v in self.arrays.values() if v is not None))

    def algorithmic_bytes_per_problem(self, unique_costmap: bool) -> int:
        """SURVEY §8d: 8*[3 + P + 2(S+1) + 1 + 6A(S+1)] + map + outputs 8*[P + 2(S+1) + 2] + 12."""
        S, A, P = self.n_steps, self.n_agents, self.dof * self.n_blocks
        inp = 8 * (3 + P + 2 * (S + 1) + 1 + 6 * A * (S + 1))
        outp = 8 * (P + 2 * (S + 1) + 2) + 12
        return inp + outp + (self.size_x * self.size_y if unique_costmap else 0)


def _rng(config_id: int) -> np.random.Generator:
    return np.random.Generator(np.random.Philox(SEED_BASE + config_id))


def wall_costmap(size_x: int, size_y: int, res: float, walls_y, boxes=(), decay: float = 3.0) -> np.ndarray:
    """Inflation-like field 252*exp(-decay*d) around horizontal walls and axis-aligned boxes, u8 [size_y][size_x].
    Cell (row, col) holds the cost at world (col*res, row*res) (no half-cell offset, SURVEY Q8)."""
    ys = np.arange(size_y)[:, None] * res
    xs = np.arange(size_x)[None, :] * res
    d = np.full((size_y, size_x), np.inf)
    for wy in walls_y:
        d = np.minimum(d, np.abs(ys - wy) + 0.0 * xs)
    for (bx, by, hw, hh) in boxes:
        dx = np.maximum(np.abs(xs - bx) - hw, 0.0)
        dy = np.maximum(np.abs(ys - by) - hh, 0.0)
        d = np.minimum(d, np.sqrt(dx * dx + dy * dy))
    return np.clip(np.floor(252.0 * np.exp(-decay * d)), 0, 254).astype(np.uint8)


def _straight_path(B: int, x0, y0, length: float = 3.0, step: float = 0.05) -> np.ndarray:
    n = int(round(length / step)) + 1
    s = np.arange(n) * step
    path = np.empty((B, n, 2))
    path[:, :, 0] = np.asarray(x0)[:, None] + s[None, :]
    path[:, :, 1] = np.asarray(y0)[:, None]
    return path


def _cv_agents(rng, B: int, A: int, S: int, dt: float, pos, heading, speed, valid=None) -> np.ndarray:
    """Constant-velocity people projection, layout [B][A][6][S+1] (x, y, yaw, t, lv, av)."""
    ag = np.zeros((B, A, 6, S + 1))
    t = np.arange(S + 1)[None, None, :] * dt
    ag[:, :, 0, :] = pos[:, :, 0, None] + speed[:, :, None] * np.cos(heading)[:, :, None] * t
    ag[:, :, 1, :] = pos[:, :, 1, None] + speed[:, :, None] * np.sin(heading)[:, :, None] * t
    ag[:, :, 2, :] = heading[:, :, None]
    ag[:, :, 3, :] = t
    ag[:, :, 4, :] = speed[:, :, None]
    if valid is not None:
        inv = ~valid
        ag[inv] = 0.0
        ag[inv, 3, :] = -1.0  # padded agent (0,0,0,-1,0,0), reference src/optimizer.cpp:468-474
    return ag


def _finish(p, seed, S, agents, has_people, costmaps, origin, cmap_index, res) -> Batch:
    B = seed["pose0"].shape[0]
    A = 0 if agents is None else agents.shape[1]
    arrays = dict(seed)
    arrays["agents"] = None if agents is None else np.ascontiguousarray(agents, dtype=np.float64)
    arrays["has_people"] = np.ascontiguousarray(has_people, dtype=np.uint8)
    arrays["costmaps"] = np.ascontiguousarray(costmaps, dtype=np.uint8)
    arrays["costmap_origin"] = np.ascontiguousarray(origin, dtype=np.float64)
    arrays["costmap_index"] = None if cmap_index is None else np.ascontiguousarray(cmap_index, dtype=np.int32)
    return Batch(params=p, n_problems=B, n_steps=S, n_agents=A, n_costmaps=costmaps.shape[0],
                 size_x=costmaps.shape[2], size_y=costmaps.shape[1], resolution=res, dt=f32(p.time_step),
                 arrays=arrays)


def single(param_set: str = "readme", n_people: int = 3, n_agent_cols: int | None = None, seed_offset: int = 0,
           **overrides) -> Batch:
    """BASELINE config 1: one solve, robot at (2,2,0), straight +x path, people walking toward the robot,
    two walls at y=0.6 / y=3.4 (SURVEY §8d-1)."""
    p = make_params(param_set, **overrides)
    rng = _rng(1 + seed_offset)
    res, n = 0.05, 80
    pose = np.array([[2.0, 2.0, 0.0]])
    path = _straight_path(1, pose[:, 0], pose[:, 1])
    poses, cmds = pure_pursuit_seed(path, pose, p)
    seed, S, _ = format_seed(poses, cmds, np.array([[0.3, 0.0]]), p)
    A = n_agent_cols if n_agent_cols is not None else max(3, n_people)
    r = rng.uniform(0.8, 1.8, size=(1, A))
    bearing = rng.uniform(-math.pi / 4, math.pi / 4, size=(1, A))
    pos = np.stack([pose[:, 0, None] + r * np.cos(bearing), pose[:, 1, None] + r * np.sin(bearing)], axis=-1)
    heading = np.arctan2(pose[:, 1, None] - pos[:, :, 1], pose[:, 0, None] - pos[:, :, 0]) + rng.uniform(-0.3, 0.3, (1, A))
    speed = np.full((1, A), 0.5)
    valid = np.zeros((1, A), dtype=bool)
    valid[:, :n_people] = True
    agents = _cv_agents(rng, 1, A, S, f32(p.time_step), pos, heading, speed, valid)
    cm = wall_costmap(n, n, res, walls_y=(0.6, 3.4))[None]
    return _finish(p, seed, S, agents, np.array([1 if n_people > 0 else 0]), cm, np.zeros((1, 2)), None, res)


def corridor(B: int = 4096, param_set: str = "obst_only", config_id: int = 2, unique_maps: bool = True,
             **overrides) -> Batch:
    """BASELINE config 2: obstacle-grid + path critics only, synthetic corridor scenarios (SURVEY §8d-2):
    corridor width U[1.2,2.5], one box obstacle on the path, start lateral offset U[-0.3,0.3], yaw U[-0.5,0.5],
    one costmap per problem."""
    p = make_params(param_set, **overrides)
    rng = _rng(config_id)
    res, n = 0.05, 80
    width = rng.uniform(1.2, 2.5, B)
    box_x = rng.uniform(1.0, 2.2, B) + 0.6
    box_y = 2.0 + rng.uniform(-0.25, 0.25, B)
    box_h = rng.uniform(0.05, 0.15, (B, 2))
    lat = rng.uniform(-0.3, 0.3, B)
    yaw = rng.uniform(-0.5, 0.5, B)
    speed = np.stack([rng.uniform(0.0, 0.6, B), rng.uniform(-0.3, 0.3, B)], axis=1)
    pose = np.stack([np.full(B, 0.6), 2.0 + lat, yaw], axis=1)
    path = _straight_path(B, np.full(B, 0.6), np.full(B, 2.0))
    poses, cmds = pure_pursuit_seed(path, pose, p)
    seed, S, _ = format_seed(poses, cmds, speed, p)
    M = B if unique_maps else min(B, 256)
    cms = np.empty((M, n, n), dtype=np.uint8)
    for m in range(M):
        cms[m] = wall_costmap(n, n, res, walls_y=(2.0 - width[m] / 2, 2.0 + width[m] / 2),
                              boxes=((box_x[m], box_y[m], box_h[m, 0], box_h[m, 1]),))
    idx = (np.arange(B) % M).astype(np.int32)
    return _finish(p, seed, S, None, np.zeros(B), cms, np.zeros((M, 2)), idx, res)


def crowd(B: int = 65536, A: int = 20, param_set: str = "soc_work_obst", config_id: int = 3, n_maps: int = 256,
          n_valid: int | None = None, **overrides) -> Batch:
    """BASELINE config 3 / 5: full social + proxemics + obstacle critics, A agents uniform in the 4x4 m window with
    |p - robot| > 0.4, speeds U[0,1.2], headings U(-pi,pi], constant-velocity projection, `n_maps` costmaps shared
    round-robin (SURVEY §8d-3)."""
    p = make_params(param_set, **overrides)
    rng = _rng(config_id)
    res, n = 0.05, 80
    lat = rng.uniform(-0.3, 0.3, B)
    yaw = rng.uniform(-0.5, 0.5, B)
    speed = np.stack([rng.uniform(0.0, 0.6, B), rng.uniform(-0.3, 0.3, B)], axis=1)
    pose = np.stack([np.full(B, 0.8), 2.0 + lat, yaw], axis=1)
    path = _straight_path(B, np.full(B, 0.8), np.full(B, 2.0))
    poses, cmds = pure_pursuit_seed(path, pose, p)
    seed, S, _ = format_seed(poses, cmds, speed, p)
    pos = rng.uniform(0.2, 3.8, (B, A, 2))
    for _ in range(8):  # re-draw agents that start within 0.4 m of the robot
        near = np.hypot(pos[:, :, 0] - pose[:, None, 0], pos[:, :, 1] - pose[:, None, 1]) <= 0.4
        if not near.any():
            break
        pos[near] = rng.uniform(0.2, 3.8, (int(near.sum()), 2))
    heading = rng.uniform(-math.pi, math.pi, (B, A))
    spd = rng.uniform(0.0, 1.2, (B, A))
    valid = None
    if n_valid is not None:
        valid = np.zeros((B, A), dtype=bool)
        valid[:, :n_valid] = True
    agents = _cv_agents(rng, B, A, S, f32(p.time_step), pos, heading, spd, valid)
    M = min(n_maps, B)
    width = rng.uniform(2.0, 3.2, M)
    bx = rng.uniform(1.6, 3.2, M)
    by = 2.0 + rng.uniform(-0.6, 0.6, M)
    cms = np.empty((M, n, n), dtype=np.uint8)
    for m in range(M):
        cms[m] = wall_costmap(n, n, res, walls_y=(2.0 - width[m] / 2, 2.0 + width[m] / 2),
                              boxes=((bx[m], by[m], 0.1, 0.1),))
    idx = (np.arange(B) % M).astype(np.int32)
    return _finish(p, seed, S, agents, np.ones(B), cms, np.zeros((M, 2)), idx, res)


EPISODE_MARGIN = 0.8  # m between a person's constant-velocity track and the edge of the obstacle grid


def episodes(B: int, K: int, param_set: str = "soc_work_obst", seed: int = 6, ticks: int = 200,
             control_period: float = 0.05, n_maps: int = 16, path_length: float = 10.0, **overrides) -> dict:
    """Closed-loop scenes for FleetOptimizer.run_episodes: a 12 m x 4 m corridor at 0.05 m (walls at y = 0.3 / 3.7,
    lethal beyond them, one lethal box near a wall per costmap, `n_maps` costmaps shared round-robin), an
    obstacle-distance grid to the walls over the whole corridor, a straight global path of `path_length` m along
    y = 2 from x = 1, start poses near its first pose. K people per scene, half oncoming, half crossing diagonally, at
    0.3-1.2 m/s. Their constant-velocity tracks stay EPISODE_MARGIN inside the obstacle grid for the whole run plus one
    projection horizon (ticks * control_period + max_time): a person who leaves the grid makes the reference's
    computeObstacle throw (project_status), and the crowd projection may move a person up to 0.75 m off its track.
    Speeds are drawn up to what fits the corridor for the run. Returns the keyword arguments of
    run_episodes plus `params`."""
    p = make_params(param_set, **overrides)
    rng = _rng(500 + seed)
    res, W, H = 0.05, 240, 80
    wall_lo, wall_hi = 0.3, 3.7
    horizon = ticks * control_period + f32(p.max_time)
    M = max(1, min(n_maps, B))
    ys = np.arange(H)[:, None] * res
    xs = np.arange(W)[None, :] * res
    cms = np.empty((M, H, W), dtype=np.uint8)
    for m in range(M):
        side = 1.0 if m % 2 else -1.0
        bx, by = rng.uniform(3.0, 9.0), 2.0 + side * rng.uniform(0.9, 1.2)
        cm = wall_costmap(W, H, res, walls_y=(wall_lo, wall_hi), boxes=((bx, by, 0.15, 0.15),))
        lethal = (ys <= wall_lo) | (ys >= wall_hi) | ((np.abs(xs - bx) <= 0.15) & (np.abs(ys - by) <= 0.15))
        cm[np.broadcast_to(lethal, cm.shape)] = 254
        cms[m] = cm
    rows = np.arange(H)[:, None] * np.ones((1, W), dtype=int)
    cols = np.ones((H, 1), dtype=int) * np.arange(W)[None, :]
    r_lo, r_hi = int(round(wall_lo / res)), int(round(wall_hi / res))
    near = np.where(np.abs(rows - r_lo) <= np.abs(rows - r_hi), r_lo, r_hi)
    od = dict(width=W, height=H, resolution=res, origins=np.zeros((1, 2)),
              indexes=(near * W + cols).astype(np.uint32).ravel())

    pose = np.stack([np.full(B, 1.0), 2.0 + rng.uniform(-0.2, 0.2, B), rng.uniform(-0.3, 0.3, B)], axis=1)
    gpath = _straight_path(B, np.full(B, 1.0), np.full(B, 2.0), length=path_length)
    speed = np.stack([rng.uniform(0.0, 0.4, B), np.zeros(B)], axis=1)

    lo = np.array([EPISODE_MARGIN, EPISODE_MARGIN])
    hi = np.array([W * res - EPISODE_MARGIN, H * res - EPISODE_MARGIN])
    people = np.zeros((B, K, 5))
    if K > 0:
        oncoming = (np.arange(K) % 2 == 0)[None, :].repeat(B, axis=0)
        heading = np.empty((B, K))
        v = np.empty((B, K))
        todo = np.ones((B, K), dtype=bool)
        for _ in range(64):  # draw headings until the slowest allowed speed fits the corridor
            n = int(todo.sum())
            if n == 0:
                break
            onc = oncoming[todo]
            off = np.where(onc, rng.uniform(-0.15, 0.15, n), rng.choice([-1.0, 1.0], n) * rng.uniform(0.25, 0.6, n))
            base = np.where(onc, math.pi, rng.choice([0.0, math.pi], n))
            h = base + off
            vmax = np.minimum((hi[0] - lo[0]) / (horizon * np.maximum(np.abs(np.cos(h)), 1e-9)),
                              (hi[1] - lo[1]) / (horizon * np.maximum(np.abs(np.sin(h)), 1e-9)))
            ok = vmax >= 0.3
            vv = 0.3 + (np.minimum(vmax, 1.2) - 0.3) * rng.uniform(0.0, 1.0, n)
            idx = np.argwhere(todo)[ok]
            heading[idx[:, 0], idx[:, 1]] = h[ok]
            v[idx[:, 0], idx[:, 1]] = vv[ok]
            todo[idx[:, 0], idx[:, 1]] = False
        assert not todo.any(), "corridor too short for the requested number of ticks"
        vel = np.stack([v * np.cos(heading), v * np.sin(heading)], axis=-1)
        ext = vel * horizon  # displacement over the run
        start_lo = lo - np.minimum(ext, 0.0)
        start_hi = hi - np.maximum(ext, 0.0)
        pos = start_lo + (start_hi - start_lo) * rng.uniform(0.0, 1.0, (B, K, 2))
        for _ in range(16):  # nobody starts within 0.6 m of the robot
            close = np.hypot(pos[..., 0] - pose[:, None, 0], pos[..., 1] - pose[:, None, 1]) < 0.6
            if not close.any():
                break
            u = rng.uniform(0.0, 1.0, (int(close.sum()), 2))
            pos[close] = start_lo[close] + (start_hi[close] - start_lo[close]) * u
        people[:, :, 0:2] = pos
        people[:, :, 2:4] = vel
    return dict(params=p, global_path=gpath, pose=pose, speed=speed, people=people,
                n_people=np.full(B, K, dtype=np.int32), costmaps=cms, costmap_origin=np.zeros((M, 2)),
                costmap_resolution=res, od=od, costmap_index=(np.arange(B) % M).astype(np.int32), ticks=ticks,
                control_period=control_period)


CROWD_SPACING = 0.7    # m between two people's starts
CROWD_CLEARANCE = 0.6  # m between a start and the robot, and between a start and any lethal cell
GOAL_BAND = 3.0  # m of corridor at each end that holds the goals of the walkers along it (denser crowds push each other
                 # past their goals and out of the corridor's open ends)


def _lethal_clearance_ok(costmaps, res: float, clearance: float) -> np.ndarray:
    """[M][H][W] bool: no lethal cell centre lies within `clearance` m of any point of this cell."""
    M, H, W = costmaps.shape
    lethal = costmaps >= 253
    r = clearance + res * math.sqrt(0.5)  # the farthest point of a cell is half a diagonal from its centre
    n = int(math.ceil(r / res))
    near = np.zeros_like(lethal)
    pad = np.pad(lethal, ((0, 0), (n, n), (n, n)))
    for dy in range(-n, n + 1):
        for dx in range(-n, n + 1):
            if dx * dx + dy * dy <= (r / res) ** 2:
                near |= pad[:, n + dy: n + dy + H, n + dx: n + dx + W]
    return ~near


def crowd_episodes(B: int, K: int, seed: int = 6, ticks: int = 200, substeps: int = 1,
                   param_set: str = "soc_work_obst", **kw) -> dict:
    """Closed-loop scenes with a reactive crowd for FleetOptimizer.run_crowd_episodes: the corridors, costmaps, paths
    and start poses of episodes(B, 0, ...) and K people per scene who walk to goals of their own. People i % 3 == 0
    walk toward the robot (goals near the robot's start end), i % 3 == 1 walk the robot's way (goals at the far end),
    i % 3 == 2 cross the corridor (goals on the other side, 0.8-1.0 m from its centre line). Desired speeds are
    0.3-1.2 m/s and every person starts at its desired speed toward its goal. Starts keep CROWD_CLEARANCE from the
    robot's start and from every lethal cell and CROWD_SPACING from each other. Goals keep EPISODE_MARGIN + 0.5 m/s *
    max_time from the ends of the obstacle-distance grid: 0.5 m/s caps the controller's projection of a person, so a
    projected person never leaves the grid. Returns the keyword arguments of run_crowd_episodes plus `params` and
    `ticks`."""
    s = episodes(B, 0, param_set=param_set, seed=seed, ticks=ticks, **kw)
    people, goal, vdes = _place_crowd(s, K, seed, s["pose"][:, None, :2])
    s.update(people=people, n_people=np.full(B, K, dtype=np.int32), goals=goal, desired_speed=vdes,
             substeps=substeps)
    return s


EPISODE_ROWS = ("global_path", "pose", "speed", "people", "n_people", "costmap_index", "goals", "desired_speed")


def tile_scenes(s: dict, P: int) -> dict:
    """The one-robot scenes of episodes / crowd_episodes repeated P times: episode p * B0 + i is scene i. The maps stay
    shared and costmap_index is tiled, so every copy keeps its scene's map. With per-episode critic weights
    (weights=(table, np.repeat(np.arange(P), B0))) copy p runs under row p: P tunings on the same scenes in one call."""
    t = dict(s)
    for k in EPISODE_ROWS:
        if k in s:
            t[k] = np.concatenate([np.asarray(s[k])] * P)
    return t


def _place_crowd(s: dict, K: int, seed: int, robots: np.ndarray):
    """The people of crowd_episodes for the scenes of s (episodes(B, 0, ...)): starts keep CROWD_CLEARANCE from every
    robot start robots [B][R][2] and from lethal cells. Returns people [B][K][5], goals [B][K][2], desired speeds."""
    B = robots.shape[0]
    p = s["params"]
    rng = _rng(900 + seed)
    od, res = s["od"], s["costmap_resolution"]
    W, H = int(od["width"]), int(od["height"])
    x_lo = EPISODE_MARGIN + 0.5 * f32(p.max_time)
    x_hi = W * od["resolution"] - x_lo
    y_mid = 2.0
    kind = np.arange(K) % 3
    onc, same, cross = kind == 0, kind == 1, kind == 2
    clear_ok = _lethal_clearance_ok(s["costmaps"], res, CROWD_CLEARANCE)
    cidx = s["costmap_index"]

    def draw(n):
        """starts [n][K][2] and goals [n][K][2] of n scenes"""
        start = np.empty((n, K, 2))
        goal = np.empty((n, K, 2))
        u = lambda lo, hi: rng.uniform(lo, hi, (n, K))  # noqa: E731
        start[..., 0] = np.where(onc, u(x_lo + GOAL_BAND + 1.0, x_hi), np.where(same, u(x_lo, x_hi - GOAL_BAND - 1.0),
                                                                                 u(2.5, x_hi - 0.5)))
        side = rng.choice([-1.0, 1.0], (n, K))
        start[..., 1] = np.where(cross, y_mid + side * u(0.8, 1.0), u(y_mid - 1.0, y_mid + 1.0))
        goal[..., 0] = np.where(onc, u(x_lo, x_lo + GOAL_BAND), np.where(same, u(x_hi - GOAL_BAND, x_hi),
                                                                            np.clip(start[..., 0] + u(-1.0, 1.0), x_lo,
                                                                                    x_hi)))
        goal[..., 1] = np.where(cross, y_mid - side * u(0.8, 1.0), u(y_mid - 1.0, y_mid + 1.0))
        return start, goal

    start, goal = draw(B)
    todo = np.arange(B) if K > 0 else np.arange(0)
    for it in range(2000):  # redraw the people who break a rule; only scenes with such people are looked at again
        st = start[todo]
        mx = np.clip((st[..., 0] / res).astype(np.int64), 0, W - 1)
        my = np.clip((st[..., 1] / res).astype(np.int64), 0, H - 1)
        bad = ~clear_ok[cidx[todo][:, None], my, mx]
        rs = robots[todo]
        bad |= np.hypot(st[:, :, None, 0] - rs[:, None, :, 0], st[:, :, None, 1] - rs[:, None, :, 1]).min(
            axis=2, initial=np.inf) < CROWD_CLEARANCE
        d = np.hypot(st[:, :, None, 0] - st[:, None, :, 0], st[:, :, None, 1] - st[:, None, :, 1])
        d[:, np.tril_indices(K)[0], np.tril_indices(K)[1]] = np.inf  # each pair once: the later person moves
        bad |= (d < CROWD_SPACING).any(axis=1)
        keep = bad.any(axis=1)
        todo, bad = todo[keep], bad[keep]
        if todo.size == 0:
            break
        if it % 50 == 49:  # a scene still stuck after 50 rounds: draw all of its people again
            bad[:] = True
        s2, g2 = draw(todo.size)
        st, gl = start[todo], goal[todo]
        st[bad], gl[bad] = s2[bad], g2[bad]
        start[todo], goal[todo] = st, gl
    else:
        raise AssertionError("could not place the crowd: fewer people or a longer corridor")
    vdes = rng.uniform(0.3, 1.2, (B, K))
    dg = goal - start
    heading = dg / np.linalg.norm(dg, axis=-1, keepdims=True) if K > 0 else dg
    people = np.zeros((B, K, 5))
    people[..., 0:2] = start
    people[..., 2:4] = heading * vdes[..., None]
    return people, goal, vdes


SHARED_STAGGER = 1.5  # m between the starts (and the goals) of two robots of a scene going the same way
SHARED_SPACING = 1.0  # m between any two robot starts of a scene
SHARED_LATERAL = 0.3  # m: robot lanes lie within this distance of the corridor's centre line y = 2


def shared_episodes(S: int, R: int, K: int, seed: int = 6, ticks: int = 200, substeps: int = 1,
                    param_set: str = "soc_work_obst", **kw) -> dict:
    """Shared scenes for FleetOptimizer.run_shared_episodes: the corridors of crowd_episodes(S, K, ...), each with R
    robots (robot r of scene c is robot c * R + r) and one crowd of K people. Even robots drive +x, odd robots -x, so
    they meet head-on. Each robot follows a straight path along its own lane y = 2 + u, |u| <= SHARED_LATERAL; robots
    going the same way start (and end) SHARED_STAGGER apart along x, any two starts are at least SHARED_SPACING apart
    and keep CROWD_CLEARANCE from lethal cells, and every path endpoint keeps EPISODE_MARGIN + 0.5 m/s * max_time from
    the ends of the obstacle grid: the other robots enter a robot's controller as people, and a projected person must
    not leave the grid. The people are placed as in crowd_episodes, clear of every robot start. Returns the keyword
    arguments of run_shared_episodes (per robot: global_path, pose, speed, costmap_index; per scene: people, n_people,
    goals, desired_speed) plus `params` and `ticks`. Raises ValueError when R robots do not fit the corridor."""
    s = episodes(S, 0, param_set=param_set, seed=seed, ticks=ticks, **kw)
    p = s["params"]
    rng = _rng(1300 + seed)
    od, res = s["od"], s["costmap_resolution"]
    x_lo = EPISODE_MARGIN + 0.5 * f32(p.max_time)
    x_hi = int(od["width"]) * od["resolution"] - x_lo
    r = np.arange(R)
    fwd = r % 2 == 0
    n_fwd = (R + 1) // 2
    length = x_hi - x_lo - SHARED_STAGGER * (n_fwd - 1)
    x0 = np.where(fwd, x_lo + SHARED_STAGGER * (r // 2), x_hi - SHARED_STAGGER * (r // 2))
    dx = np.abs(x0[:, None] - x0[None, :]) + np.where(np.eye(R, dtype=bool), np.inf, 0.0)
    if R > 1 and (length < 1.0 or np.any(dx * dx + (2 * SHARED_LATERAL) ** 2 < SHARED_SPACING ** 2)):
        raise ValueError(f"{R} robots per scene do not fit the corridor")
    clear_ok = _lethal_clearance_ok(s["costmaps"], res, CROWD_CLEARANCE)
    H, W = s["costmaps"].shape[1:]
    cidx = s["costmap_index"]
    mx = np.clip((x0 / res).astype(np.int64), 0, W - 1)
    y = np.empty((S, R))
    todo = np.arange(S)
    for _ in range(400):  # redraw the lanes of scenes whose starts are too close or near a lethal cell
        y[todo] = 2.0 + rng.uniform(-SHARED_LATERAL, SHARED_LATERAL, (todo.size, R))
        yt = y[todo]
        my = np.clip((yt / res).astype(np.int64), 0, H - 1)
        bad = ~clear_ok[cidx[todo][:, None], my, mx[None, :]].all(axis=1)
        d = np.hypot(dx[None], yt[:, :, None] - yt[:, None, :])
        bad |= (d < SHARED_SPACING).any(axis=(1, 2))
        todo = todo[bad]
        if todo.size == 0:
            break
    else:
        raise AssertionError("could not place the robots of a scene")
    direction = np.where(fwd, 1.0, -1.0)
    N = int(round(length / 0.05)) + 1
    gpath = np.empty((S, R, N, 2))
    gpath[..., 0] = x0[None, :, None] + direction[None, :, None] * np.linspace(0.0, length, N)[None, None, :]
    gpath[..., 1] = y[:, :, None]
    yaw = np.where(fwd, 0.0, math.pi)[None, :] + rng.uniform(-0.2, 0.2, (S, R))
    pose = np.stack([np.broadcast_to(x0, (S, R)), y, yaw], axis=-1)
    speed = np.stack([rng.uniform(0.0, 0.4, (S, R)), np.zeros((S, R))], axis=-1)
    people, goal, vdes = _place_crowd(s, K, seed, pose[..., :2])
    s.update(global_path=gpath.reshape(S * R, N, 2), pose=pose.reshape(S * R, 3), speed=speed.reshape(S * R, 2),
             costmap_index=np.repeat(cidx, R).astype(np.int32), people=people,
             n_people=np.full(S, K, dtype=np.int32), goals=goal, desired_speed=vdes, substeps=substeps,
             robots_per_scene=R)
    return s


def with_horizons(batch: Batch, n_steps_each) -> Batch:
    """The same batch with per-problem horizons S_b <= n_steps (include/smpc.h n_steps_each): robots near their goal get
    a shorter seed from the trajectorizer (reference src/path_trajectorizer.cpp:152) and with it fewer steps, a shorter
    control horizon and fewer parameter blocks (src/optimizer.cpp:248-249). Arrays keep the stride of n_steps."""
    n = np.ascontiguousarray(n_steps_each, dtype=np.int32).reshape(batch.n_problems)
    assert n.min() >= 1 and n.max() <= batch.n_steps
    arr = dict(batch.arrays)
    arr["n_steps_each"] = n
    return dataclasses.replace(batch, arrays=arr)


def omni(batch: Batch, vy_sigma: float = 0.05, config_id: int = 70) -> Batch:
    """The same scenarios for the OMNIDIRECTIONAL solve (extension, BASELINE configs[4]): blocks become (vx, vy, w); the
    unicycle seed gives vx and w, the lateral start velocity is a small random value so that the vy coordinates are
    exercised from the first iteration. The reference has no omnidirectional solve (only its trajectorizer has an omni
    branch), so these batches are checked against this repo's own oracle functors only."""
    rng = _rng(config_id)
    p = abi.SmpcParams.from_buffer_copy(bytes(batch.params))
    p.omni_solve = 1
    u0 = batch.arrays["u0"]
    B, nb, _ = u0.shape
    u3 = np.zeros((B, nb, 3))
    u3[:, :, 0], u3[:, :, 2] = u0[:, :, 0], u0[:, :, 1]
    u3[:, :, 1] = rng.normal(0.0, vy_sigma, (B, nb))
    arr = dict(batch.arrays)
    arr["u0"] = np.ascontiguousarray(u3)
    return dataclasses.replace(batch, params=p, arrays=arr)


def multistart(n_robots: int = 256, n_starts: int = 1024, config_id: int = 4, shared: bool = False, **overrides) -> Batch:
    """BASELINE config 4: `n_starts` perturbed initial control sequences per robot (start 0 unperturbed),
    u0 = clamp(seed u0 + N(0, diag(0.1, 0.3)^2)) per block (SURVEY §8d-4). Problems of one robot are contiguous.
    shared = True: the scene arrays keep ONE row per robot and `scenario_index` maps the starts onto them
    (smpc_batch.scenario_index); Batch.expanded() gives the same problems written out per start."""
    base = crowd(B=n_robots, A=3, config_id=config_id, n_maps=min(256, n_robots), **overrides)
    rng = _rng(config_id + 100)
    B = n_robots * n_starts
    arr = {}
    for k, v in base.arrays.items():
        if v is None or k in ("costmaps", "costmap_origin") or (shared and k in abi.SCENE_FIELDS):
            arr[k] = v
        else:
            arr[k] = np.ascontiguousarray(np.repeat(v, n_starts, axis=0))
    if shared:
        arr["u0"] = np.ascontiguousarray(np.repeat(base.arrays["u0"], n_starts, axis=0))
        arr["scenario_index"] = np.repeat(np.arange(n_robots, dtype=np.int32), n_starts)
        if arr.get("costmap_index") is None:
            arr["costmap_index"] = (np.arange(n_robots) % base.n_costmaps).astype(np.int32)
    nb = base.n_blocks
    noise = rng.normal(0.0, 1.0, (n_robots, n_starts, nb, 2)) * np.array([0.1, 0.3])
    noise[:, 0] = 0.0
    u0 = arr["u0"].reshape(n_robots, n_starts, nb, 2) + noise
    u0[..., 0] = np.clip(u0[..., 0], 0.0, 0.6)
    u0[..., 1] = np.clip(u0[..., 1], -1.4, 1.4)
    arr["u0"] = np.ascontiguousarray(u0.reshape(B, nb, 2))
    return dataclasses.replace(base, n_problems=B, arrays=arr)
