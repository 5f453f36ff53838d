"""Fleet tick on one GPU: the whole Optimizer::optimize pipeline (reference src/optimizer.cpp:148-452) for B robots
per call through ONE C-ABI call, smpc_optimize_batch — TrajectoryMemory seeding, people_to_status, format_to_optimize,
project_people (SFM), the bounded TR-LM solve with its post-solve expansion and the memory update are kernels of
libsmpc.so; the per-robot warm-start memory and the costmaps stay on the device between ticks. Robots may have
different path lengths (the trajectorizer stops early near the goal). This file only marshals numpy buffers; torch is
used by trajectorize_batch alone (device buffers for the seed-generation kernel)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib, abi
from .optimizer import Optimizer


def weight_sets_arg(weights, n_robots: int):
    """The smpc_weight_sets of the `weights=(table [P][9], set_index [B])` keyword, with the arrays it points to (keep
    them alive for the call). Raises ValueError on a shape or an index the table does not have."""
    table, set_index = weights
    table = np.ascontiguousarray(table, dtype=np.float64)
    set_index = np.asarray(set_index)
    if table.ndim != 2 or table.shape[1] != len(abi.WEIGHT_NAMES) or table.shape[0] < 1:
        raise ValueError(f"weights table must be [P][{len(abi.WEIGHT_NAMES)}] with P >= 1, got {table.shape}")
    if set_index.shape != (n_robots,) or not np.issubdtype(set_index.dtype, np.integer):
        raise ValueError(f"set_index must be {n_robots} integers, got {set_index.dtype} {set_index.shape}")
    if n_robots and (set_index.min() < 0 or set_index.max() >= table.shape[0]):
        raise ValueError(f"set_index outside 0..{table.shape[0] - 1}")
    set_index = np.ascontiguousarray(set_index, dtype=np.int32)
    return abi.SmpcWeightSets(table.shape[0], table.ctypes.data, set_index.ctypes.data), (table, set_index)


def perception_arg(perception, n_robots: int, ticks: int, n_rows: int, want_logs: bool):
    """The smpc_perception of the `perception=` keyword (an abi.SmpcPerception, or a dict of abi.perception_params
    overrides that may also hold `stream_index` [B]) with its outputs pointed at new arrays: (struct, outputs dict,
    arrays to keep alive for the call). n_rows = L, the rows of the perceived list."""
    if isinstance(perception, abi.SmpcPerception):
        pc = abi.SmpcPerception.from_buffer_copy(perception)
        stream_index = None
    else:
        over = dict(perception)
        stream_index = over.pop("stream_index", None)
        pc = abi.perception_params(**over)
    keep = []
    if stream_index is not None:
        stream_index = np.ascontiguousarray(stream_index, dtype=np.int32)
        if stream_index.shape != (n_robots,):
            raise ValueError(f"stream_index must be {n_robots} integers, got {stream_index.shape}")
        pc.stream_index = stream_index.ctypes.data
        keep.append(stream_index)
    out = dict(unseen_personal_ticks=np.zeros(n_robots, np.int32))
    if want_logs:
        out.update(seen_log=np.zeros((n_robots, ticks, n_rows, 5)), n_seen_log=np.zeros((n_robots, ticks), np.int32))
    for k, v in out.items():
        setattr(pc, k, v.ctypes.data)
    return pc, out, keep


def tracker_arg(tracker, pc, n_robots: int, ticks: int, n_rows: int, want_logs: bool):
    """The smpc_tracker of the `tracker=` keyword (an abi.SmpcTracker, or a dict of abi.tracker_params overrides) with
    its outputs pointed at new arrays: (struct, raw outputs dict). pc: the smpc_perception it follows, which must report
    positions only (vel_noise 0); n_rows = L, the rows of the perceived list."""
    if pc.vel_noise != 0.0:
        raise ValueError("tracker= estimates velocities from detected positions: the perception needs vel_noise=0, "
                         f"got {pc.vel_noise}")
    if isinstance(tracker, abi.SmpcTracker):
        tk = abi.SmpcTracker.from_buffer_copy(tracker)
    else:
        tk = abi.tracker_params(**dict(tracker))
    raw = dict(untracked_personal_ticks=np.zeros(n_robots, np.int32), track_rows=np.zeros(n_robots, np.int32),
               track_pos_err=np.zeros(n_robots), track_vel_err=np.zeros(n_robots))
    if want_logs:
        raw["track_id_log"] = np.full((n_robots, ticks, n_rows), -1, np.int32)
    for k, v in raw.items():
        setattr(tk, k, v.ctypes.data)
    return tk, raw


def tracker_results(raw) -> dict:
    """The result entries of a tracked run from tracker_arg's raw outputs: the summed errors become means over the
    people rows the FOV filter received (NaN for a robot that received none)."""
    rows = raw["track_rows"]
    out = dict(untracked_personal_ticks=raw["untracked_personal_ticks"], track_rows=rows)
    for name, key in (("mean_track_pos_error", "track_pos_err"), ("mean_track_vel_error", "track_vel_err")):
        out[name] = np.divide(raw[key], rows, out=np.full(rows.shape, np.nan), where=rows > 0)
    if "track_id_log" in raw:
        out["track_id_log"] = raw["track_id_log"]
    return out


def local_costmap_arg(local_costmap, n_robots: int, ticks: int, want_logs: bool):
    """The smpc_local_costmap of the `local_costmap=` keyword (an abi.SmpcLocalCostmap, or a dict of
    abi.local_costmap_params overrides) with its outputs pointed at new arrays: (struct, outputs dict). The logs hold
    one row per build, n_builds = ceil(ticks / update_period_ticks)."""
    if isinstance(local_costmap, abi.SmpcLocalCostmap):
        lc = abi.SmpcLocalCostmap.from_buffer_copy(local_costmap)
    else:
        lc = abi.local_costmap_params(**dict(local_costmap))
    out = dict(marked_rows=np.zeros(n_robots, np.int32))
    fields = dict(marked_rows="marked_rows")
    if want_logs:
        n_builds = -(-ticks // max(int(lc.update_period_ticks), 1))
        out.update(local_costmap_log=np.zeros((n_robots, n_builds, lc.size_y, lc.size_x), np.uint8),
                   local_origin_log=np.zeros((n_robots, n_builds, 2)))
        fields.update(local_costmap_log="costmap_log", local_origin_log="origin_log")
    for k, f in fields.items():
        setattr(lc, f, out[k].ctypes.data)
    return lc, out


def local_costmap_stencil(resolution: float, local_costmap=None) -> np.ndarray:
    """The inflation stencil smpc_run_local_costmap_episodes splats on a marked row at this resolution
    (smpc_local_costmap_stencil, no GPU): uint8 [2 hw + 1][2 hw + 1], row dy + hw, column dx + hw. local_costmap: as the
    keyword of run_episodes (None: the defaults). Raises SmpcError for what the episode entry rejects."""
    lc = local_costmap_arg({} if local_costmap is None else local_costmap, 0, 0, False)[0]
    L, hw = _lib.lib(), C.c_int(0)
    _lib.check(L.smpc_local_costmap_stencil(C.byref(lc), float(resolution), None, 0, C.byref(hw)))
    out = np.zeros((2 * hw.value + 1, 2 * hw.value + 1), np.uint8)
    _lib.check(L.smpc_local_costmap_stencil(C.byref(lc), float(resolution), out.ctypes.data, out.size, C.byref(hw)))
    return out


class FleetOptimizer:
    def __init__(self, params, n_robots: int, n_agents: int = 3, device: int = 0):
        self.device = device
        self.opt = Optimizer(device)
        self.opt.initialize(params)
        self.p = self.opt.params
        self.B, self.A = n_robots, n_agents
        self._maps_key = None
        self._maps_version = 0
        self._torch = None

    def close(self):
        self.opt.close()

    def reset_memory(self):
        """Forget every robot's previous path / cmds (fresh TrajectoryMemory)."""
        self.opt.reset_memory()

    @property
    def torch(self):
        if self._torch is None:
            import torch
            self._torch = torch
            self.dev = torch.device("cuda", self.device)
            self.stream = torch.cuda.Stream(device=self.dev)
        return self._torch

    def _t(self, a, dtype):
        return self.torch.as_tensor(np.ascontiguousarray(a, dtype=dtype)).to(self.dev)

    def trajectorize_batch(self, global_path, pose):
        """Batched PathTrajectorizer::trajectorize (reference src/path_trajectorizer.cpp:120-288) on the GPU.
        global_path [B][N][2], pose [B][3] -> poses [B][max_steps+1][3], cmds [B][max_steps][3], n_steps [B]."""
        torch, L, h, p = self.torch, _lib.lib(), self.opt._h, self.p
        gp = np.ascontiguousarray(global_path, dtype=np.float64)
        B, N, _ = gp.shape
        max_steps = int(round(float(p.max_time) / round(float(p.time_step), 6)))
        with torch.cuda.stream(self.stream):
            d_gp, d_pose = self._t(gp, np.float64), self._t(pose, np.float64)
            poses = torch.zeros(B, max_steps + 1, 3, dtype=torch.float64, device=self.dev)
            cmds = torch.zeros(B, max_steps, 3, dtype=torch.float64, device=self.dev)
            n_steps = torch.zeros(B, dtype=torch.int32, device=self.dev)
            a = abi.SmpcTrajectorizeArgs()
            a.n_problems, a.n_path, a.max_steps, a.omnidirectional = B, N, max_steps, int(p.omnidirectional)
            a.desired_linear_vel, a.lookahead_dist = p.traj_desired_linear_vel, p.lookahead_dist
            a.max_angular_vel, a.time_step = p.max_angular_vel, round(float(p.time_step), 6)
            a.global_path, a.path_index, a.pose = d_gp.data_ptr(), None, d_pose.data_ptr()
            a.poses, a.cmds, a.n_steps = poses.data_ptr(), cmds.data_ptr(), n_steps.data_ptr()
            _lib.check(L.smpc_trajectorize_batch_device(h, C.byref(a), self.stream.cuda_stream))
        self.stream.synchronize()
        return poses.cpu().numpy(), cmds.cpu().numpy(), n_steps.cpu().numpy()

    def filter_people_fov(self, people, n_people, pose, costmap_origin, size_x, size_y, resolution, fov_angle=None,
                          costmap_index=None, n_out_max=None):
        """FOV filter of SocialMPCController::computeVelocityCommands (reference src/social_mpc_controller.cpp:198-214)
        for the fleet, on the GPU: people [B][K][5], n_people [B], pose [B][3] -> (people [B][n_out_max][5], n [B])."""
        torch, L, h = self.torch, _lib.lib(), self.opt._h
        people = np.ascontiguousarray(people, dtype=np.float64)
        B, K, _ = people.shape
        n_out_max = self.A if n_out_max is None else n_out_max
        morg = np.ascontiguousarray(costmap_origin, dtype=np.float64).reshape(-1, 2)
        with torch.cuda.stream(self.stream):
            d_in, d_n = self._t(people, np.float64), self._t(n_people, np.int32)
            d_pose, d_org = self._t(pose, np.float64), self._t(morg, np.float64)
            d_idx = None if costmap_index is None else self._t(costmap_index, np.int32)
            out = torch.zeros(B, n_out_max, 5, dtype=torch.float64, device=self.dev)
            n_out = torch.zeros(B, dtype=torch.int32, device=self.dev)
            a = abi.SmpcFovArgs()
            a.n_robots, a.n_in_max, a.n_out_max, a.n_costmaps = B, K, n_out_max, morg.shape[0]
            a.size_x, a.size_y, a.resolution = int(size_x), int(size_y), float(resolution)
            a.fov_angle = float(self.p.fov_angle if fov_angle is None else fov_angle)
            a.people_in, a.n_people_in, a.pose = d_in.data_ptr(), d_n.data_ptr(), d_pose.data_ptr()
            a.costmap_origin = d_org.data_ptr()
            a.costmap_index = None if d_idx is None else d_idx.data_ptr()
            a.people_out, a.n_people_out = out.data_ptr(), n_out.data_ptr()
            _lib.check(L.smpc_fov_filter_batch_device(h, C.byref(a), self.stream.cuda_stream))
        self.stream.synchronize()
        return out.cpu().numpy(), n_out.cpu().numpy()

    def optimize_batch(self, poses, cmds, people_raw, n_people, speed, costmaps, costmap_origin, costmap_resolution,
                       od: dict, costmap_index=None, od_index=None, n_poses=None, want_people_proj=True,
                       inplace=False, weights=None) -> dict:
        """One controller tick for the fleet (smpc_optimize_batch). poses [B][n][3], cmds [B][>= n-1][2] (trajectorizer
        seeds; n_poses [B] = valid poses per robot, default n for all), people_raw [B][A][5], n_people [B], speed [B][2],
        costmaps [M][sy][sx] u8, od = dict(width, height, resolution, origins [Mo][2], indexes u32 [Mo][h*w]).
        Returns host numpy: optimized [B] (the reference's bool), n_out [B], cmds [B][n][2], path [B][n][3] (rows valid
        up to n_out[b]), people_proj [B][A][6][n], termination, iterations, cost_initial, cost_final, project_status.
        Costmaps / obstacle grids are re-sent to the GPU only when the arrays passed here change identity.
        inplace = True: poses [B][n][3] and cmds [B][n][2] (C-contiguous float64) are the in/out buffers of the C call
        themselves, like the reference's in-out path / cmds arguments — no copies on the Python side.
        weights = (table [P][9], set_index [B]): robot b's critics use row set_index[b] (abi.WEIGHT_NAMES columns;
        optimizer.weight_sets builds the table) instead of the handle's weights (smpc_optimize_batch_weighted)."""
        p = self.p
        poses = np.ascontiguousarray(poses, dtype=np.float64)
        B, n, _ = poses.shape
        assert B == self.B
        if inplace:
            if not (isinstance(cmds, np.ndarray) and cmds.dtype == np.float64 and cmds.flags.c_contiguous
                    and cmds.shape == (B, n, 2)):
                raise ValueError("inplace needs cmds as a C-contiguous float64 array of shape [B][n][2]")
            cmd_rows, pose_rows = cmds, poses
        else:
            cmds_in = np.ascontiguousarray(cmds, dtype=np.float64)
            cmd_rows = np.zeros((B, n, 2))
            k = min(n, cmds_in.shape[1])
            cmd_rows[:, :k] = cmds_in[:, :k]
            pose_rows = poses.copy()
        n_poses = np.full(B, n, dtype=np.int32) if n_poses is None else np.ascontiguousarray(n_poses, dtype=np.int32)
        people_raw = np.ascontiguousarray(people_raw, dtype=np.float64).reshape(B, self.A, 5)
        n_people = np.ascontiguousarray(n_people, dtype=np.int32)
        speed = np.ascontiguousarray(speed, dtype=np.float64).reshape(B, 2)
        costmaps = np.ascontiguousarray(costmaps, dtype=np.uint8)
        morg = np.ascontiguousarray(costmap_origin, dtype=np.float64).reshape(-1, 2)
        oorg = np.ascontiguousarray(od["origins"], dtype=np.float64).reshape(-1, 2)
        oidx = np.ascontiguousarray(od["indexes"], dtype=np.uint32).reshape(oorg.shape[0], -1)
        key = (id(costmaps), costmaps.shape, id(od["indexes"]), morg.tobytes(), oorg.tobytes())
        if key != self._maps_key:
            self._maps_key = key
            self._maps_version += 1
        midx = None if costmap_index is None else np.ascontiguousarray(costmap_index, dtype=np.int32)
        osel = None if od_index is None else np.ascontiguousarray(od_index, dtype=np.int32)
        out = dict(n_out=np.zeros(B, np.int32), optimized=np.zeros(B, np.uint8), termination=np.zeros(B, np.int32),
                   iterations=np.zeros(B, np.int32), cost_initial=np.zeros(B), cost_final=np.zeros(B),
                   project_status=np.zeros(B, np.int32))
        proj = np.zeros((B, self.A, 6, n)) if want_people_proj else None
        io = abi.SmpcFleetIo()
        io.n_robots, io.max_poses, io.n_agents, io.time_step = B, n, self.A, float(p.time_step)
        io.n_poses, io.people, io.n_people, io.speed = (n_poses.ctypes.data, people_raw.ctypes.data,
                                                          n_people.ctypes.data, speed.ctypes.data)
        io.costmaps, io.costmap_origin = costmaps.ctypes.data, morg.ctypes.data
        io.costmap_index = None if midx is None else midx.ctypes.data
        io.n_costmaps, io.size_x, io.size_y = costmaps.shape[0], costmaps.shape[2], costmaps.shape[1]
        io.resolution = float(costmap_resolution)
        io.od_indexes, io.od_origin = oidx.ctypes.data, oorg.ctypes.data
        io.od_index = None if osel is None else osel.ctypes.data
        io.n_od_grids, io.od_width, io.od_height = oorg.shape[0], int(od["width"]), int(od["height"])
        io.od_resolution = float(od["resolution"])
        io.maps_version = self._maps_version
        io.poses, io.cmds = pose_rows.ctypes.data, cmd_rows.ctypes.data
        for k2, v in out.items():
            setattr(io, k2, v.ctypes.data)
        io.people_proj = None if proj is None else proj.ctypes.data
        if weights is None:
            _lib.check(_lib.lib().smpc_optimize_batch(self.opt._h, C.byref(io)))
        else:
            ws, keep = weight_sets_arg(weights, B)
            _lib.check(_lib.lib().smpc_optimize_batch_weighted(self.opt._h, C.byref(io), C.byref(ws)))
        res = dict(out)
        res["optimized"] = out["optimized"].astype(bool)
        res["path"], res["cmds"], res["people_proj"] = pose_rows, cmd_rows, proj
        return res

    EPISODE_METRICS = (("reached", np.uint8), ("ticks", np.int32), ("path_length", np.float64),
                       ("min_person_dist", np.float64), ("intimate_ticks", np.int32), ("personal_ticks", np.int32),
                       ("collision_ticks", np.int32), ("not_optimized_ticks", np.int32), ("cmd_variation", np.float64))

    def run_episodes(self, global_path, pose, speed, people, n_people, costmaps, costmap_origin, costmap_resolution,
                     od: dict, ticks: int, control_period=0.05, goal_tolerance=0.25, costmap_index=None, od_index=None,
                     want_logs=False, weights=None, perception=None, tracker=None, local_costmap=None) -> dict:
        """Closed-loop episodes on the GPU (smpc_run_episodes): each of the B robots runs its crowd scene for up to
        `ticks` controller ticks — trajectorizer seed, constant-velocity people, FOV filter, the fleet tick, a unicycle
        world step — with one upload and one download for the whole run. global_path [B][N][2], pose [B][3],
        speed [B][2], people [B][K][5] at t = 0 (x, y, vx, vy, vz), n_people [B] <= K, maps as in optimize_batch.
        Returns host numpy per episode: reached (bool), ticks, path_length, min_person_dist (inf without people),
        intimate_ticks, personal_ticks, collision_ticks, not_optimized_ticks, cmd_variation; with want_logs also
        pose_log [B][T+1][3], cmd_log [B][T][2], optimized_log [B][T] (bool).
        weights = (table [P][9], set_index [B]) as in optimize_batch: episode b runs with row set_index[b]
        (smpc_run_weighted_episodes).
        perception: abi.perception_params(...), or a dict of its overrides plus an optional stream_index [B], puts a
        sensor between the people and the FOV filter (smpc_run_perceived_episodes): range, occlusion by walls and people,
        missed detections and noisy tracks. The dict then also holds unseen_personal_ticks [B] (ticks with a person
        within 1.2 m that went unreported) and, with want_logs, seen_log [B][T][K][5] and n_seen_log [B][T] (what the
        FOV filter received at each tick).
        tracker: abi.tracker_params(...), or a dict of its overrides, puts a people tracker after the sensor
        (smpc_run_tracked_episodes): a constant-velocity Kalman track per person, published after confirm_hits
        detections, coasted through max_coast_ticks misses and delivered latency_ticks late. It needs perception=, with
        vel_noise=0. The dict then also holds untracked_personal_ticks [B] (ticks with a person within 1.2 m missing
        from what the FOV filter received), track_rows [B] (people rows it received), mean_track_pos_error and
        mean_track_vel_error [B] (their mean distance from the true position and velocity of the same tick, NaN
        without rows) and, with want_logs, track_id_log [B][T][K] (the agent ids of the seen_log rows, -1 past
        n_seen_log); seen_log and n_seen_log then hold the tracker's delayed list.
        local_costmap: abi.local_costmap_params(...), or a dict of its overrides, makes the FOV filter and the fleet
        tick read a rolling robot-centred window of each robot's costmap with the people in it marked and inflated
        (smpc_run_local_costmap_episodes), rebuilt every update_period_ticks; it works with every keyword above. The dict
        then also holds marked_rows [B] (people rows marked, summed over the builds) and, with want_logs,
        local_costmap_log [B][n_builds][size_y][size_x] and local_origin_log [B][n_builds][2] (each build's window and
        origin; zero and NaN for builds after the episode was done)."""
        if tracker is not None and perception is None:
            raise ValueError("tracker= needs perception=: the tracker follows the sensor")
        io, out, logs, keep = self.episode_io(global_path, pose, speed, people, n_people, costmaps, costmap_origin,
                                              costmap_resolution, od, ticks, control_period, goal_tolerance,
                                              costmap_index, od_index, want_logs)
        if perception is not None or local_costmap is not None:
            ws, wkeep = weight_sets_arg(weights, self.B) if weights is not None else (None, None)
            out.update(self._perceived(io, None, None, ws, None, perception, tracker, io.n_people, want_logs,
                                       local_costmap))
        elif weights is None:
            _lib.check(_lib.lib().smpc_run_episodes(self.opt._h, C.byref(io)))
        else:
            ws, wkeep = weight_sets_arg(weights, self.B)
            _lib.check(_lib.lib().smpc_run_weighted_episodes(self.opt._h, C.byref(io), None, None, C.byref(ws)))
        res = dict(out, **logs)
        res["reached"] = out["reached"].astype(bool)
        if want_logs:
            res["optimized_log"] = logs["optimized_log"].astype(bool)
        return res

    def run_crowd_episodes(self, global_path, pose, speed, people, n_people, costmaps, costmap_origin,
                           costmap_resolution, od: dict, ticks: int, goals, desired_speed, substeps=1,
                           control_period=0.05, goal_tolerance=0.25, costmap_index=None, od_index=None,
                           want_logs=False, weights=None, orca=None, perception=None, tracker=None,
                           local_costmap=None) -> dict:
        """Closed-loop episodes with a reactive crowd (smpc_run_crowd_episodes): run_episodes, but the people walk to
        their goals [B][K][2] at their desired speeds [B][K] under the lightsfm social force model, `substeps` updates
        per control period, and give way to the robot; people [B][K][5] is their state at t = 0. Returns the dict of
        run_episodes plus people_disturbance [B] (sum of |F(robot -> person)| * dt_s over ticks, substeps and people);
        with want_logs also people_log [B][T+1][K][5] (x, y, vx, vy, vz at every tick, row 0 = the input).
        weights: as in run_episodes. orca: abi.orca_params(...) (or a dict of its overrides) moves the people by ORCA
        instead (smpc_run_orca_episodes), a crowd model the controller does not predict with; people_disturbance is
        then the velocity change the robot demanded, in m. perception, tracker, local_costmap: as in run_episodes."""
        return self._crowd_run(None, global_path, pose, speed, people, n_people, costmaps, costmap_origin,
                               costmap_resolution, od, ticks, goals, desired_speed, substeps, control_period,
                               goal_tolerance, costmap_index, od_index, want_logs, weights, orca, perception, tracker,
                               local_costmap)

    def run_shared_episodes(self, global_path, pose, speed, people, n_people, costmaps, costmap_origin,
                            costmap_resolution, od: dict, ticks: int, goals, desired_speed, robots_per_scene,
                            substeps=1, control_period=0.05, goal_tolerance=0.25, costmap_index=None, od_index=None,
                            want_logs=False, weights=None, orca=None, perception=None, tracker=None,
                            local_costmap=None) -> dict:
        """Closed-loop episodes in shared scenes (smpc_run_shared_episodes): run_crowd_episodes with the B robots
        grouped into S = B / R scenes of R = robots_per_scene consecutive robots that share one crowd, costmap and
        obstacle grid, and that see each other as people. Per robot: global_path [B][N][2], pose [B][3],
        speed [B][2], costmap_index / od_index [B] (equal within a scene). Per scene: people [S][K][5],
        n_people [S], goals [S][K][2], desired_speed [S][K]. Returns the dict of run_crowd_episodes plus
        robot_min_dist [B] (nearest other robot of the scene, inf for R = 1) and robot_intimate_ticks [B]; with
        want_logs people_log is per scene, [S][T+1][K][5]. weights: as in run_episodes, set_index per robot.
        orca: as in run_crowd_episodes. perception: as in run_episodes; a robot's list is its scene view, the other
        R - 1 robots then the people, so seen_log is [B][T][R-1+K][5]. tracker: as in run_episodes; the other robots
        are tracked too (ids K + r) but count in none of its metrics. local_costmap: as in run_episodes; the other
        robots of the scene are marked like people."""
        return self._crowd_run(int(robots_per_scene), global_path, pose, speed, people, n_people, costmaps,
                               costmap_origin, costmap_resolution, od, ticks, goals, desired_speed, substeps,
                               control_period, goal_tolerance, costmap_index, od_index, want_logs, weights, orca,
                               perception, tracker, local_costmap)

    def _crowd_run(self, R, global_path, pose, speed, people, n_people, costmaps, costmap_origin, costmap_resolution,
                   od, ticks, goals, desired_speed, substeps, control_period, goal_tolerance, costmap_index, od_index,
                   want_logs, weights=None, orca=None, perception=None, tracker=None, local_costmap=None) -> dict:
        """run_crowd_episodes (R None) or run_shared_episodes (R robots per scene); orca: the ORCA crowd; perception:
        the sensor between the scene and the FOV filter; tracker: the people tracker after it; local_costmap: the
        rolling windows the FOV filter and the fleet tick read."""
        if tracker is not None and perception is None:
            raise ValueError("tracker= needs perception=: the tracker follows the sensor")
        io, out, logs, keep = self.episode_io(global_path, pose, speed, people, n_people, costmaps, costmap_origin,
                                              costmap_resolution, od, ticks, control_period, goal_tolerance,
                                              costmap_index, od_index, want_logs, robots_per_scene=R or 1)
        B, T, K = self.B, int(ticks), io.n_people
        S = B // (R or 1)
        goals = np.ascontiguousarray(goals, dtype=np.float64).reshape(S, K, 2)
        vdes = np.ascontiguousarray(desired_speed, dtype=np.float64).reshape(S, K)
        crowd = abi.SmpcCrowdIo()
        crowd.goals = goals.ctypes.data if K > 0 else None
        crowd.desired_speed = vdes.ctypes.data if K > 0 else None
        crowd.substeps = int(substeps)
        disturbance = np.zeros(B)
        crowd.people_disturbance = disturbance.ctypes.data
        people_log = np.zeros((S, T + 1, K, 5)) if want_logs else None
        crowd.people_log = None if people_log is None else people_log.ctypes.data
        res = dict(out, **logs)
        scene = None
        if R is not None:
            res.update(robot_min_dist=np.zeros(B), robot_intimate_ticks=np.zeros(B, np.int32))
            scene = abi.SmpcSceneIo(R, res["robot_min_dist"].ctypes.data, res["robot_intimate_ticks"].ctypes.data)
        if perception is not None or local_costmap is not None:
            op = None if orca is None else orca if isinstance(orca, abi.SmpcOrcaParams) else abi.orca_params(**orca)
            ws, wkeep = weight_sets_arg(weights, B) if weights is not None else (None, None)
            res.update(self._perceived(io, crowd, scene, ws, op, perception, tracker, (R or 1) - 1 + K, want_logs,
                                       local_costmap))
        elif orca is not None:
            op = orca if isinstance(orca, abi.SmpcOrcaParams) else abi.orca_params(**orca)
            ws, wkeep = weight_sets_arg(weights, B) if weights is not None else (None, None)
            _lib.check(_lib.lib().smpc_run_orca_episodes(self.opt._h, C.byref(io), C.byref(crowd),
                                                         None if scene is None else C.byref(scene),
                                                         None if ws is None else C.byref(ws), C.byref(op)))
        elif weights is not None:
            ws, wkeep = weight_sets_arg(weights, B)
            _lib.check(_lib.lib().smpc_run_weighted_episodes(self.opt._h, C.byref(io), C.byref(crowd),
                                                             None if scene is None else C.byref(scene), C.byref(ws)))
        elif R is None:
            _lib.check(_lib.lib().smpc_run_crowd_episodes(self.opt._h, C.byref(io), C.byref(crowd)))
        else:
            _lib.check(_lib.lib().smpc_run_shared_episodes(self.opt._h, C.byref(io), C.byref(crowd), C.byref(scene)))
        res["reached"] = out["reached"].astype(bool)
        res["people_disturbance"] = disturbance
        if want_logs:
            res["optimized_log"] = logs["optimized_log"].astype(bool)
            res["people_log"] = people_log
        return res

    def _perceived(self, io, crowd, scene, ws, op, perception, tracker, n_rows, want_logs, local_costmap=None) -> dict:
        """smpc_run_perceived_episodes (tracker None), smpc_run_tracked_episodes or, with local_costmap,
        smpc_run_local_costmap_episodes (perception may then be None) on the built arguments: the results of the
        perception, the tracker and the local costmap. n_rows = L, the rows of the perceived list."""
        out, pc, tk = {}, None, None
        if perception is not None:
            pc, out, keep = perception_arg(perception, self.B, io.n_ticks, n_rows, want_logs)
        args = [self.opt._h, C.byref(io), None if crowd is None else C.byref(crowd),
                None if scene is None else C.byref(scene), None if ws is None else C.byref(ws),
                None if op is None else C.byref(op), None if pc is None else C.byref(pc)]
        if tracker is not None:
            tk, raw = tracker_arg(tracker, pc, self.B, io.n_ticks, n_rows, want_logs)
        if local_costmap is not None:
            lc, lout = local_costmap_arg(local_costmap, self.B, io.n_ticks, want_logs)
            _lib.check(_lib.lib().smpc_run_local_costmap_episodes(*args, None if tk is None else C.byref(tk),
                                                                  C.byref(lc)))
            out = dict(out, **lout)
        elif tk is None:
            _lib.check(_lib.lib().smpc_run_perceived_episodes(*args))
        else:
            _lib.check(_lib.lib().smpc_run_tracked_episodes(*args, C.byref(tk)))
        return out if tk is None else dict(out, **tracker_results(raw))

    def episode_io(self, global_path, pose, speed, people, n_people, costmaps, costmap_origin, costmap_resolution,
                   od: dict, ticks: int, control_period=0.05, goal_tolerance=0.25, costmap_index=None, od_index=None,
                   want_logs=False, robots_per_scene=1):
        """The smpc_episode_io of run_episodes with its output arrays: (io, metrics, logs, inputs kept alive).
        people and n_people have one row per scene of robots_per_scene robots."""
        B, T = self.B, int(ticks)
        S = B // robots_per_scene
        gp = np.ascontiguousarray(global_path, dtype=np.float64)
        assert gp.ndim == 3 and gp.shape[0] == B and gp.shape[2] == 2
        pose = np.ascontiguousarray(pose, dtype=np.float64).reshape(B, 3)
        speed = np.ascontiguousarray(speed, dtype=np.float64).reshape(B, 2)
        people = np.ascontiguousarray(people, dtype=np.float64)
        K = people.shape[1] if people.ndim == 3 else 0
        people = people.reshape(S, K, 5)
        n_people = np.ascontiguousarray(n_people, dtype=np.int32).reshape(S)
        costmaps = np.ascontiguousarray(costmaps, dtype=np.uint8)
        morg = np.ascontiguousarray(costmap_origin, dtype=np.float64).reshape(-1, 2)
        oorg = np.ascontiguousarray(od["origins"], dtype=np.float64).reshape(-1, 2)
        oidx = np.ascontiguousarray(od["indexes"], dtype=np.uint32).reshape(oorg.shape[0], -1)
        midx = None if costmap_index is None else np.ascontiguousarray(costmap_index, dtype=np.int32)
        osel = None if od_index is None else np.ascontiguousarray(od_index, dtype=np.int32)
        out = {k: np.zeros(B, dt) for k, dt in self.EPISODE_METRICS}
        logs = dict(pose_log=np.zeros((B, T + 1, 3)), cmd_log=np.zeros((B, T, 2)),
                    optimized_log=np.zeros((B, T), np.uint8)) if want_logs else {}
        io = abi.SmpcEpisodeIo()
        io.n_episodes, io.n_ticks, io.n_path, io.n_people, io.n_agents = B, T, gp.shape[1], K, self.A
        io.control_period, io.goal_tolerance = float(control_period), float(goal_tolerance)
        io.global_path, io.pose, io.speed = gp.ctypes.data, pose.ctypes.data, speed.ctypes.data
        io.people = people.ctypes.data if K > 0 else None
        io.n_people_each = n_people.ctypes.data
        io.costmaps, io.costmap_origin = costmaps.ctypes.data, morg.ctypes.data
        io.costmap_index = None if midx is None else midx.ctypes.data
        io.n_costmaps, io.size_x, io.size_y = costmaps.shape[0], costmaps.shape[2], costmaps.shape[1]
        io.resolution = float(costmap_resolution)
        io.od_indexes, io.od_origin = oidx.ctypes.data, oorg.ctypes.data
        io.od_index = None if osel is None else osel.ctypes.data
        io.n_od_grids, io.od_width, io.od_height = oorg.shape[0], int(od["width"]), int(od["height"])
        io.od_resolution = float(od["resolution"])
        for k, v in list(out.items()) + list(logs.items()):
            setattr(io, k, v.ctypes.data)
        keep = (gp, pose, speed, people, n_people, costmaps, morg, oorg, oidx, midx, osel)
        return io, out, logs, keep
