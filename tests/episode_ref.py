"""numpy restatement of the world of smpc_run_episodes (include/smpc.h): the robot's forward-Euler step, the
constant-velocity people and the per-episode metrics recomputed from the logs. Products and sums are rounded one at a
time, as the kernels write them (__dmul_rn / __dadd_rn), so people positions and distances agree bit for bit."""
from __future__ import annotations

import numpy as np

INTIMATE, PERSONAL, LETHAL = 0.45, 1.2, 253


def yaw_roundtrip(yaw):
    h = np.asarray(yaw, dtype=np.float64) * 0.5
    qz, qw = np.sin(h), np.cos(h)
    return np.arctan2(2.0 * (qw * qz), qw * qw - qz * qz)


def euler_step(pose, cmd, dt_c):
    """pose [..][3], cmd [..][2] -> the next pose: unicycle forward Euler, yaw through setRPY / getYaw."""
    pose = np.asarray(pose, dtype=np.float64)
    cmd = np.asarray(cmd, dtype=np.float64)
    x, y, th = pose[..., 0], pose[..., 1], pose[..., 2]
    v, w = cmd[..., 0], cmd[..., 1]
    return np.stack([x + (v * np.cos(th)) * dt_c, y + (v * np.sin(th)) * dt_c, yaw_roundtrip(th + w * dt_c)], axis=-1)


def people_at(people0, t):
    """people [..][K][5] at time t (constant velocity; velocity columns unchanged)."""
    p = np.array(people0, dtype=np.float64, copy=True)
    p[..., 0] = p[..., 0] + p[..., 2] * t
    p[..., 1] = p[..., 1] + p[..., 3] * t
    return p


def cell_cost(costmap, origin, res, x, y):
    """Costmap2D::worldToMap of (x, y); a cell outside the map reads as 255."""
    if x < origin[0] or y < origin[1]:
        return 255
    mx, my = int((x - origin[0]) / res), int((y - origin[1]) / res)
    if mx >= costmap.shape[1] or my >= costmap.shape[0]:
        return 255
    return int(costmap[my, mx])


def metrics_from_logs(pose_log, cmd_log, optimized_log, ticks, people0, n_people, global_path, costmaps,
                      costmap_origin, res, costmap_index, dt_c, goal_tol, eps=1e-9):
    """Every metric of smpc_episode_io recomputed from the logs of the ticks each episode ran. Also returns
    `near_threshold` [B]: some tick's nearest-person distance lies within eps of 0.45 or 1.2 m (its counts may
    legitimately differ in the last bit of a distance)."""
    B = pose_log.shape[0]
    M = costmaps.shape[0]
    out = {k: np.zeros(B, np.int32) for k in ("intimate_ticks", "personal_ticks", "collision_ticks",
                                                "not_optimized_ticks")}
    out.update(path_length=np.zeros(B), min_person_dist=np.full(B, np.inf), cmd_variation=np.zeros(B),
               reached=np.zeros(B, bool), near_threshold=np.zeros(B, bool), goal_first=np.full(B, -1))
    for b in range(B):
        m = int(costmap_index[b]) if costmap_index is not None else b % M
        goal = global_path[b, -1]
        for k in range(int(ticks[b])):
            p0, p1 = pose_log[b, k], pose_log[b, k + 1]
            out["path_length"][b] += np.sqrt((p1[0] - p0[0]) * (p1[0] - p0[0]) + (p1[1] - p0[1]) * (p1[1] - p0[1]))
            ppl = people_at(people0[b, : int(n_people[b])], (k + 1) * dt_c)
            dmin = np.inf
            if ppl.shape[0]:
                dx, dy = ppl[:, 0] - p1[0], ppl[:, 1] - p1[1]
                dmin = float(np.sqrt(dx * dx + dy * dy).min())
            out["min_person_dist"][b] = min(out["min_person_dist"][b], dmin)
            out["intimate_ticks"][b] += dmin < INTIMATE
            out["personal_ticks"][b] += dmin < PERSONAL
            if abs(dmin - INTIMATE) <= eps or abs(dmin - PERSONAL) <= eps:
                out["near_threshold"][b] = True
            out["collision_ticks"][b] += cell_cost(costmaps[m], costmap_origin[m], res, p1[0], p1[1]) >= LETHAL
            out["not_optimized_ticks"][b] += not optimized_log[b, k]
            if k >= 1:
                out["cmd_variation"][b] += (abs(cmd_log[b, k, 0] - cmd_log[b, k - 1, 0]) +
                                            abs(cmd_log[b, k, 1] - cmd_log[b, k - 1, 1]))
            gd = np.sqrt((p1[0] - goal[0]) * (p1[0] - goal[0]) + (p1[1] - goal[1]) * (p1[1] - goal[1]))
            if gd <= goal_tol and out["goal_first"][b] < 0:
                out["goal_first"][b] = k
        out["reached"][b] = out["goal_first"][b] >= 0
    return out
