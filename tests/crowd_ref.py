"""numpy restatement of the reactive crowd of smpc_run_crowd_episodes (include/smpc.h): one controller tick of the
people of one scene under the lightsfm social force model, built on the projection's reference in tests/presolve_ref.py
(sfm_forces, sfm_update, compute_obstacle), and the episode metrics recomputed with the people taken from a log."""
from __future__ import annotations

import math

import numpy as np

from tests import episode_ref
from tests import presolve_ref as pr

GOAL_RADIUS = 0.25


def od_of(od: dict, grid: int = 0) -> dict:
    """One grid of an obstacle-distance dict of the scenarios (origins [Mo][2], indexes [Mo][h*w]) in the form of
    presolve_ref.compute_obstacle."""
    org = np.asarray(od["origins"], dtype=np.float64).reshape(-1, 2)
    idx = np.asarray(od["indexes"], dtype=np.uint32).reshape(org.shape[0], -1)
    return dict(width=int(od["width"]), height=int(od["height"]), resolution=od["resolution"],
                origin_x=float(org[grid, 0]), origin_y=float(org[grid, 1]), indexes=idx[grid])


def obstacle_cell(pos, od):
    """Position of the nearest obstacle cell of the grid at pos (float-rounded like computeObstacle), None outside it."""
    res = pr.f32(od["resolution"])
    xc = math.floor((pos[0] - od["origin_x"]) / res)
    yc = math.floor((pos[1] - od["origin_y"]) / res)
    if not (0 <= xc < od["width"] and 0 <= yc < od["height"]):
        return None
    if int(od["indexes"][xc + yc * od["width"]]) >= od["width"] * od["height"]:
        return None
    v = pr.compute_obstacle(pos, od)  # agent - cell (the projection's obstacles1)
    return [pos[0] - v[0], pos[1] - v[1]]


def _robot_force(a, robot):
    """The pair force of the robot on person a: sfm_forces on the two of them with a's goal and obstacle off, minus the
    braking term that is then a's desired force."""
    me = dict(a, goal=None, obstacle=None)
    pair = [me, dict(robot)]
    pr.sfm_forces(pair)
    return [me["force"][0] - (-a["vel"][0] / 0.5), me["force"][1] - (-a["vel"][1] / 0.5)]


def crowd_step(people, has_goal, goals, vdes, robot_pose, robot_cmd, od, dt_c, substeps, near_eps=None):
    """One tick of the crowd of one scene: people [n][5] (x, y, vx, vy, vz), has_goal [n], goals [n][2], vdes [n], the
    robot's pose (x, y, yaw) and command (v, w) of the tick, od = one grid (od_of), `substeps` synchronous updates of
    dt_c / substeps. Returns (people [n][5], has_goal [n], disturbance = sum of |F(robot -> i)| * dt_s). With near_eps
    also a mask [n] of people whose distance to the goal came within near_eps of 0.25 m while the goal was held."""
    people = np.asarray(people, dtype=np.float64)
    n = people.shape[0]
    dts = dt_c / substeps
    rx, ry, th = (float(c) for c in robot_pose)
    v = float(robot_cmd[0])
    rvx, rvy = v * math.cos(th), v * math.sin(th)
    agents = []
    for i in range(n):
        x, y, vx, vy, vz = (float(c) for c in people[i])
        agents.append(dict(pos=[x, y], vel=[vx, vy], yaw=math.atan2(vy, vx), lv=math.hypot(vx, vy), av=vz,
                           vdes=float(vdes[i]), radius=0.5, goal=[float(goals[i][0]), float(goals[i][1])]
                           if has_goal[i] else None, obstacle=None, force=[0.0, 0.0]))
    near = np.zeros(n, bool)
    dist = 0.0
    for s in range(substeps):
        ts = s * dts
        robot = dict(pos=[rx + ts * rvx, ry + ts * rvy], vel=[rvx, rvy], yaw=th, lv=v, av=0.0, vdes=0.6, radius=0.5,
                     goal=None, obstacle=None, force=[0.0, 0.0])
        for a in agents:
            a["obstacle"] = obstacle_cell(a["pos"], od)
            f = _robot_force(a, robot)
            dist += math.sqrt(f[0] * f[0] + f[1] * f[1]) * dts
        held = [a["goal"] for a in agents]
        pr.sfm_forces(agents + [robot])
        pr.sfm_update(agents, dts)
        for i, a in enumerate(agents):
            if held[i] is not None:
                d = math.hypot(held[i][0] - a["pos"][0], held[i][1] - a["pos"][1])
                if near_eps is not None and abs(d - GOAL_RADIUS) <= near_eps:
                    near[i] = True
    out = np.array([[a["pos"][0], a["pos"][1], a["vel"][0], a["vel"][1], a["av"]] for a in agents]).reshape(n, 5)
    flags = np.array([a["goal"] is not None for a in agents], dtype=bool)
    if near_eps is not None:
        return out, flags, dist, near
    return out, flags, dist


def metrics_from_people_log(pose_log, cmd_log, optimized_log, ticks, people_log, n_people, global_path, costmaps,
                            costmap_origin, res, costmap_index, goal_tol, eps=1e-9):
    """episode_ref.metrics_from_logs with the people of tick k + 1 taken from people_log [B][T+1][K][5]."""
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
            ppl = people_log[b, k + 1, : int(n_people[b])]
            dmin = np.inf
            if ppl.shape[0]:
                dx, dy = ppl[:, 0] - p1[0], ppl[:, 1] - p1[1]
                dmin = float(np.sqrt(dx * dx + dy * dy).min())
            out["min_person_dist"][b] = min(out["min_person_dist"][b], dmin)
            out["intimate_ticks"][b] += dmin < episode_ref.INTIMATE
            out["personal_ticks"][b] += dmin < episode_ref.PERSONAL
            if abs(dmin - episode_ref.INTIMATE) <= eps or abs(dmin - episode_ref.PERSONAL) <= eps:
                out["near_threshold"][b] = True
            cost = episode_ref.cell_cost(costmaps[m], costmap_origin[m], res, p1[0], p1[1])
            out["collision_ticks"][b] += cost >= episode_ref.LETHAL
            out["not_optimized_ticks"][b] += not optimized_log[b, k]
            if k >= 1:
                out["cmd_variation"][b] += (abs(cmd_log[b, k, 0] - cmd_log[b, k - 1, 0]) +
                                            abs(cmd_log[b, k, 1] - cmd_log[b, k - 1, 1]))
            gd = np.sqrt((p1[0] - goal[0]) * (p1[0] - goal[0]) + (p1[1] - goal[1]) * (p1[1] - goal[1]))
            if gd <= goal_tol and out["goal_first"][b] < 0:
                out["goal_first"][b] = k
        out["reached"][b] = out["goal_first"][b] >= 0
    return out
