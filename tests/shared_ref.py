"""numpy restatement of the shared scenes of smpc_run_shared_episodes (include/smpc.h): the crowd step of one scene with
R robots as agents (built like tests/crowd_ref.py on tests/presolve_ref.py), the scene view each robot's FOV filter
reads, and the robot-robot metrics."""
from __future__ import annotations

import math

import numpy as np

from tests import crowd_ref as cref
from tests import episode_ref
from tests import presolve_ref as pr


def crowd_step(people, has_goal, goals, vdes, robot_poses, robot_cmds, running, od, dt_c, substeps, near_eps=None):
    """One tick of the crowd of one scene: people [n][5], has_goal [n], goals [n][2], vdes [n], the R robots' poses
    [R][3] and commands [R][2] of the tick, running [R] (a finished robot stands still), od = one grid
    (crowd_ref.od_of). The people feel every other person, then robots 0 .. R-1 in order. Returns (people [n][5],
    has_goal [n], disturbance [R] = per robot the sum of |F(robot -> i)| * dt_s); with near_eps also the mask of
    crowd_ref.crowd_step. With one running robot this is crowd_ref.crowd_step."""
    people = np.asarray(people, dtype=np.float64)
    n = people.shape[0]
    R = len(robot_poses)
    dts = dt_c / substeps
    state = []
    for r in range(R):
        rx, ry, th = (float(c) for c in robot_poses[r])
        v = float(robot_cmds[r][0]) if running[r] else 0.0
        state.append((rx, ry, th, v, v * math.cos(th), v * math.sin(th)))
    agents = []
    for i in range(n):
        x, y, vx, vy, vz = (float(c) for c in people[i])
        agents.append(dict(pos=[x, y], vel=[vx, vy], yaw=math.atan2(vy, vx), lv=math.hypot(vx, vy), av=vz,
                           vdes=float(vdes[i]), radius=0.5, goal=[float(goals[i][0]), float(goals[i][1])]
                           if has_goal[i] else None, obstacle=None, force=[0.0, 0.0]))
    near = np.zeros(n, bool)
    dist = np.zeros(R)
    for s in range(substeps):
        ts = s * dts
        robots = [dict(pos=[rx + ts * rvx, ry + ts * rvy], vel=[rvx, rvy], yaw=th, lv=v, av=0.0, vdes=0.6, radius=0.5,
                       goal=None, obstacle=None, force=[0.0, 0.0]) for rx, ry, th, v, rvx, rvy in state]
        for a in agents:
            a["obstacle"] = cref.obstacle_cell(a["pos"], od)
            for r, robot in enumerate(robots):
                f = cref._robot_force(a, robot)
                dist[r] += math.sqrt(f[0] * f[0] + f[1] * f[1]) * dts
        held = [a["goal"] for a in agents]
        pr.sfm_forces(agents + robots)
        pr.sfm_update(agents, dts)
        for i, a in enumerate(agents):
            if held[i] is not None:
                d = math.hypot(held[i][0] - a["pos"][0], held[i][1] - a["pos"][1])
                if near_eps is not None and abs(d - cref.GOAL_RADIUS) <= near_eps:
                    near[i] = True
    out = np.array([[a["pos"][0], a["pos"][1], a["vel"][0], a["vel"][1], a["av"]] for a in agents]).reshape(n, 5)
    flags = np.array([a["goal"] is not None for a in agents], dtype=bool)
    if near_eps is not None:
        return out, flags, dist, near
    return out, flags, dist


def scene_views(poses, speeds, running, people, n_people, R, cos=np.cos, sin=np.sin):
    """The FOV filter's input of every robot at one tick: poses [B][3] of the tick, speeds [B][2] (the measured speed),
    running [B], people [S][K][5] and n_people [S] of the scenes. Returns views [B][R-1+K][5] (the other robots of the
    scene in index order as (x, y, v cos th, v sin th, w), zero velocity once done, then the scene's people) and
    n_view [B]. cos / sin: the trigonometry, which the caller may take from the device's math library."""
    B = poses.shape[0]
    K = people.shape[1]
    c, s = cos(poses[:, 2]), sin(poses[:, 2])
    v = np.where(running, speeds[:, 0], 0.0)
    w = np.where(running, speeds[:, 1], 0.0)
    as_person = np.stack([poses[:, 0], poses[:, 1], v * c, v * s, w], axis=1)
    views = np.zeros((B, R - 1 + K, 5))
    n_view = np.zeros(B, np.int32)
    for b in range(B):
        sc, me = divmod(b, R)
        others = [sc * R + r for r in range(R) if r != me]
        views[b, : R - 1] = as_person[others]
        views[b, R - 1:] = people[sc]
        n_view[b] = R - 1 + int(n_people[sc])
    return views, n_view


def robot_metrics(pose_log, ticks, R):
    """robot_min_dist [B] and robot_intimate_ticks [B] from pose_log [B][T+1][3] (rows after an episode repeat its
    final pose) and ticks [B]."""
    B = pose_log.shape[0]
    dmin = np.full(B, np.inf)
    intimate = np.zeros(B, np.int32)
    for b in range(B):
        sc = b // R
        for k in range(int(ticks[b])):
            d = np.inf
            for o in range(sc * R, sc * R + R):
                if o == b:
                    continue
                dx, dy = pose_log[o, k + 1, 0] - pose_log[b, k + 1, 0], pose_log[o, k + 1, 1] - pose_log[b, k + 1, 1]
                d = min(d, float(np.sqrt(dx * dx + dy * dy)))
            dmin[b] = min(dmin[b], d)
            intimate[b] += d < episode_ref.INTIMATE
    return dmin, intimate
