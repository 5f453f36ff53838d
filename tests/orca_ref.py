"""numpy restatement of the ORCA crowd of smpc_run_orca_episodes (include/smpc.h): one controller tick of the people of
one scene, RVO2's Agent::computeNewVelocity / linearProgram1/2/3 / Agent::update in FP64, written operation for operation
like smpc_orca_step_kernel (compiled without FMA contraction), so that the device's lines are reproduced bit for bit.
A "near tie" is a branch test of the model that came within NEAR_EPS of flipping: such a person's result may differ
from the device's by more than rounding."""
from __future__ import annotations

import math

import numpy as np

from tests import crowd_ref as cref
from tests import presolve_ref as pr

RVO_EPSILON = 1e-5
NEAR_EPS = 1e-9
GOAL_RADIUS = 0.25
DEFAULTS = dict(neighbor_dist=10.0, max_neighbors=10, time_horizon=5.0, time_horizon_obst=5.0, person_radius=0.3,
                robot_radius=0.3, robot_responsibility=0.5)


class _Tie:
    """Collects whether any branch test came within NEAR_EPS of its threshold."""

    def __init__(self):
        self.near = False

    def __call__(self, a, b=0.0):
        if abs(a - b) <= NEAR_EPS:
            self.near = True


def _det(ax, ay, bx, by):
    return ax * by - ay * bx


def linear_program1(lines, no, radius, opt, dir_opt, tie=None):
    """RVO2 linearProgram1: the optimum on line `no` (point px, py, direction dx, dy) within the circle and the lines
    before it, or None."""
    tie = tie or _Tie()
    px, py, dx, dy = lines[no]
    dot = px * dx + py * dy
    disc = dot * dot + radius * radius - (px * px + py * py)
    tie(disc)
    if disc < 0.0:
        return None
    sq = math.sqrt(disc)
    tl, tr = -dot - sq, -dot + sq
    for i in range(no):
        qx, qy, ex, ey = lines[i]
        den = _det(dx, dy, ex, ey)
        num = _det(ex, ey, px - qx, py - qy)
        tie(abs(den), RVO_EPSILON)
        if abs(den) <= RVO_EPSILON:
            tie(num)
            if num < 0.0:
                return None
            continue
        t = num / den
        tie(den)
        if den >= 0.0:
            tie(t, tr)
            tr = min(tr, t)
        else:
            tie(t, tl)
            tl = max(tl, t)
        tie(tl, tr)
        if tl > tr:
            return None
    if dir_opt:
        d = opt[0] * dx + opt[1] * dy
        tie(d)
        t = tr if d > 0.0 else tl
    else:
        t = dx * (opt[0] - px) + dy * (opt[1] - py)
        tie(t, tl)
        tie(t, tr)
        if t < tl:
            t = tl
        elif t > tr:
            t = tr
    return (px + t * dx, py + t * dy)


def linear_program2(lines, radius, opt, dir_opt, tie=None):
    """RVO2 linearProgram2: (first line it could not satisfy or len(lines), result)."""
    tie = tie or _Tie()
    ox, oy = opt
    if dir_opt:
        res = (ox * radius, oy * radius)
    elif ox * ox + oy * oy > radius * radius:  # both branches agree to rounding: no tie
        ln = math.sqrt(ox * ox + oy * oy)
        res = (ox / ln * radius, oy / ln * radius)
    else:
        res = (ox, oy)
    for i, (px, py, dx, dy) in enumerate(lines):
        v = _det(dx, dy, px - res[0], py - res[1])
        tie(v)
        if v > 0.0:
            r = linear_program1(lines, i, radius, opt, dir_opt, tie)
            if r is None:
                return i, res
            res = r
    return len(lines), res


def linear_program3(lines, n_obst, begin, radius, res, tie=None):
    """RVO2 linearProgram3: from line `begin` on, the velocity that minimises the largest violation of the soft lines,
    the first n_obst lines kept hard."""
    tie = tie or _Tie()
    distance = 0.0
    for i in range(begin, len(lines)):
        pix, piy, dix, diy = lines[i]
        v = _det(dix, diy, pix - res[0], piy - res[1])
        tie(v, distance)
        if v > distance:
            proj = list(lines[:n_obst])
            for j in range(n_obst, i):
                pjx, pjy, djx, djy = lines[j]
                dt = _det(dix, diy, djx, djy)
                tie(abs(dt), RVO_EPSILON)
                if abs(dt) <= RVO_EPSILON:
                    d = dix * djx + diy * djy
                    tie(d)
                    if d > 0.0:
                        continue
                    qx, qy = 0.5 * (pix + pjx), 0.5 * (piy + pjy)
                else:
                    s = _det(djx, djy, pix - pjx, piy - pjy) / dt
                    qx, qy = pix + s * dix, piy + s * diy
                ddx, ddy = djx - dix, djy - diy
                ln = math.sqrt(ddx * ddx + ddy * ddy)
                proj.append((qx, qy, ddx / ln, ddy / ln))
            fail, r = linear_program2(proj, radius, (-diy, dix), True, tie)
            if fail >= len(proj):
                res = r
            distance = _det(dix, diy, pix - res[0], piy - res[1])
    return res


def orca_line(rp, rv, cr, inv_t, inv_dt, v, resp, tie=None):
    """The ORCA line (px, py, dx, dy) of an agent at relative position rp = other - me with relative velocity
    rv = mine - other's, combined radius cr, and u; None for a collision with |w| == 0."""
    tie = tie or _Tie()
    rpx, rpy = rp
    rvx, rvy = rv
    dist_sq = rpx * rpx + rpy * rpy
    cr_sq = cr * cr
    tie(dist_sq, cr_sq)
    if dist_sq > cr_sq:
        wx, wy = rvx - inv_t * rpx, rvy - inv_t * rpy
        wl_sq = wx * wx + wy * wy
        dp1 = wx * rpx + wy * rpy
        tie(dp1)
        if dp1 < 0.0:
            tie(dp1 * dp1, cr_sq * wl_sq)
        if dp1 < 0.0 and dp1 * dp1 > cr_sq * wl_sq:
            wl = math.sqrt(wl_sq)
            uwx, uwy = wx / wl, wy / wl
            dx, dy = uwy, -uwx
            s = cr * inv_t - wl
            ux, uy = s * uwx, s * uwy
        else:
            leg = math.sqrt(dist_sq - cr_sq)
            side = _det(rpx, rpy, wx, wy)
            tie(side)
            if side > 0.0:
                dx, dy = (rpx * leg - rpy * cr) / dist_sq, (rpx * cr + rpy * leg) / dist_sq
            else:
                dx, dy = -(rpx * leg + rpy * cr) / dist_sq, -(-rpx * cr + rpy * leg) / dist_sq
            dp2 = rvx * dx + rvy * dy
            ux, uy = dp2 * dx - rvx, dp2 * dy - rvy
    else:
        wx, wy = rvx - inv_dt * rpx, rvy - inv_dt * rpy
        wl = math.sqrt(wx * wx + wy * wy)
        tie(wl)
        if wl == 0.0:
            return None
        uwx, uwy = wx / wl, wy / wl
        dx, dy = uwy, -uwx
        s = cr * inv_dt - wl
        ux, uy = s * uwx, s * uwy
    return (v[0] + resp * ux, v[1] + resp * uy, dx, dy), (ux, uy)


def obstacle_offset(pos, od):
    """computeObstacle's agent - nearest obstacle cell at pos, None outside the grid (as smpc::nearest_obstacle with
    the x >= origin test of the crowd kernels)."""
    if cref.obstacle_cell(pos, od) is None:
        return None
    return pr.compute_obstacle(pos, od)


def neighbours(pos, i, n_agents, rng0, max_neighbors, tie=None):
    """RVO2's neighbour list of agent i among positions pos[:n_agents] (scan order): indices sorted by distSq."""
    tie = tie or _Tie()
    nd, ni = [], []
    rng = rng0
    for j in range(n_agents):
        if j == i:
            continue
        dx, dy = pos[j][0] - pos[i][0], pos[j][1] - pos[i][1]
        d = dx * dx + dy * dy
        tie(d, rng)
        if not d < rng:
            continue
        if len(nd) < max_neighbors:
            nd.append(d)
            ni.append(j)
        k = len(nd) - 1
        while k != 0:
            tie(d, nd[k - 1])
            if not d < nd[k - 1]:
                break
            nd[k], ni[k] = nd[k - 1], ni[k - 1]
            k -= 1
        nd[k], ni[k] = d, j
        if len(nd) == max_neighbors:
            rng = nd[-1]
    return ni


def new_velocity(i, pos, vel, n_people, pref, vmax, obstacle, orca, dts, tie=None):
    """The new velocity of person i (agents pos / vel: people 0 .. n_people-1, then the robots that are agents), its
    obstacle offset (agent - cell or None). Returns (velocity, {robot r: (violated, |u|)})."""
    tie = tie or _Tie()
    o = dict(DEFAULTS, **orca)
    inv_t, inv_to, inv_dt = 1.0 / o["time_horizon"], 1.0 / o["time_horizon_obst"], 1.0 / dts
    pr_ = o["person_radius"]
    vx, vy = vel[i]
    lines = []
    if obstacle is not None:
        rpx, rpy = -obstacle[0], -obstacle[1]
        reach = o["time_horizon_obst"] * vmax + pr_
        tie(rpx * rpx + rpy * rpy, reach * reach)
        if rpx * rpx + rpy * rpy < reach * reach:
            r = orca_line((rpx, rpy), (vx, vy), pr_, inv_to, inv_dt, (vx, vy), 1.0, tie)
            if r is not None:
                lines.append(r[0])
    n_obst = len(lines)
    robots = {}
    for j in neighbours(pos, i, len(pos), o["neighbor_dist"] * o["neighbor_dist"], o["max_neighbors"], tie):
        robot = j >= n_people
        cr = pr_ + (o["robot_radius"] if robot else pr_)
        resp = o["robot_responsibility"] if robot else 0.5
        r = orca_line((pos[j][0] - pos[i][0], pos[j][1] - pos[i][1]), (vx - vel[j][0], vy - vel[j][1]), cr, inv_t,
                      inv_dt, (vx, vy), resp, tie)
        if r is None:
            continue
        line, u = r
        if robot:
            v = _det(line[2], line[3], line[0] - vx, line[1] - vy)
            tie(v)
            robots[j - n_people] = (v > 0.0, math.sqrt(u[0] * u[0] + u[1] * u[1]))
        lines.append(line)
    fail, res = linear_program2(lines, vmax, pref, False, tie)
    if fail < len(lines):
        res = linear_program3(lines, n_obst, fail, vmax, res, tie)
    return res, robots


def crowd_step(people, has_goal, goals, vdes, robots_pose, robots_cmd, od, dt_c, substeps, orca, running=None,
               cos=math.cos, sin=math.sin):
    """One tick of the ORCA crowd of one scene: people [n][5] (x, y, vx, vy, vz), has_goal [n], goals [n][2], vdes [n],
    the R robots' poses [R][3] and commands [R][2] of the tick, od = one grid (crowd_ref.od_of), `substeps` synchronous
    updates of dt_c / substeps, orca = dict of smpc_orca_params fields (missing ones take DEFAULTS); running [R]
    (default all): a finished robot stands still and adds no disturbance; cos / sin of the robots' headings, which the
    caller may take from the device's math library. Returns (people [n][5], has_goal [n],
    disturbance [R], near [n])."""
    o = dict(DEFAULTS, **orca)
    people = np.asarray(people, dtype=np.float64)
    n = people.shape[0]
    R = len(robots_pose)
    running = np.ones(R, bool) if running is None else np.asarray(running, bool)
    dts = dt_c / substeps
    rstate = []
    for r in range(R):
        rx, ry, th = (float(c) for c in robots_pose[r])
        v = float(robots_cmd[r][0]) if running[r] else 0.0
        rstate.append((rx, ry, v * float(cos(th)), v * float(sin(th))))
    n_robots = R if o["robot_responsibility"] > 0.0 else 0
    pos = [[float(p[0]), float(p[1])] for p in people]
    vel = [[float(p[2]), float(p[3])] for p in people]
    vz = [float(p[4]) for p in people]
    yaw = [math.atan2(p[3], p[2]) for p in people]
    goal = [bool(g) for g in has_goal]
    near = np.zeros(n, bool)
    dist = np.zeros(R)
    for s in range(substeps):
        ts = s * dts
        apos = pos + [[rx + ts * rvx, ry + ts * rvy] for rx, ry, rvx, rvy in rstate[:n_robots]]
        avel = vel + [[rvx, rvy] for _, _, rvx, rvy in rstate[:n_robots]]
        nxt = []
        for i in range(n):
            tie = _Tie()
            px, py = pos[i]
            vmax = float(vdes[i])
            pref = (0.0, 0.0)
            if goal[i]:
                dx, dy = float(goals[i][0]) - px, float(goals[i][1]) - py
                z = dx * dx + dy * dy
                if z > 0.0:
                    sq = math.sqrt(z)
                    pref = (vmax * (dx / sq), vmax * (dy / sq))
            res, robots = new_velocity(i, apos, avel, n, pref, vmax, obstacle_offset(pos[i], od), o, dts, tie)
            for r, (violated, ulen) in robots.items():
                if violated and running[r]:
                    dist[r] += o["robot_responsibility"] * ulen * dts
            nvx, nvy = res
            y0 = yaw[i]
            yaw[i] = pr.wrap_pi(math.atan2(nvy, nvx))
            vz[i] = pr.wrap_pi(yaw[i] - y0) / dts
            npx, npy = px + nvx * dts, py + nvy * dts
            if goal[i]:
                dx, dy = float(goals[i][0]) - npx, float(goals[i][1]) - npy
                d = math.sqrt(dx * dx + dy * dy)
                tie(d, GOAL_RADIUS)
                if d <= GOAL_RADIUS:
                    goal[i] = False
            if tie.near:
                # a flip before the last substep moves this person, and so everyone's next lines: mark the scene
                near[:] = near[:] | (s < substeps - 1)
                near[i] = True
            nxt.append((npx, npy, nvx, nvy))
        for i, (npx, npy, nvx, nvy) in enumerate(nxt):
            pos[i], vel[i] = [npx, npy], [nvx, nvy]
    out = np.array([[pos[i][0], pos[i][1], vel[i][0], vel[i][1], vz[i]] for i in range(n)]).reshape(n, 5)
    return out, np.array(goal, dtype=bool), dist, near
