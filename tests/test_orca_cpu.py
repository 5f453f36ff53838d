"""CPU tests of the ORCA crowd (smpc_run_orca_episodes): its parameter block mirrors include/smpc.h, the numpy
restatement the GPU tests compare with (tests/orca_ref.py) solves its linear programs as scipy does, and its people
behave as ORCA people should in hand-built scenes."""
import math
import os
import re

import numpy as np
import pytest
from scipy.optimize import minimize

from nav2_social_mpc_controller_b200 import abi, scenarios as sc
from tests import crowd_ref as cref
from tests import orca_ref as oref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_OD = dict(width=1, height=1, resolution=0.05, origin_x=1000.0, origin_y=1000.0,
             indexes=np.zeros(1, dtype=np.uint32))  # every position lies outside this grid: no obstacle


def test_orca_params_field_order_and_defaults_match_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_orca_params \{(.*?)\} smpc_orca_params;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [d.strip().split()[-1] for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in abi.SmpcOrcaParams._fields_]
    assert re.search(r"int smpc_run_orca_episodes\(smpc_handle\* h, smpc_episode_io\* io, const smpc_crowd_io\* crowd,",
                     hdr)
    p = abi.orca_params()
    assert {f: getattr(p, f) for f, _ in abi.SmpcOrcaParams._fields_} == oref.DEFAULTS
    assert abi.orca_params(max_neighbors=3).max_neighbors == 3
    with pytest.raises(TypeError):
        abi.orca_params(radius=0.2)


def _violation(line, v):
    px, py, dx, dy = line
    return dx * (py - v[1]) - dy * (px - v[0])  # det(dir, point - v) > 0: v violates the line


def _feasible_lines(rng, n, radius):
    """n lines that all admit a point f inside the circle: point = f - margin * left normal, so det(dir, point - f) < 0."""
    f = rng.uniform(-0.5, 0.5, 2) * radius
    lines = []
    for _ in range(n):
        a = rng.uniform(-math.pi, math.pi)
        dx, dy = math.cos(a), math.sin(a)
        m, t = rng.uniform(0.01, 0.5), rng.uniform(-1.0, 1.0)
        lines.append((f[0] + t * dx + m * dy, f[1] + t * dy - m * dx, dx, dy))
    return lines


def _cons(lines):
    return [dict(type="ineq", fun=lambda v, l=l: -_violation(l, v)) for l in lines]


def _solved(r, cons):
    """SLSQP ended at a feasible point; it may stop at the optimum with "positive directional derivative" (status 8)."""
    return r.status in (0, 8) and min(c["fun"](r.x) for c in cons) >= -1e-10


def test_lp2_finds_the_nearest_feasible_point():
    rng = np.random.default_rng(1)
    for trial in range(200):
        radius = rng.uniform(0.5, 1.5)
        lines = _feasible_lines(rng, int(rng.integers(1, 18)), radius)
        pref = rng.uniform(-1.5, 1.5, 2) * radius
        fail, v = oref.linear_program2(lines, radius, tuple(pref), False)
        assert fail == len(lines), trial
        assert max(_violation(l, v) for l in lines) <= 1e-12, trial
        assert v[0] * v[0] + v[1] * v[1] <= radius * radius * (1 + 1e-12)
        cons = _cons(lines) + [dict(type="ineq", fun=lambda x: radius * radius - x @ x)]
        best = None
        for x0 in ([0.0, 0.0], list(v), list(pref)):
            r = minimize(lambda x: (x - pref) @ (x - pref), x0, jac=lambda x: 2 * (x - pref), constraints=cons,
                         method="SLSQP", options=dict(ftol=1e-15, maxiter=500))
            if _solved(r, cons) and (best is None or r.fun < best.fun):
                best = r
        assert best is not None
        assert np.hypot(*(np.asarray(v) - best.x)) <= 1e-7, (trial, v, best.x)


def test_lp3_minimises_the_largest_violation_of_the_soft_lines():
    rng = np.random.default_rng(2)
    checked = 0
    for trial in range(300):
        radius = rng.uniform(0.5, 1.5)
        n_obst = int(rng.integers(0, 2))
        hard = _feasible_lines(rng, n_obst, radius)
        soft = []
        for _ in range(int(rng.integers(3, 17))):  # half-planes {n . v >= d}, n = (-sin a, cos a), in all directions
            a = rng.uniform(-math.pi, math.pi)
            d = rng.uniform(0.2, 1.5) * radius
            soft.append((-d * math.sin(a), d * math.cos(a), math.cos(a), math.sin(a)))
        lines = hard + soft
        pref = tuple(rng.uniform(-1.0, 1.0, 2) * radius)
        fail, v = oref.linear_program2(lines, radius, pref, False)
        if fail == len(lines):
            continue
        v = oref.linear_program3(lines, n_obst, fail, radius, v)
        got = max(_violation(l, v) for l in soft)
        assert all(_violation(l, v) <= 1e-12 for l in hard), trial
        assert v[0] * v[0] + v[1] * v[1] <= radius * radius * (1 + 1e-12)
        # scipy: min t subject to det(dir, point - v) <= t (soft), <= 0 (hard), |v| <= radius
        cons = [dict(type="ineq", fun=lambda x, l=l: x[2] - _violation(l, x[:2])) for l in soft]
        cons += [dict(type="ineq", fun=lambda x, l=l: -_violation(l, x[:2])) for l in hard]
        cons += [dict(type="ineq", fun=lambda x: radius * radius - x[:2] @ x[:2])]
        best = None
        for x0 in ([0.0, 0.0], list(v)):
            t0 = max(_violation(l, x0) for l in soft) + 0.1
            r = minimize(lambda x: x[2], x0 + [t0], jac=lambda x: np.array([0.0, 0.0, 1.0]), constraints=cons,
                         method="SLSQP", options=dict(ftol=1e-15, maxiter=1000))
            if _solved(r, cons) and (best is None or r.fun < best.fun):
                best = r
        assert best is not None
        assert got > 0.0
        assert abs(got - best.fun) <= 1e-7, (trial, got, best.fun)
        checked += 1
    assert checked >= 100


def _swap(T=200):
    """Two people swapping ends of 6 m of open space head-on, 0.1 m apart laterally, at 1.0 and 0.8 m/s."""
    people = np.array([[0.0, 0.05, 1.0, 0.0, 0.0], [6.0, -0.05, -0.8, 0.0, 0.0]])
    goals = np.array([[6.0, 0.05], [0.0, -0.05]])
    vdes = np.array([1.0, 0.8])
    flags = np.ones(2, bool)
    dmin = np.inf
    for _ in range(T):
        people, flags, _, _ = oref.crowd_step(people, flags, goals, vdes, [], [], NO_OD, 0.05, 1, {})
        dmin = min(dmin, float(np.hypot(*(people[0, :2] - people[1, :2]))))
    return people, flags, dmin


def test_two_people_swapping_head_on_pass_without_touching():
    people, flags, dmin = _swap()
    assert not flags.any()  # both reached (and cleared) their goals
    assert np.all(np.hypot(people[:, 0] - [6.0, 0.0], people[:, 1] - [0.05, -0.05]) <= 0.25)
    # ORCA picks velocities outside each other's truncated velocity obstacle, so the positions after each step keep
    # 2 r apart up to the rounding of the linear programs: the run comes within ~1e-15 of 0.6 m (the two glide along
    # each other's leg) and never below by more than 1e-9.
    assert dmin >= 2 * 0.3 - 1e-9, dmin
    assert dmin < 0.7  # they did come close: the scene tests avoidance


def test_mirror_symmetric_scene_stays_mirror_symmetric():
    """People i and i + n are mirror images about y = 0 (negation is exact, so rounding cannot break the symmetry),
    and so is the robot on the axis driving along it. The halves stay farther apart than neighbor_dist: a person and
    its own mirror image would meet exactly head-on, where ORCA (like RVO2) takes the right leg on both sides, which is
    point-symmetric, not mirror-symmetric."""
    rng = np.random.default_rng(4)
    n = 5
    xy = np.stack([rng.uniform(1.0, 8.0, n), rng.uniform(1.1, 2.0, n)], axis=1)
    v = rng.uniform(-0.6, 0.6, (n, 2))
    g = np.stack([rng.uniform(1.0, 8.0, n), rng.uniform(1.1, 2.0, n)], axis=1)
    mirror = lambda a: np.stack([a[:, 0], -a[:, 1]], axis=1)  # noqa: E731
    people = np.zeros((2 * n, 5))
    people[:n, :2], people[n:, :2] = xy, mirror(xy)
    people[:n, 2:4], people[n:, 2:4] = v, v * [1.0, -1.0]
    goals = np.concatenate([g, mirror(g)])
    vdes = np.tile(rng.uniform(0.5, 1.2, n), 2)
    flags = np.ones(2 * n, bool)
    for _ in range(40):
        people, flags, _, _ = oref.crowd_step(people, flags, goals, vdes, [[3.0, 0.0, 0.0]], [[0.5, 0.0]], NO_OD,
                                              0.05, 2, dict(max_neighbors=6, neighbor_dist=2.0))
        a, b = people[:n], people[n:]
        assert np.abs(a[:, 0] - b[:, 0]).max() <= 1e-12
        assert np.abs(a[:, 1] + b[:, 1]).max() <= 1e-12
        assert np.abs(a[:, 2] - b[:, 2]).max() <= 1e-12 and np.abs(a[:, 3] + b[:, 3]).max() <= 1e-12
        assert np.array_equal(flags[:n], flags[n:])
        assert np.abs(people[:n, 1] - people[n:, 1]).min() > 2.0  # the halves never became neighbours


def test_zero_responsibility_makes_the_robot_invisible():
    s = sc.crowd_episodes(3, 9, seed=2, ticks=10)
    od = cref.od_of(s["od"], 0)
    for b in range(3):
        p, f = s["people"][b], np.ones(9, bool)
        q, fq = p, f
        for k in range(10):
            robot = [s["pose"][b] + [0.1 * k, 0.0, 0.0]]
            p, f, d, _ = oref.crowd_step(p, f, s["goals"][b], s["desired_speed"][b], robot, [[0.5, 0.2]], od, 0.05, 2,
                                         dict(robot_responsibility=0.0))
            q, fq, _, _ = oref.crowd_step(q, fq, s["goals"][b], s["desired_speed"][b], [], [], od, 0.05, 2, {})
            assert np.array_equal(p, q) and np.array_equal(f, fq) and np.all(d == 0.0)


def test_a_robot_in_the_way_is_avoided_and_counts_as_disturbance():
    """A person walking at a robot that drives at it: with responsibility the person swerves and the robot's line
    was violated; the disturbance grows with the person's share."""
    people = np.array([[3.0, 0.0, -1.0, 0.0, 0.0]])
    out = {}
    for resp in (0.0, 0.5, 1.0):
        p, f = people, np.ones(1, bool)
        dist = 0.0
        for k in range(20):
            p, f, d, _ = oref.crowd_step(p, f, [[-3.0, 0.0]], [1.0], [[0.02 * k, 0.02, 0.0]], [[0.4, 0.0]], NO_OD,
                                         0.05, 1, dict(robot_responsibility=resp))
            dist += d[0]
        out[resp] = (p, dist)
    assert out[0.0][1] == 0.0 and abs(out[0.0][0][0, 1]) == 0.0  # straight on
    assert out[0.5][1] > 0.0 and out[1.0][1] > 0.0
    assert abs(out[0.5][0][0, 1]) > 0.05 and abs(out[1.0][0][0, 1]) > abs(out[0.5][0][0, 1])


def test_crowd_scenes_clear_two_orca_radii():
    """The scenes of crowd_episodes / shared_episodes start every person CROWD_SPACING = 0.7 m from the others and
    CROWD_CLEARANCE = 0.6 m from robots and lethal cells: no ORCA pair (2 x 0.3 m) starts in collision."""
    assert sc.CROWD_SPACING > 2 * oref.DEFAULTS["person_radius"]
    assert sc.CROWD_CLEARANCE >= oref.DEFAULTS["person_radius"] + oref.DEFAULTS["robot_radius"]
    for s, R in ((sc.crowd_episodes(64, 20, seed=3), 1), (sc.shared_episodes(16, 2, 20, seed=3), 2)):
        xy = s["people"][..., :2]
        d = np.hypot(xy[:, :, None, 0] - xy[:, None, :, 0], xy[:, :, None, 1] - xy[:, None, :, 1])
        d[:, np.arange(20), np.arange(20)] = np.inf
        assert d.min() >= 0.6
        robots = s["pose"].reshape(-1, R, 3)[..., :2]
        dr = np.hypot(xy[:, :, None, 0] - robots[:, None, :, 0], xy[:, :, None, 1] - robots[:, None, :, 1])
        assert dr.min() >= 0.6
