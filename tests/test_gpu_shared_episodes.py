"""GPU tests of the shared-scene episode entry smpc_run_shared_episodes (FleetOptimizer.run_shared_episodes): every
tick is replayed through the public path (trajectorize_batch, filter_people_fov on each robot's scene view,
optimize_batch), the crowd through the numpy reference of tests/shared_ref.py and the world and metrics through
tests/episode_ref.py and tests/crowd_ref.py."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from tests import crowd_ref as cref
from tests import episode_ref as ref
from tests import shared_ref as sref

pytestmark = pytest.mark.gpu

A = 3
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
CROWD_OUT = METRICS + ("people_disturbance",)
SHARED_OUT = CROWD_OUT + ("robot_min_dist", "robot_intimate_ticks")
LOGS = ("pose_log", "cmd_log", "optimized_log", "people_log")
ARG, UNSUP = -1, -3
LAUNCHES_PER_TICK = 15  # documented in DESIGN.md


def _fleet(p, B):
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    return FleetOptimizer(p, n_robots=B, n_agents=A)


def _args(s, **kw):
    a = {k: v for k, v in s.items() if k not in ("params", "ticks")}
    a.update(kw)
    return a


def _run(fleet, s, T, want_logs=True, **kw):
    return fleet.run_shared_episodes(ticks=T, want_logs=want_logs, **_args(s, **kw))


def _device_trig():
    """cos / sin from the device's math library, which the scene view kernel uses."""
    import torch

    def f(fn):
        return lambda x: fn(torch.as_tensor(np.asarray(x, dtype=np.float64), device="cuda")).cpu().numpy()
    return f(torch.cos), f(torch.sin)


def _short(s, b, length):
    """robot b drives only `length` m along its path's direction."""
    N = s["global_path"].shape[1]
    p0, p1 = s["global_path"][b, 0], s["global_path"][b, -1]
    u = (p1 - p0) / np.linalg.norm(p1 - p0)
    s["global_path"][b] = p0 + u * np.linspace(0.0, length, N)[:, None]


def _replay_scenes(R, T, substeps):
    """S = 4 scenes of R robots, K = 6: a people-free scene (0), one robot that arrives early (robot 0 of scene 1)."""
    s = sc.shared_episodes(4, R, 6, seed=11 + R, ticks=T, substeps=substeps)
    s["n_people"][0] = 0
    _short(s, R, 1.0)
    return s


@pytest.mark.parametrize("R", [2, 3])
@pytest.mark.parametrize("substeps", [1, 4])
def test_shared_episodes_replay_through_the_public_path_and_the_numpy_crowd(R, substeps):
    T = 60
    s = _replay_scenes(R, T, substeps)
    p, S, dt_c = s["params"], 4, s["control_period"]
    B = S * R
    fleet, replay = _fleet(p, B), _fleet(p, B)
    cos, sin = _device_trig()
    try:
        got = _run(fleet, s, T)
        pl, cl, ol, ticks, ppl = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"], got["people_log"]
        assert ppl.shape == (S, T + 1, 6, 5)
        H, W = s["costmaps"].shape[1:]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
        flags = [np.ones(int(s["n_people"][c]), bool) for c in range(S)]
        skip = [np.zeros(int(s["n_people"][c]), bool) for c in range(S)]
        dist = np.zeros(B)
        od = cref.od_of(s["od"], 0)
        checked = 0
        for k in range(T):
            pk = pl[:, k]
            act = ~done
            poses, cmds3, n_steps = replay.trajectorize_batch(s["global_path"], pk)
            cmds = np.ascontiguousarray(cmds3[:, :, [0, 2]])
            views, n_view = sref.scene_views(pk, speed, act, ppl[:, k], s["n_people"], R, cos=cos, sin=sin)
            fp, fn = replay.filter_people_fov(views, n_view, pk, s["costmap_origin"], W, H, s["costmap_resolution"],
                                              costmap_index=s["costmap_index"])
            n_poses = np.where(done, 0, n_steps + 1).astype(np.int32)
            r = replay.optimize_batch(poses, cmds, fp, fn, speed, s["costmaps"], s["costmap_origin"],
                                      s["costmap_resolution"], s["od"], costmap_index=s["costmap_index"],
                                      n_poses=n_poses, want_people_proj=False)
            cmd = r["cmds"][:, 0]
            assert np.array_equal(cl[act, k], cmd[act]), k
            assert np.array_equal(ol[act, k], r["optimized"][act]), k
            assert np.all(cl[done, k] == 0.0) and not ol[done, k].any()
            want = ref.euler_step(pk[act], cl[act, k], dt_c)
            assert np.abs(pl[act, k + 1] - want).max() <= 1e-12, k
            assert np.array_equal(pl[done, k + 1], pk[done])
            for c in range(S):
                rb = slice(c * R, c * R + R)
                n = int(s["n_people"][c])
                if done[rb].all():
                    assert np.array_equal(ppl[c, k + 1], ppl[c, k])  # every robot finished: the people stand still
                    continue
                q, flags[c], d, near = sref.crowd_step(ppl[c, k, :n], flags[c], s["goals"][c, :n],
                                                       s["desired_speed"][c, :n], pk[rb], cl[rb, k], act[rb], od,
                                                       dt_c, substeps, near_eps=1e-9)
                skip[c] |= near
                dist[rb] += np.where(act[rb], d, 0.0)
                ok = ~skip[c]
                assert np.abs(ppl[c, k + 1, :n][ok] - q[ok]).max(initial=0.0) <= 1e-12, (k, c)
                checked += int(ok.sum())
            speed[act] = cmd[act]
            done |= ticks == k + 1
        assert checked >= 0.5 * T * int(s["n_people"].sum())
        sc_of = np.arange(B) // R
        m = cref.metrics_from_people_log(pl, cl, ol, ticks, ppl[sc_of], s["n_people"][sc_of], s["global_path"],
                                         s["costmaps"], s["costmap_origin"], s["costmap_resolution"],
                                         s["costmap_index"], 0.25)
        assert np.array_equal(got["reached"], m["reached"])
        assert np.all(ticks[m["reached"]] == m["goal_first"][m["reached"]] + 1)
        assert np.all(ticks[~m["reached"]] == T)
        for k in ("collision_ticks", "not_optimized_ticks"):
            assert np.array_equal(got[k], m[k]), k
        ok = ~m["near_threshold"]
        for k in ("intimate_ticks", "personal_ticks"):
            assert np.array_equal(got[k][ok], m[k][ok]), k
        for k in ("path_length", "min_person_dist", "cmd_variation"):
            assert np.allclose(got[k], m[k], rtol=0, atol=1e-9), k
        assert np.allclose(got["people_disturbance"], dist, rtol=1e-9, atol=1e-300)
        rmin, rint = sref.robot_metrics(pl, ticks, R)
        assert np.array_equal(got["robot_min_dist"], rmin)
        assert np.array_equal(got["robot_intimate_ticks"], rint)
        # the scenes do what they were built for
        assert np.all(got["min_person_dist"][:R] == np.inf)
        assert got["reached"][R] and got["ticks"][R] < T and got["ticks"][R + 1: 2 * R].min() > got["ticks"][R]
        assert np.all(np.isfinite(got["robot_min_dist"]))
    finally:
        fleet.close()
        replay.close()


def test_one_robot_per_scene_is_run_crowd_episodes():
    s = sc.crowd_episodes(8, 6, ticks=60, seed=7, substeps=2)
    fleet = _fleet(s["params"], 8)
    try:
        a = _run(fleet, dict(s, robots_per_scene=1), 60)
        b = fleet.run_crowd_episodes(ticks=60, want_logs=True, **_args(s))
    finally:
        fleet.close()
    for k in CROWD_OUT + LOGS:
        assert np.array_equal(a[k], b[k]), k
    assert np.all(a["robot_min_dist"] == np.inf) and np.all(a["robot_intimate_ticks"] == 0)


def test_robots_that_cannot_see_each_other_change_nothing():
    """K = 0, two robots back to back driving apart: neither is ever in the other's field of view."""
    s = sc.shared_episodes(3, 2, 0, seed=3, ticks=80)
    N = s["global_path"].shape[1]
    for c in range(3):
        x, y = 6.0, 2.0 + 0.1 * c
        for r, sign in ((0, 1.0), (1, -1.0)):
            b = 2 * c + r
            s["global_path"][b, :, 0] = x + sign * (0.3 + np.linspace(0.0, 3.5, N))
            s["global_path"][b, :, 1] = y
            s["pose"][b] = [x + sign * 0.3, y, 0.0 if sign > 0 else np.pi]
    B = 6
    shared, alone = _fleet(s["params"], B), _fleet(s["params"], 1)
    try:
        got = _run(shared, s, 80)
        plain = {k: v for k, v in _args(s).items()
                 if k not in ("goals", "desired_speed", "substeps", "robots_per_scene", "people", "n_people")}
        for b in range(B):
            one = {k: (v[b:b + 1] if k in ("global_path", "pose", "speed", "costmap_index") else v)
                   for k, v in plain.items()}
            want = alone.run_episodes(ticks=80, want_logs=True, people=np.zeros((1, 0, 5)), n_people=[0], **one)
            for k in METRICS + ("pose_log", "cmd_log", "optimized_log"):
                assert np.array_equal(got[k][b], want[k][0]), (b, k)
    finally:
        shared.close()
        alone.close()
    assert np.all(got["robot_min_dist"] >= 0.6) and np.all(got["robot_intimate_ticks"] == 0)


def test_head_on_pair_in_an_empty_corridor():
    s = sc.shared_episodes(4, 2, 0, seed=8, ticks=200)
    fleet = _fleet(s["params"], 8)
    try:
        got = _run(fleet, s, 200, want_logs=False)
    finally:
        fleet.close()
    start = s["pose"].reshape(4, 2, 3)
    sep = np.hypot(start[:, 0, 0] - start[:, 1, 0], start[:, 0, 1] - start[:, 1, 1]).repeat(2)
    assert np.all(np.isfinite(got["robot_min_dist"])) and np.all(got["robot_min_dist"] < sep - 1.0)


def _short_scenes(S, R, K=4):
    """Short paths for everyone, people walking off to the middle of the corridor: all robots arrive early, at
    different ticks. The robots start at both ends (+x robots near x = 1.55, -x robots near x = 10.45), so a goal at
    either end would gather the crowd on some robot's path."""
    s = sc.shared_episodes(S, R, K, seed=5, ticks=400)
    for b in range(S * R):
        _short(s, b, 0.8 + 0.3 * (b % R))
    s["goals"][:, :, 0] = 6.0
    return s


def test_logs_and_early_stop():
    S, R = 4, 2
    s = _short_scenes(S, R)
    fleet = _fleet(s["params"], S * R)
    try:
        long = _run(fleet, s, 400)
        quiet = _run(fleet, s, 400, want_logs=False)
        for k in SHARED_OUT:
            assert np.array_equal(long[k], quiet[k]), k
        assert "people_log" not in quiet
        assert long["reached"].all()
        t_last = int(long["ticks"].max())
        assert t_last < 200
        short = _run(fleet, s, t_last)
        for k in SHARED_OUT:
            assert np.array_equal(long[k], short[k]), k
        for k in ("pose_log", "people_log"):
            assert np.array_equal(long[k][:, : t_last + 1], short[k]), k
        for k in ("cmd_log", "optimized_log"):
            assert np.array_equal(long[k][:, :t_last], short[k]), k
        for c in range(S):
            tb = long["ticks"][c * R: c * R + R]
            assert tb.min() < tb.max()  # one robot finished first: its people kept moving until the other did
            tc = int(tb.max())
            assert not np.array_equal(long["people_log"][c, tc], long["people_log"][c, int(tb.min())])
            assert np.all(long["people_log"][c, tc:] == long["people_log"][c, tc:tc + 1])
        assert np.array_equal(long["people_log"][:, 0], s["people"])
    finally:
        fleet.close()


def test_shared_episodes_leave_the_fleet_tick_memory_alone():
    s = sc.shared_episodes(3, 2, 5, ticks=20, seed=9)
    B = 6
    p = s["params"]
    poses, cmds = sc.pure_pursuit_seed(s["global_path"], s["pose"], p)
    people = np.ascontiguousarray(s["people"][np.arange(B) // 2, :A])
    n_people = np.full(B, A, np.int32)
    maps = (s["costmaps"], s["costmap_origin"], s["costmap_resolution"], s["od"])

    def tick(fl):
        return fl.optimize_batch(poses, cmds, people, n_people, s["speed"], *maps, costmap_index=s["costmap_index"])

    a, b = _fleet(p, B), _fleet(p, B)
    try:
        a1 = tick(a)
        _run(a, s, 20, want_logs=False)
        a2 = tick(a)
        b1, b2 = tick(b), tick(b)
        for x, y in ((a1, b1), (a2, b2)):
            for k in ("cmds", "path", "optimized", "n_out", "termination", "cost_final"):
                assert np.array_equal(x[k], y[k]), k
    finally:
        a.close()
        b.close()


@pytest.mark.parametrize("R,K", [(2, 6), (3, 0), (1, 6)])
def test_launches_per_tick(R, K):
    s = sc.shared_episodes(4, R, K, ticks=3, seed=4)
    fleet = _fleet(s["params"], 4 * R)
    try:
        counts = {}
        for T in (1, 3):
            c0 = fleet.opt.launch_count()
            _run(fleet, s, T, want_logs=False)
            counts[T] = fleet.opt.launch_count() - c0
    finally:
        fleet.close()
    assert counts[1] == LAUNCHES_PER_TICK and counts[3] == 3 * LAUNCHES_PER_TICK, counts


def test_shared_argument_errors_launch_nothing():
    S, R = 3, 2
    B = S * R
    s = sc.shared_episodes(S, R, 5, ticks=10, seed=4)
    p = s["params"]

    def raw(fleet, crowd_fields=None, scene_fields=None, null_crowd=False, null_scene=False, n_episodes=None, **kw):
        a = {k: v for k, v in _args(s, **kw).items() if k not in ("goals", "desired_speed", "substeps",
                                                                  "robots_per_scene")}
        io, out, logs, keep = fleet.episode_io(**a, ticks=10, robots_per_scene=R)
        if n_episodes is not None:
            io.n_episodes = n_episodes
        goals = np.ascontiguousarray(kw.get("goals", s["goals"]), dtype=np.float64)
        vdes = np.ascontiguousarray(kw.get("desired_speed", s["desired_speed"]), dtype=np.float64)
        dist, rmin, rint = np.zeros(B), np.zeros(B), np.zeros(B, np.int32)
        crowd = abi.SmpcCrowdIo(goals.ctypes.data, vdes.ctypes.data, 1, dist.ctypes.data, None)
        scene = abi.SmpcSceneIo(R, rmin.ctypes.data, rint.ctypes.data)
        for f, v in (crowd_fields or {}).items():
            setattr(crowd, f, v)
        for f, v in (scene_fields or {}).items():
            setattr(scene, f, v)
        c0 = fleet.opt.launch_count()
        rc = _lib.lib().smpc_run_shared_episodes(fleet.opt._h, C.byref(io), None if null_crowd else C.byref(crowd),
                                                 None if null_scene else C.byref(scene))
        if rc != 0:
            assert fleet.opt.launch_count() == c0
        return rc

    for bad, code in ((dict(omni_solve=1), UNSUP), (dict(omnidirectional=1), UNSUP)):
        fleet = _fleet(sc.make_params("soc_work_obst", **bad), B)
        try:
            assert raw(fleet) == code
        finally:
            fleet.close()
    fleet = _fleet(p, B)
    try:
        assert raw(fleet, null_scene=True) == ARG
        assert raw(fleet, null_crowd=True) == ARG
        for r in (0, 9, 4):  # outside 1..8; 4 does not divide 6
            assert raw(fleet, scene_fields=dict(robots_per_scene=r)) == ARG
        assert raw(fleet, n_episodes=5) == ARG  # not a multiple of R
        assert raw(fleet, scene_fields=dict(robot_min_dist=None)) == ARG
        assert raw(fleet, scene_fields=dict(robot_intimate_ticks=None)) == ARG
        assert raw(fleet, crowd_fields=dict(people_disturbance=None)) == ARG
        assert raw(fleet, crowd_fields=dict(goals=None)) == ARG
        assert raw(fleet, crowd_fields=dict(substeps=0)) == ARG
        K = 63  # people + 2 robots above the kernel's 64 agent slots
        wide = np.zeros((S, K, 5))
        wide[:, :5] = s["people"]
        assert raw(fleet, people=wide, goals=np.zeros((S, K, 2)) + 2.0, desired_speed=np.ones((S, K))) == ARG
        ci = s["costmap_index"].copy()
        ci[1] = (ci[0] + 1) % s["costmaps"].shape[0]
        assert raw(fleet, costmap_index=ci) == ARG
        assert raw(fleet, od_index=np.array([0, 1, 0, 0, 0, 0], np.int32)) == ARG  # also outside the one grid
        od2 = dict(s["od"], origins=np.zeros((2, 2)), indexes=np.tile(np.asarray(s["od"]["indexes"]), 2))
        assert raw(fleet, od=od2, od_index=np.array([0, 1, 0, 0, 1, 1], np.int32)) == ARG
        assert raw(fleet, od=od2, od_index=None) == ARG  # NULL: robot b uses grid b % 2, which differs in a scene
        bad_n = s["n_people"].copy()
        bad_n[2] = 6
        assert raw(fleet, n_people=bad_n) == ARG
        g = s["goals"].copy()
        g[1, 2] = np.nan
        assert raw(fleet, goals=g) == ARG
        assert raw(fleet, goal_tolerance=0.15) == ARG
        assert raw(fleet) == 0  # the block as built is valid
        assert raw(fleet, od=od2, od_index=np.array([0, 0, 1, 1, 0, 0], np.int32)) == 0
    finally:
        fleet.close()
