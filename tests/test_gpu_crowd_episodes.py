"""GPU tests of the reactive-crowd episode entry smpc_run_crowd_episodes (FleetOptimizer.run_crowd_episodes): every
tick is replayed through the public path (trajectorize_batch, filter_people_fov on the logged people, optimize_batch),
the crowd through the numpy reference of tests/crowd_ref.py and the world and metrics through tests/episode_ref.py."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from tests import crowd_ref as cref
from tests import episode_ref as ref

pytestmark = pytest.mark.gpu

A = 3
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
ARG, UNSUP = -1, -3


def _fleet(p, B):
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    return FleetOptimizer(p, n_robots=B, n_agents=A)


def _path(B, N, x0, y0, length):
    path = np.zeros((B, N, 2))
    path[:, :, 0] = x0 + np.linspace(0.0, length, N)[None, :]
    path[:, :, 1] = y0
    return path


def _args(s, **kw):
    a = {k: v for k, v in s.items() if k not in ("params", "ticks")}
    a.update(kw)
    return a


def _run(fleet, s, T, want_logs=True, **kw):
    return fleet.run_crowd_episodes(ticks=T, want_logs=want_logs, **_args(s, **kw))


def _replay_scenes(T, substeps):
    """B = 8, K = 6: a people-free episode (0), one that reaches its goal early (1), a person walking head-on at the
    robot (2), the rest from the crowd generator."""
    s = sc.crowd_episodes(8, 6, ticks=T, n_maps=2, seed=11, substeps=substeps)
    N = s["global_path"].shape[1]
    s["n_people"][0] = 0
    s["global_path"][1] = _path(1, N, 1.0, 2.0, 1.0)[0]
    s["pose"][1] = [1.0, 2.0, 0.0]
    s["pose"][2] = [1.0, 2.0, 0.0]
    s["people"][2, 0] = [2.4, 2.0, -0.6, 0.0, 0.0]  # head-on along the robot's track
    s["goals"][2, 0] = [1.6, 2.0]
    s["desired_speed"][2, 0] = 0.6
    return s


@pytest.mark.parametrize("substeps", [1, 4])
def test_crowd_episodes_replay_through_the_public_path_and_the_numpy_crowd(substeps):
    T = 60
    s = _replay_scenes(T, substeps)
    p, B, dt_c = s["params"], 8, s["control_period"]
    fleet, replay = _fleet(p, B), _fleet(p, B)
    try:
        got = _run(fleet, s, T)
        pl, cl, ol, ticks, ppl = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"], got["people_log"]
        H, W = s["costmaps"].shape[1:]
        n_od = np.asarray(s["od"]["origins"]).reshape(-1, 2).shape[0]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
        flags = [np.ones(int(s["n_people"][b]), bool) for b in range(B)]
        skip = [np.zeros(int(s["n_people"][b]), bool) for b in range(B)]
        dist = np.zeros(B)
        checked = 0
        for k in range(T):
            pk = pl[:, k]
            poses, cmds3, n_steps = replay.trajectorize_batch(s["global_path"], pk)
            cmds = np.ascontiguousarray(cmds3[:, :, [0, 2]])
            fp, fn = replay.filter_people_fov(ppl[:, k], s["n_people"], pk, s["costmap_origin"], W, H,
                                              s["costmap_resolution"], costmap_index=s["costmap_index"])
            n_poses = np.where(done, 0, n_steps + 1).astype(np.int32)
            r = replay.optimize_batch(poses, cmds, fp, fn, speed, s["costmaps"], s["costmap_origin"],
                                      s["costmap_resolution"], s["od"], costmap_index=s["costmap_index"],
                                      n_poses=n_poses, want_people_proj=False)
            act = ~done
            cmd = r["cmds"][:, 0]
            assert np.array_equal(cl[act, k], cmd[act]), k
            assert np.array_equal(ol[act, k], r["optimized"][act]), k
            assert np.all(cl[done, k] == 0.0) and not ol[done, k].any()
            want = ref.euler_step(pk[act], cl[act, k], dt_c)
            assert np.abs(pl[act, k + 1] - want).max() <= 1e-12, k
            assert np.array_equal(pl[done, k + 1], pk[done])
            for b in range(B):
                n = int(s["n_people"][b])
                if done[b]:
                    assert np.array_equal(ppl[b, k + 1], ppl[b, k])  # finished: the people stand still
                    continue
                q, flags[b], d, near = cref.crowd_step(ppl[b, k, :n], flags[b], s["goals"][b, :n],
                                                       s["desired_speed"][b, :n], pk[b], cl[b, k],
                                                       cref.od_of(s["od"], b % n_od), dt_c, substeps, near_eps=1e-9)
                skip[b] |= near
                dist[b] += d
                ok = ~skip[b]
                assert np.abs(ppl[b, k + 1, :n][ok] - q[ok]).max(initial=0.0) <= 1e-12, (k, b)
                assert np.array_equal(ppl[b, k + 1, n:], ppl[b, k, n:])
                checked += int(ok.sum())
            speed[act] = cmd[act]
            done |= ticks == k + 1
        assert checked >= 0.5 * T * int(s["n_people"].sum())
        m = cref.metrics_from_people_log(pl, cl, ol, ticks, ppl, s["n_people"], s["global_path"], s["costmaps"],
                                         s["costmap_origin"], s["costmap_resolution"], s["costmap_index"], 0.25)
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
        # the scenes do what they were built for
        assert got["min_person_dist"][0] == np.inf and got["people_disturbance"][0] == 0.0
        assert got["reached"][1] and got["ticks"][1] < T
        # the robot's pair force is positive at any range (exp does not underflow here): a head-on encounter must
        # make it count
        assert got["min_person_dist"][2] < 1.2 and got["people_disturbance"][2] > 1e-3
    finally:
        fleet.close()
        replay.close()


def test_without_people_the_crowd_entry_is_run_episodes():
    s = sc.crowd_episodes(6, 0, ticks=40, seed=2)
    fleet = _fleet(s["params"], 6)
    try:
        a = _run(fleet, s, 40)
        plain = {k: v for k, v in _args(s).items() if k not in ("goals", "desired_speed", "substeps")}
        b = fleet.run_episodes(ticks=40, want_logs=True, **plain)
    finally:
        fleet.close()
    for k in METRICS + ("pose_log", "cmd_log", "optimized_log"):
        assert np.array_equal(a[k], b[k]), k
    assert np.all(a["people_disturbance"] == 0.0) and a["people_log"].shape == (6, 41, 0, 5)


def test_one_more_launch_per_tick_than_run_episodes():
    s = sc.crowd_episodes(8, 6, ticks=3, seed=4)
    plain = {k: v for k, v in _args(s).items() if k not in ("goals", "desired_speed", "substeps")}
    fleet = _fleet(s["params"], 8)
    try:
        counts = {}
        for T in (1, 3):
            c0 = fleet.opt.launch_count()
            fleet.run_episodes(ticks=T, want_logs=False, **plain)
            c1 = fleet.opt.launch_count()
            _run(fleet, s, T, want_logs=False)
            counts[T] = (c1 - c0, fleet.opt.launch_count() - c1)
    finally:
        fleet.close()
    for T, (plain_n, crowd_n) in counts.items():
        assert crowd_n == plain_n + T, counts
    assert counts[3] == (3 * counts[1][0], 3 * counts[1][1]), counts  # every launch belongs to a tick


def _short_scenes(B, K=4):
    """1.2 m paths; every person walks off to the far end of the corridor, so all robots arrive early."""
    s = sc.crowd_episodes(B, K, ticks=400, seed=5)
    N = s["global_path"].shape[1]
    s["global_path"][:] = _path(B, N, 1.0, 2.0, 1.2)
    s["pose"][:, 1] = 2.0
    s["goals"][:, :, 0] = 10.0
    return s


def test_logs_and_early_stop():
    B = 8
    s = _short_scenes(B)
    fleet = _fleet(s["params"], B)
    try:
        long = _run(fleet, s, 400)
        quiet = _run(fleet, s, 400, want_logs=False)
        for k in METRICS + ("people_disturbance",):
            assert np.array_equal(long[k], quiet[k]), k
        assert "people_log" not in quiet
        assert long["reached"].all()
        t_last = int(long["ticks"].max())
        assert t_last < 200
        short = _run(fleet, s, t_last)
        for k in METRICS + ("people_disturbance",):
            assert np.array_equal(long[k], short[k]), k
        assert np.array_equal(long["people_log"][:, : t_last + 1], short["people_log"])
        assert np.array_equal(long["pose_log"][:, : t_last + 1], short["pose_log"])
        for b in range(B):
            tb = int(long["ticks"][b])
            assert np.all(long["people_log"][b, tb:] == long["people_log"][b, tb:tb + 1])
        assert np.array_equal(long["people_log"][:, 0], s["people"])
    finally:
        fleet.close()


def test_crowd_episodes_leave_the_fleet_tick_memory_alone():
    B = 6
    s = sc.crowd_episodes(B, 5, ticks=20, seed=9)
    p = s["params"]
    poses, cmds = sc.pure_pursuit_seed(s["global_path"], s["pose"], p)
    people = np.ascontiguousarray(s["people"][:, :A])
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


def test_crowd_argument_errors_launch_nothing():
    B = 4
    s = sc.crowd_episodes(B, 5, ticks=10, seed=4)
    p = s["params"]

    def expect(fleet, code, T=10, **kw):
        c0 = fleet.opt.launch_count()
        with pytest.raises(_lib.SmpcError) as e:
            _run(fleet, s, T, want_logs=False, **kw)
        assert e.value.code == code, kw
        assert fleet.opt.launch_count() == c0

    def raw(fleet, crowd_fields=None, null_crowd=False, **kw):
        io, out, logs, keep = fleet.episode_io(**{k: v for k, v in _args(s, **kw).items()
                                                   if k not in ("goals", "desired_speed", "substeps")}, ticks=10)
        goals = np.ascontiguousarray(s["goals"])
        vdes = np.ascontiguousarray(s["desired_speed"])
        dist = np.zeros(B)
        crowd = abi.SmpcCrowdIo(goals.ctypes.data, vdes.ctypes.data, 1, dist.ctypes.data, None)
        for f, v in (crowd_fields or {}).items():
            setattr(crowd, f, v)
        c0 = fleet.opt.launch_count()
        rc = _lib.lib().smpc_run_crowd_episodes(fleet.opt._h, C.byref(io), None if null_crowd else C.byref(crowd))
        assert fleet.opt.launch_count() == c0
        return rc

    for bad, code in ((dict(omni_solve=1), UNSUP), (dict(omnidirectional=1), UNSUP),
                      (dict(max_time=0.1, time_step=0.05), ARG)):
        fleet = _fleet(sc.make_params("soc_work_obst", **bad), B)
        try:
            expect(fleet, code)
        finally:
            fleet.close()
    fleet = _fleet(p, B)
    try:
        assert raw(fleet, null_crowd=True) == ARG
        assert raw(fleet, dict(goals=None)) == ARG
        assert raw(fleet, dict(desired_speed=None)) == ARG
        assert raw(fleet, dict(people_disturbance=None)) == ARG
        for n in (0, 65):
            expect(fleet, ARG, substeps=n)
        K = 64  # people + robot above the kernel's 64 agent slots
        wide = np.zeros((B, K, 5))
        wide[:, :5] = s["people"]
        goals = np.zeros((B, K, 2)) + 2.0
        vd = np.ones((B, K))
        expect(fleet, ARG, people=wide, goals=goals, desired_speed=vd)
        for field, val in (("goals", np.nan), ("goals", np.inf), ("desired_speed", 0.0), ("desired_speed", -0.5),
                           ("desired_speed", np.inf), ("desired_speed", np.nan)):
            bad = s[field].copy()
            bad[1, 2] = val
            expect(fleet, ARG, **{field: bad})
        expect(fleet, ARG, T=0)
        expect(fleet, ARG, goal_tolerance=0.15)
        bad_n = s["n_people"].copy()
        bad_n[2] = 6
        expect(fleet, ARG, n_people=bad_n)
        # beyond n_people_each nothing is read: padding may hold anything
        n = s["n_people"].copy()
        n[1] = 2
        g, v = s["goals"].copy(), s["desired_speed"].copy()
        g[1, 3], v[1, 4] = np.nan, 0.0
        got = _run(fleet, s, 2, want_logs=False, n_people=n, goals=g, desired_speed=v)
        assert np.all(np.isfinite(got["people_disturbance"]))
    finally:
        fleet.close()


def test_generated_crowds_stay_inside_the_obstacle_grid():
    s = sc.crowd_episodes(64, 20, ticks=200)
    fleet = _fleet(s["params"], 64)
    try:
        got = _run(fleet, s, 200)
    finally:
        fleet.close()
    od = s["od"]
    xy = got["people_log"][..., :2]
    assert np.all(np.isfinite(got["people_log"]))
    assert xy[..., 0].min() >= 0.0 and xy[..., 0].max() < od["width"] * od["resolution"]
    assert xy[..., 1].min() >= 0.0 and xy[..., 1].max() < od["height"] * od["resolution"]
    v = np.linalg.norm(got["people_log"][..., 2:4], axis=-1)
    assert np.all(v <= s["desired_speed"][:, None, :] + 1e-12)
    assert np.all(got["people_disturbance"] > 1e-3)  # every robot drives through its crowd
