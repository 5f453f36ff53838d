"""GPU tests of the closed-loop episode entry smpc_run_episodes (FleetOptimizer.run_episodes): every tick is replayed
through the existing public path (trajectorize_batch, filter_people_fov, optimize_batch) and the world and metrics
through the numpy reference of tests/episode_ref.py."""
import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, scenarios as sc
from tests import episode_ref as ref

pytestmark = pytest.mark.gpu

A = 3
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")


def _path(B, N, x0, y0, length):
    path = np.zeros((B, N, 2))
    path[:, :, 0] = x0 + np.linspace(0.0, length, N)[None, :]
    path[:, :, 1] = y0
    return path


def _replay_scenes(T=60):
    """B = 8, K = 6, two costmaps: a people-free episode (0), one that reaches its goal early (1), a close crossing (2),
    a person who walks out of the obstacle grid (3), the rest from the episode generator."""
    s = sc.episodes(8, 6, ticks=T, n_maps=2, seed=11)
    N = s["global_path"].shape[1]
    s["n_people"][0] = 0
    s["global_path"][1] = _path(1, N, 1.0, 2.0, 1.0)[0]
    s["pose"][1] = [1.0, 2.0, 0.0]
    s["people"][2, 0] = [2.0, 1.3, 0.0, 0.4, 0.0]  # crosses the robot's track about 1.7 s in
    s["pose"][2] = [1.0, 2.0, 0.0]
    s["people"][3, 0] = [3.2, 3.8, 0.0, 0.3, 0.0]  # in view beyond the wall, leaves the 4 m grid when projected
    s["pose"][3] = [1.0, 2.0, 0.0]
    return s


def _run(fleet, s, T, want_logs=True, **kw):
    args = {k: v for k, v in s.items() if k not in ("params", "ticks")}
    args.update(kw)
    return fleet.run_episodes(ticks=T, want_logs=want_logs, **args)


def test_episodes_replay_bit_identical_through_the_public_path():
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    T = 60
    s = _replay_scenes(T)
    p, B, dt_c = s["params"], 8, s["control_period"]
    fleet = FleetOptimizer(p, n_robots=B, n_agents=A)
    replay = FleetOptimizer(p, n_robots=B, n_agents=A)
    try:
        got = _run(fleet, s, T)
        pl, cl, ol, ticks = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"]
        H, W = s["costmaps"].shape[1:]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
        for k in range(T):
            pk = pl[:, k]
            poses, cmds3, n_steps = replay.trajectorize_batch(s["global_path"], pk)
            cmds = np.ascontiguousarray(cmds3[:, :, [0, 2]])
            fp, fn = replay.filter_people_fov(ref.people_at(s["people"], k * dt_c), s["n_people"], pk,
                                              s["costmap_origin"], W, H, s["costmap_resolution"],
                                              costmap_index=s["costmap_index"])
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
            speed[act] = cmd[act]
            done |= ticks == k + 1
        m = ref.metrics_from_logs(pl, cl, ol, ticks, s["people"], s["n_people"], s["global_path"], s["costmaps"],
                                  s["costmap_origin"], s["costmap_resolution"], s["costmap_index"], dt_c, 0.25)
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
        # the scenes do what they were built for
        assert got["min_person_dist"][0] == np.inf and got["personal_ticks"][0] == 0
        assert got["reached"][1] and got["ticks"][1] < T
        assert got["min_person_dist"][2] < 1.2
        assert got["not_optimized_ticks"][3] > 0
    finally:
        fleet.close()
        replay.close()


def test_episode_metrics_do_not_depend_on_the_logs():
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    s = sc.episodes(16, 8, ticks=40, seed=3)
    fleet = FleetOptimizer(s["params"], n_robots=16, n_agents=A)
    try:
        a = _run(fleet, s, 40, want_logs=True)
        b = _run(fleet, s, 40, want_logs=False)
        for k in METRICS:
            assert np.array_equal(a[k], b[k]), k
        assert "pose_log" not in b
    finally:
        fleet.close()


def _short_scenes(B, K=2):
    s = sc.episodes(B, K, ticks=400, seed=5)
    N = s["global_path"].shape[1]
    s["global_path"][:] = _path(B, N, 1.0, 2.0, 1.2)
    s["pose"][:, 1] = 2.0
    return s


def test_early_stop_gives_the_results_of_the_last_arrival_tick():
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    B = 8
    s = _short_scenes(B)
    fleet = FleetOptimizer(s["params"], n_robots=B, n_agents=A)
    try:
        c0 = fleet.opt.launch_count()
        _run(fleet, s, 1, want_logs=False)
        per_tick = fleet.opt.launch_count() - c0
        c1 = fleet.opt.launch_count()
        long = _run(fleet, s, 400)
        used = fleet.opt.launch_count() - c1
        assert long["reached"].all()
        t_last = int(long["ticks"].max())
        assert t_last < 200
        assert used < 400 * per_tick
        short = _run(fleet, s, t_last)
        for k in METRICS:
            assert np.array_equal(long[k], short[k]), k
        assert np.array_equal(long["pose_log"][:, : t_last + 1], short["pose_log"])
        assert np.array_equal(long["cmd_log"][:, :t_last], short["cmd_log"])
        assert np.all(long["pose_log"][:, t_last:] == long["pose_log"][:, t_last:t_last + 1])
        assert np.all(long["cmd_log"][:, t_last:] == 0.0) and not long["optimized_log"][:, t_last:].any()
    finally:
        fleet.close()


def test_episodes_leave_the_fleet_tick_memory_alone():
    """optimize_batch tick 1, run_episodes, tick 2 == ticks 1 and 2 of a fresh fleet (episodes have their own state)."""
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    B = 6
    s = sc.episodes(B, 5, ticks=20, seed=9)
    p = s["params"]
    poses, cmds = sc.pure_pursuit_seed(s["global_path"], s["pose"], p)
    people = np.ascontiguousarray(s["people"][:, :A])
    n_people = np.full(B, A, np.int32)
    maps = (s["costmaps"], s["costmap_origin"], s["costmap_resolution"], s["od"])

    def tick(fl):
        return fl.optimize_batch(poses, cmds, people, n_people, s["speed"], *maps, costmap_index=s["costmap_index"])

    a, b = FleetOptimizer(p, n_robots=B, n_agents=A), FleetOptimizer(p, n_robots=B, n_agents=A)
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


def test_people_free_straight_corridor_reaches_the_goal():
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    B = 4
    s = sc.episodes(B, 0, ticks=200, seed=2)
    N = s["global_path"].shape[1]
    s["global_path"][:] = _path(B, N, 1.0, 2.0, 3.0)
    s["pose"][:, 1] = 2.0
    s["costmaps"][:] = sc.wall_costmap(240, 80, 0.05, walls_y=(0.3, 3.7))  # no box
    fleet = FleetOptimizer(s["params"], n_robots=B, n_agents=A)
    try:
        got = _run(fleet, s, 200, want_logs=False)
    finally:
        fleet.close()
    assert got["reached"].all() and np.all(got["ticks"] < 200)
    assert np.all(got["collision_ticks"] == 0) and np.all(got["min_person_dist"] == np.inf)
    assert np.all(got["personal_ticks"] == 0) and np.all(got["path_length"] > 2.5)


def test_episode_argument_errors_launch_nothing():
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    import ctypes as C
    B = 4
    s = sc.episodes(B, 3, ticks=10, seed=4)
    p = s["params"]
    ARG, UNSUP = -1, -3

    def expect(fleet, code, **kw):
        c0 = fleet.opt.launch_count()
        with pytest.raises(_lib.SmpcError) as e:
            _run(fleet, s, kw.pop("T", 10), want_logs=False, **kw)
        assert e.value.code == code, kw
        assert fleet.opt.launch_count() == c0

    for bad, code in ((dict(omni_solve=1), UNSUP), (dict(omnidirectional=1), UNSUP),
                      (dict(max_time=0.1, time_step=0.05), ARG)):
        pb = sc.make_params("soc_work_obst", **bad)
        fleet = FleetOptimizer(pb, n_robots=B, n_agents=A)
        try:
            expect(fleet, code)
        finally:
            fleet.close()
    fleet = FleetOptimizer(p, n_robots=B, n_agents=A)
    try:
        expect(fleet, ARG, global_path=s["global_path"][:, :1])
        expect(fleet, ARG, T=0)
        expect(fleet, ARG, control_period=0.0)
        expect(fleet, ARG, goal_tolerance=0.15)  # below the trajectorizer's 0.2 m stop: no seed short of the goal
        bad_n = s["n_people"].copy()
        bad_n[2] = 4
        expect(fleet, ARG, n_people=bad_n)
        for field in ("costmaps", "od_indexes", "reached", "cmd_variation"):
            io, out, logs, keep = fleet.episode_io(**{k: v for k, v in s.items() if k != "params"})
            setattr(io, field, None)
            c0 = fleet.opt.launch_count()
            assert _lib.lib().smpc_run_episodes(fleet.opt._h, C.byref(io)) == ARG, field
            assert fleet.opt.launch_count() == c0
    finally:
        fleet.close()
    for n_agents in (0, 64):
        fleet = FleetOptimizer(p, n_robots=B, n_agents=n_agents)
        try:
            expect(fleet, ARG)
        finally:
            fleet.close()
