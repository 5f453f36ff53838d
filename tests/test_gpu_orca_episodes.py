"""GPU tests of the ORCA crowd entry smpc_run_orca_episodes (FleetOptimizer.run_crowd_episodes / run_shared_episodes
with orca=...): every tick is replayed through the public path (trajectorize_batch, filter_people_fov, optimize_batch),
the crowd through the numpy restatement of tests/orca_ref.py and the world and metrics through tests/episode_ref.py,
tests/crowd_ref.py and tests/shared_ref.py."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from tests import crowd_ref as cref
from tests import episode_ref as ref
from tests import orca_ref as oref
from tests import shared_ref as sref

pytestmark = pytest.mark.gpu

A = 3
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
CROWD_OUT = METRICS + ("people_disturbance",)
SHARED_OUT = CROWD_OUT + ("robot_min_dist", "robot_intimate_ticks")
LOGS = ("pose_log", "cmd_log", "optimized_log", "people_log")
ARG = -1
ORCA = dict(oref.DEFAULTS)


def _fleet(p, B):
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    return FleetOptimizer(p, n_robots=B, n_agents=A)


def _args(s, **kw):
    a = {k: v for k, v in s.items() if k not in ("params", "ticks")}
    a.update(kw)
    return a


def _run(fleet, s, T, want_logs=True, orca=None, **kw):
    fn = fleet.run_shared_episodes if "robots_per_scene" in s else fleet.run_crowd_episodes
    return fn(ticks=T, want_logs=want_logs, orca=abi.orca_params(**(orca or {})), **_args(s, **kw))


def _device_trig():
    """cos / sin from the device's math library, which the kernels use for the robots' headings."""
    import torch

    def f(fn):
        return lambda x: fn(torch.as_tensor(np.asarray(x, dtype=np.float64), device="cuda")).cpu().numpy()
    return f(torch.cos), f(torch.sin)


def _scenes(R, T, substeps):
    """R None: 8 one-robot scenes of run_crowd_episodes (K = 6) with a people-free scene (0), a robot with a 0.5 m
    path (1) and a person walking head-on at the robot (2). R >= 2: 4 shared scenes of R robots, K = 6, scene 0
    people-free, robot 0 of scene 1 with a 0.5 m path."""
    if R is None:
        s = sc.crowd_episodes(8, 6, ticks=T, seed=11, substeps=substeps)
        N = s["global_path"].shape[1]
        s["n_people"][0] = 0
        s["global_path"][1, :, 0] = 1.0 + np.linspace(0.0, 0.5, N)
        s["global_path"][1, :, 1] = 2.0
        s["pose"][1] = [1.0, 2.0, 0.0]
        s["pose"][2] = [1.0, 2.0, 0.0]
        s["people"][2, 0] = [2.4, 2.0, -0.6, 0.0, 0.0]
        s["goals"][2, 0] = [1.6, 2.0]
        s["desired_speed"][2, 0] = 0.6
        return s
    s = sc.shared_episodes(4, R, 6, seed=11 + R, ticks=T, substeps=substeps)
    s["n_people"][0] = 0
    N = s["global_path"].shape[1]
    p0, p1 = s["global_path"][R, 0], s["global_path"][R, -1]
    s["global_path"][R] = p0 + (p1 - p0) / np.linalg.norm(p1 - p0) * np.linspace(0.0, 0.5, N)[:, None]
    return s


def _replay(R, substeps, T=60):
    s = _scenes(R, T, substeps)
    shared = R is not None
    R = R or 1
    p, dt_c = s["params"], s["control_period"]
    B = s["pose"].shape[0]
    S = B // R
    fleet, replay = _fleet(p, B), _fleet(p, B)
    cos, sin = _device_trig()
    n_od = np.asarray(s["od"]["origins"]).reshape(-1, 2).shape[0]
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
        checked = 0
        for k in range(T):
            pk = pl[:, k]
            act = ~done
            poses, cmds3, n_steps = replay.trajectorize_batch(s["global_path"], pk)
            cmds = np.ascontiguousarray(cmds3[:, :, [0, 2]])
            if shared:
                views, n_view = sref.scene_views(pk, speed, act, ppl[:, k], s["n_people"], R, cos=cos, sin=sin)
            else:
                views, n_view = ppl[:, k], s["n_people"]
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
                q, flags[c], d, near = oref.crowd_step(ppl[c, k, :n], flags[c], s["goals"][c, :n],
                                                       s["desired_speed"][c, :n], pk[rb], cl[rb, k],
                                                       cref.od_of(s["od"], (c * R) % n_od), dt_c, substeps, ORCA,
                                                       running=act[rb], cos=cos, sin=sin)
                skip[c] |= near
                dist[rb] += d
                # every person is compared; only a near tie may part from the reference
                bad = np.abs(ppl[c, k + 1, :n] - q).max(axis=1, initial=0.0) > 1e-12
                assert not (bad & ~skip[c]).any(), (k, c)
                assert np.array_equal(ppl[c, k + 1, n:], ppl[c, k, n:])
                checked += int((~bad).sum())
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
        for key in ("collision_ticks", "not_optimized_ticks"):
            assert np.array_equal(got[key], m[key]), key
        ok = ~m["near_threshold"]
        for key in ("intimate_ticks", "personal_ticks"):
            assert np.array_equal(got[key][ok], m[key][ok]), key
        for key in ("path_length", "min_person_dist", "cmd_variation"):
            assert np.allclose(got[key], m[key], rtol=0, atol=1e-9), key
        assert np.allclose(got["people_disturbance"], dist, rtol=1e-9, atol=1e-300)
        if shared:
            rmin, rint = sref.robot_metrics(pl, ticks, R)
            assert np.array_equal(got["robot_min_dist"], rmin)
            assert np.array_equal(got["robot_intimate_ticks"], rint)
        # the scenes do what they were built for
        assert np.all(got["min_person_dist"][:R] == np.inf) and np.all(got["people_disturbance"][:R] == 0.0)
        assert (ticks < T).any()  # an episode finished early: the replay covered finished robots
        assert (got["people_disturbance"] > 0.0).any()
        return got
    finally:
        fleet.close()
        replay.close()


@pytest.mark.parametrize("substeps", [1, 4])
def test_orca_crowd_episodes_replay_through_the_public_path_and_the_numpy_crowd(substeps):
    _replay(None, substeps)


@pytest.mark.parametrize("R", [2, 3])
def test_orca_shared_episodes_replay_through_the_public_path_and_the_numpy_crowd(R):
    _replay(R, 2)


def test_zero_responsibility_hides_the_robots():
    """robot_responsibility = 0: the people log is the people stepped alone (numpy, from the input state), whatever the
    robots do, and the disturbance is 0."""
    T = 40
    s = sc.crowd_episodes(6, 8, ticks=T, seed=5, substeps=2)
    moved = dict(s, pose=s["pose"] + [0.3, 0.2, 0.3])  # the robots start elsewhere: other commands, other paths
    fleet = _fleet(s["params"], 6)
    zero = dict(robot_responsibility=0.0)
    cos, sin = _device_trig()
    try:
        a = _run(fleet, s, T, orca=zero)
        b = _run(fleet, moved, T, orca=zero)
    finally:
        fleet.close()
    assert not np.array_equal(a["pose_log"], b["pose_log"])
    assert np.all(a["ticks"] == T) and np.all(b["ticks"] == T)
    assert np.array_equal(a["people_log"], b["people_log"])
    assert np.all(a["people_disturbance"] == 0.0) and np.all(b["people_disturbance"] == 0.0)
    n_od = np.asarray(s["od"]["origins"]).reshape(-1, 2).shape[0]
    for c in range(6):
        q, f = s["people"][c], np.ones(8, bool)
        for k in range(T):
            q, f, d, near = oref.crowd_step(q, f, s["goals"][c], s["desired_speed"][c], [], [],
                                            cref.od_of(s["od"], c % n_od), s["control_period"], 2, zero, cos=cos,
                                            sin=sin)
            assert np.abs(a["people_log"][c, k + 1] - q).max() <= 1e-12, (c, k)


def test_no_people_is_run_crowd_episodes():
    for s in (sc.crowd_episodes(8, 0, ticks=50, seed=3), sc.shared_episodes(4, 2, 0, ticks=50, seed=3)):
        B = s["pose"].shape[0]
        fleet = _fleet(s["params"], B)
        try:
            a = _run(fleet, s, 50)
            fn = fleet.run_shared_episodes if "robots_per_scene" in s else fleet.run_crowd_episodes
            b = fn(ticks=50, want_logs=True, **_args(s))
        finally:
            fleet.close()
        for k in (SHARED_OUT if "robots_per_scene" in s else CROWD_OUT) + LOGS:
            assert np.array_equal(a[k], b[k]), k


def test_weight_tables():
    """An identity table equals the unweighted ORCA call; with two rows each copy of the scenes equals its row run
    alone."""
    B0, T = 6, 50
    s = sc.crowd_episodes(B0, 5, seed=8, ticks=T, substeps=2)
    p = s["params"]
    ident = (abi.weight_row(p)[None], np.zeros(B0, np.int32))
    fleet = _fleet(p, B0)
    try:
        x, y = _run(fleet, s, T), _run(fleet, s, T, weights=ident)
        for k in CROWD_OUT + LOGS:
            assert np.array_equal(x[k], y[k]), k
        sh = sc.shared_episodes(3, 2, 5, seed=6, ticks=T)
        x, y = _run(fleet, sh, T), _run(fleet, sh, T, weights=(ident[0], np.zeros(6, np.int32)))
        for k in SHARED_OUT + LOGS:
            assert np.array_equal(x[k], y[k]), k
    finally:
        fleet.close()
    rows = [sc.make_params("obst_only"), sc.make_params("soc_work_obst")]
    table = np.stack([abi.weight_row(r) for r in rows])
    fw = _fleet(p, 2 * B0)
    try:
        got = _run(fw, sc.tile_scenes(s, 2), T, weights=(table, np.repeat(np.arange(2), B0).astype(np.int32)))
    finally:
        fw.close()
    for q in range(2):
        fq = _fleet(rows[q], B0)
        try:
            want = _run(fq, s, T)
        finally:
            fq.close()
        for k in CROWD_OUT + LOGS:
            assert np.array_equal(got[k][q * B0:(q + 1) * B0], want[k]), (q, k)
    assert not np.array_equal(got["cmd_log"][:B0], got["cmd_log"][B0:])


@pytest.mark.parametrize("R,per_tick", [(None, 13), (2, 15)])
def test_launches_per_tick(R, per_tick):
    s = sc.crowd_episodes(8, 6, ticks=3, seed=4) if R is None else sc.shared_episodes(4, R, 6, ticks=3, seed=4)
    fleet = _fleet(s["params"], s["pose"].shape[0])
    try:
        counts = {}
        for T in (1, 3):
            c0 = fleet.opt.launch_count()
            _run(fleet, s, T, want_logs=False)
            counts[T] = fleet.opt.launch_count() - c0
    finally:
        fleet.close()
    assert counts[1] == per_tick and counts[3] == 3 * per_tick, counts


def test_orca_and_lightsfm_crowds_differ():
    s = sc.crowd_episodes(8, 10, ticks=40, seed=2)
    fleet = _fleet(s["params"], 8)
    try:
        a = _run(fleet, s, 40)
        b = fleet.run_crowd_episodes(ticks=40, want_logs=True, **_args(s))
    finally:
        fleet.close()
    assert np.array_equal(a["people_log"][:, 0], b["people_log"][:, 0])
    for c in range(8):
        assert not np.array_equal(a["people_log"][c, 1:], b["people_log"][c, 1:]), c


def test_orca_argument_errors_launch_nothing_and_leave_the_fleet_state():
    S, R = 3, 2
    B = S * R
    sh = sc.shared_episodes(S, R, 5, ticks=10, seed=4)
    p = sh["params"]
    poses, cmds = sc.pure_pursuit_seed(sh["global_path"], sh["pose"], p)
    people = np.ascontiguousarray(sh["people"][np.arange(B) // 2, :A])
    maps = (sh["costmaps"], sh["costmap_origin"], sh["costmap_resolution"], sh["od"])

    def tick(fl):
        return fl.optimize_batch(poses, cmds, people, np.full(B, A, np.int32), sh["speed"], *maps,
                                 costmap_index=sh["costmap_index"])

    a, b = _fleet(p, B), _fleet(p, B)
    io, out, logs, keep = a.episode_io(**{k: v for k, v in _args(sh).items()
                                          if k not in ("goals", "desired_speed", "substeps", "robots_per_scene")},
                                       ticks=10, robots_per_scene=R)
    goals = np.ascontiguousarray(sh["goals"])
    vdes = np.ascontiguousarray(sh["desired_speed"])
    dist, rmin, rint = np.zeros(B), np.zeros(B), np.zeros(B, np.int32)
    crowd = abi.SmpcCrowdIo(goals.ctypes.data, vdes.ctypes.data, 1, dist.ctypes.data, None)
    scene = abi.SmpcSceneIo(R, rmin.ctypes.data, rint.ctypes.data)
    table = abi.weight_row(p)[None].copy()
    idx = np.zeros(B, np.int32)
    ws = abi.SmpcWeightSets(1, table.ctypes.data, idx.ctypes.data)
    L = _lib.lib()

    def call(orca=None, null_orca=False, null_crowd=False, w=None, crowd_fields=None):
        o = abi.orca_params(**(orca or {}))
        cr = abi.SmpcCrowdIo(crowd.goals, crowd.desired_speed, crowd.substeps, crowd.people_disturbance, None)
        for f, v in (crowd_fields or {}).items():
            setattr(cr, f, v)
        c0 = a.opt.launch_count()
        rc = L.smpc_run_orca_episodes(a.opt._h, C.byref(io), None if null_crowd else C.byref(cr), C.byref(scene),
                                      None if w is None else C.byref(w), None if null_orca else C.byref(o))
        if rc != 0:
            assert a.opt.launch_count() == c0
        return rc

    try:
        first = tick(a)
        assert call(null_orca=True) == ARG
        assert call(null_crowd=True) == ARG
        for f in ("neighbor_dist", "time_horizon", "time_horizon_obst", "person_radius", "robot_radius"):
            for v in (0.0, -1.0, np.nan, np.inf):
                assert call(orca={f: v}) == ARG, (f, v)
        for v in (0, 17, -1):
            assert call(orca=dict(max_neighbors=v)) == ARG, v
        for v in (-0.1, 1.5, np.nan):
            assert call(orca=dict(robot_responsibility=v)) == ARG, v
        assert call(crowd_fields=dict(substeps=0)) == ARG
        assert call(crowd_fields=dict(people_disturbance=None)) == ARG
        bad = abi.SmpcWeightSets(0, table.ctypes.data, idx.ctypes.data)
        assert call(w=bad) == ARG
        second = tick(a)
        want = [tick(b), tick(b)]
        for k in ("cmds", "path", "optimized", "n_out", "termination", "cost_final"):
            assert np.array_equal(first[k], want[0][k]) and np.array_equal(second[k], want[1][k]), k
        # the same blocks with valid parameters run
        assert call() == 0
        assert call(w=ws, orca=dict(max_neighbors=16, robot_responsibility=1.0)) == 0
        assert call(orca=dict(max_neighbors=1, robot_responsibility=0.0)) == 0
    finally:
        a.close()
        b.close()
