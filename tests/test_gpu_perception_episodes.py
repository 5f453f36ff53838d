"""GPU tests of the perceived episode entry smpc_run_perceived_episodes (FleetOptimizer.run_episodes /
run_crowd_episodes / run_shared_episodes with perception=...): neutral parameters compute what the entries without
perception compute, bit for bit; with the default sensor every tick is replayed through the numpy stage of
tests/perception_ref.py and the public path (filter_people_fov, optimize_batch); hand-built scenes check each way a row
can go unreported."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from tests import episode_ref as ref
from tests import perception_ref as pref
from tests import shared_ref as sref

pytestmark = pytest.mark.gpu

A = 3
ARG = -1
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
CROWD_OUT = METRICS + ("people_disturbance",)
SHARED_OUT = CROWD_OUT + ("robot_min_dist", "robot_intimate_ticks")
LOGS = ("pose_log", "cmd_log", "optimized_log")
PERCEIVED = ("unseen_personal_ticks", "seen_log", "n_seen_log")
NEUTRAL = dict(abi.PERCEPTION_NEUTRAL)


def _fleet(p, B):
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    return FleetOptimizer(p, n_robots=B, n_agents=A)


def _args(s, **kw):
    a = {k: v for k, v in s.items() if k not in ("params", "ticks")}
    a.update(kw)
    return a


def _run(fleet, s, T, want_logs=True, **kw):
    if "robots_per_scene" in s:
        fn = fleet.run_shared_episodes
    elif "goals" in s:
        fn = fleet.run_crowd_episodes
    else:
        fn = fleet.run_episodes
    return fn(ticks=T, want_logs=want_logs, **_args(s, **kw))


def _outputs(s):
    if "robots_per_scene" in s:
        return SHARED_OUT + LOGS + ("people_log",)
    if "goals" in s:
        return CROWD_OUT + LOGS + ("people_log",)
    return METRICS + LOGS


def _device_trig():
    """cos / sin from the device's math library, which the scene view uses for the robots' headings."""
    import torch

    def f(fn):
        return lambda x: fn(torch.as_tensor(np.asarray(x, dtype=np.float64), device="cuda")).cpu().numpy()
    return f(torch.cos), f(torch.sin)


def _scenes(kind, T):
    if kind == "cv":
        return sc.episodes(8, 6, ticks=T, n_maps=2, seed=11)
    if kind == "shared2":
        return sc.shared_episodes(4, 2, 6, seed=13, ticks=T, substeps=2)
    if kind == "shared3":
        return sc.shared_episodes(3, 3, 6, seed=14, ticks=T)
    return sc.crowd_episodes(8, 6, ticks=T, seed=11, substeps=4 if kind == "sfm4" else 1)


def _kw(kind):
    return dict(orca=abi.orca_params()) if kind == "orca" else {}


@pytest.mark.parametrize("kind", ["cv", "sfm1", "sfm4", "orca", "shared2", "shared3", "weights"])
def test_neutral_perception_is_the_entry_without_perception(kind):
    T = 50
    s = _scenes("sfm1" if kind == "weights" else kind, T)
    kw = _kw(kind)
    B = s["pose"].shape[0]
    if kind == "weights":
        rows = [sc.make_params("obst_only"), sc.make_params("soc_work_obst")]
        kw["weights"] = (np.stack([abi.weight_row(r) for r in rows]), (np.arange(B) % 2).astype(np.int32))
    fleet = _fleet(s["params"], B)
    try:
        c0 = fleet.opt.launch_count()
        a = _run(fleet, s, T, **kw)
        c1 = fleet.opt.launch_count()
        b = _run(fleet, s, T, perception=NEUTRAL, **kw)
        c2 = fleet.opt.launch_count()
    finally:
        fleet.close()
    for k in _outputs(s):
        assert np.array_equal(a[k], b[k]), k
    assert not b["unseen_personal_ticks"].any()
    loop_ticks = int(a["ticks"].max())  # ticks the loop ran (the early-stop poll may run it further)
    assert loop_ticks <= c2 - c1 - (c1 - c0) <= T
    # the logged list is the FOV filter's input without perception, for every tick a robot ran
    R = s.get("robots_per_scene", 1)
    n_list = np.repeat(s["n_people"], R) + (R - 1)
    ran = np.arange(T)[None, :] < a["ticks"][:, None]
    assert np.array_equal(b["n_seen_log"], np.where(ran, n_list[:, None], 0))
    if kind == "cv":
        dt_c = s["control_period"]
        for k in range(T):
            want = ref.people_at(s["people"], k * dt_c)
            assert np.array_equal(b["seen_log"][ran[:, k], k], want[ran[:, k]]), k
    elif R == 1:
        assert np.array_equal(b["seen_log"], np.where(ran[..., None, None], a["people_log"][:, :T], 0.0))
    assert not b["seen_log"][~ran].any()


@pytest.mark.parametrize("kind,per_tick", [("cv", 13), ("sfm1", 14), ("shared2", 16)])
def test_launches_per_tick(kind, per_tick):
    s = _scenes(kind, 3)
    fleet = _fleet(s["params"], s["pose"].shape[0])
    try:
        counts = {}
        for T in (1, 3):
            c0 = fleet.opt.launch_count()
            _run(fleet, s, T, want_logs=False, perception={})
            counts[T] = fleet.opt.launch_count() - c0
    finally:
        fleet.close()
    assert counts[1] == per_tick and counts[3] == 3 * per_tick, counts


@pytest.mark.parametrize("kind", ["cv", "sfm1", "orca", "shared2"])
def test_default_perception_replays_through_the_numpy_stage_and_the_public_path(kind):
    T = 60
    s = _scenes(kind, T)
    R = s.get("robots_per_scene", 1)
    p, dt_c = s["params"], s["control_period"]
    B = s["pose"].shape[0]
    K = s["people"].shape[1]
    prm = dict(pref.DEFAULTS)
    fleet, replay = _fleet(p, B), _fleet(p, B)
    cos, sin = _device_trig()
    try:
        got = _run(fleet, s, T, perception={}, **_kw(kind))
        pl, cl, ol, ticks = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"]
        sl, nsl = got["seen_log"], got["n_seen_log"]
        assert sl.shape == (B, T, R - 1 + K, 5) and nsl.shape == (B, T)
        H, W = s["costmaps"].shape[1:]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
        unseen = np.zeros(B, np.int32)
        hidden = 0
        for k in range(T):
            pk = pl[:, k]
            act = ~done
            if kind == "cv":
                lists, n_list = ref.people_at(s["people"], k * dt_c), s["n_people"]
            elif R == 1:
                lists, n_list = got["people_log"][:, k], s["n_people"]
            else:
                lists, n_list = sref.scene_views(pk, speed, act, got["people_log"][:, k], s["n_people"], R, cos=cos,
                                                 sin=sin)
            want, want_n, missed = pref.perceive_all(lists, n_list, pk, act, k, prm, s["costmaps"],
                                                     s["costmap_origin"], s["costmap_resolution"],
                                                     s["costmap_index"], R=R, K=K)
            assert np.array_equal(nsl[:, k], want_n), k
            assert np.abs(sl[:, k] - want).max() <= 1e-12, k
            unseen += missed & act
            hidden += int((n_list - want_n)[act].sum())
            poses, cmds3, n_steps = replay.trajectorize_batch(s["global_path"], pk)
            cmds = np.ascontiguousarray(cmds3[:, :, [0, 2]])
            fp, fn = replay.filter_people_fov(sl[:, k], nsl[:, k], pk, s["costmap_origin"], W, H,
                                              s["costmap_resolution"], costmap_index=s["costmap_index"])
            n_poses = np.where(done, 0, n_steps + 1).astype(np.int32)
            r = replay.optimize_batch(poses, cmds, fp, fn, speed, s["costmaps"], s["costmap_origin"],
                                      s["costmap_resolution"], s["od"], costmap_index=s["costmap_index"],
                                      n_poses=n_poses, want_people_proj=False)
            cmd = r["cmds"][:, 0]
            assert np.array_equal(cl[act, k], cmd[act]), k
            assert np.array_equal(ol[act, k], r["optimized"][act]), k
            speed[act] = cmd[act]
            done |= ticks == k + 1
        assert np.array_equal(got["unseen_personal_ticks"], unseen)
        assert hidden > 0  # the sensor dropped rows
    finally:
        fleet.close()
        replay.close()


def _targeted(T=1):
    """Four robots at (1, 2) facing +x with standing people: a person behind a lethal bar (0, on a costmap of its own),
    two people in line (1), a person 9.5 m away (2), a person in plain view (3)."""
    s = sc.episodes(4, 2, ticks=T, seed=3)
    s["pose"][:] = [1.0, 2.0, 0.0]
    s["people"][:] = 0.0
    s["people"][0, 0, :2] = [3.0, 2.0]
    s["people"][1, 0, :2] = [2.0, 2.0]
    s["people"][1, 1, :2] = [3.5, 2.02]
    s["people"][2, 0, :2] = [10.5, 2.0]
    s["people"][3, 0, :2] = [3.0, 2.3]
    s["n_people"][:] = [1, 2, 1, 1]
    bar = s["costmaps"][0].copy()
    res = s["costmap_resolution"]
    bar[int(1.5 / res):int(2.5 / res), int(2.0 / res)] = 254
    M = s["costmaps"].shape[0]
    s["costmaps"] = np.concatenate([s["costmaps"], bar[None]])
    s["costmap_origin"] = np.zeros((M + 1, 2))
    s["costmap_index"] = s["costmap_index"].copy()
    s["costmap_index"][0] = M
    return s


def test_targeted_scenes():
    s = _targeted()
    exact = dict(detect_prob=1.0, pos_noise=0.0, vel_noise=0.0)
    fleet = _fleet(s["params"], 4)
    try:
        got = _run(fleet, s, 1, perception=exact)
        walls_off = _run(fleet, s, 1, perception=dict(exact, occluding_cost=0))
        blind = _run(fleet, s, 1, perception=dict(exact, detect_prob=0.0))
    finally:
        fleet.close()
    assert got["n_seen_log"][:, 0].tolist() == [0, 1, 0, 1]
    assert np.array_equal(got["seen_log"][1, 0, 0], s["people"][1, 0])  # the nearer of the two in line
    assert np.array_equal(got["seen_log"][3, 0, 0], s["people"][3, 0])
    assert walls_off["n_seen_log"][:, 0].tolist() == [1, 1, 0, 1]
    assert not blind["n_seen_log"].any() and not blind["seen_log"].any()
    assert blind["unseen_personal_ticks"].tolist() == [0, 1, 0, 0]  # the person 1 m ahead of robot 1 went unseen
    assert got["unseen_personal_ticks"].tolist() == [0, 0, 0, 0]  # nobody hidden was within 1.2 m


def test_seeds_streams_and_early_stop():
    B0, T = 6, 40
    s = sc.crowd_episodes(B0, 5, seed=8, ticks=T, substeps=2)
    p = s["params"]
    fleet = _fleet(p, B0)
    try:
        x, y = _run(fleet, s, T, perception={}), _run(fleet, s, T, perception={})
        z = _run(fleet, s, T, perception=dict(seed=1))
    finally:
        fleet.close()
    for k in CROWD_OUT + LOGS + PERCEIVED:
        assert np.array_equal(x[k], y[k]), k
    assert not np.array_equal(x["seen_log"], z["seen_log"])
    # copies of the scenes under an identity table with one stream per scene see the same noise and dropouts
    t = sc.tile_scenes(s, 2)
    row = abi.weight_row(p)
    fw = _fleet(p, 2 * B0)
    try:
        got = _run(fw, t, T, weights=(np.stack([row, row]), np.repeat(np.arange(2), B0).astype(np.int32)),
                   perception=dict(stream_index=np.arange(2 * B0) % B0))
        own = _run(fw, t, T, perception={})
    finally:
        fw.close()
    for k in CROWD_OUT + LOGS + PERCEIVED:
        assert np.array_equal(got[k][:B0], got[k][B0:]), k
        assert np.array_equal(got[k][:B0], x[k]), k  # streams 0 .. B0-1 are what the untiled call drew
    assert not np.array_equal(own["seen_log"][:B0], own["seen_log"][B0:])  # streams b: other draws
    # an early stop gives the results of the run that ends at the last arrival tick
    e = sc.episodes(8, 2, ticks=400, seed=5, path_length=1.2)
    e["pose"][:, 1] = 2.0
    fe = _fleet(e["params"], 8)
    try:
        long = _run(fe, e, 400, perception={})
        last = int(long["ticks"].max())
        assert last < 400 - 16
        short = _run(fe, e, last, perception={})
    finally:
        fe.close()
    for k in METRICS + ("unseen_personal_ticks",):
        assert np.array_equal(long[k], short[k]), k
    for k in ("cmd_log", "optimized_log", "seen_log", "n_seen_log"):
        assert np.array_equal(long[k][:, :last], short[k]), k
        assert not long[k][:, last:].any(), k


def test_perceived_argument_errors_launch_nothing_and_leave_the_fleet_state():
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
    wide = sc.episodes(B, 65, ticks=10, seed=4)  # 65 people: a list longer than the stage's 64 rows
    wio, wout, wlogs, wkeep = a.episode_io(**{k: v for k, v in _args(wide).items()}, ticks=10)
    goals = np.ascontiguousarray(sh["goals"])
    vdes = np.ascontiguousarray(sh["desired_speed"])
    dist, rmin, rint = np.zeros(B), np.zeros(B), np.zeros(B, np.int32)
    crowd = abi.SmpcCrowdIo(goals.ctypes.data, vdes.ctypes.data, 1, dist.ctypes.data, None)
    scene = abi.SmpcSceneIo(R, rmin.ctypes.data, rint.ctypes.data)
    table = abi.weight_row(p)[None].copy()
    idx = np.zeros(B, np.int32)
    ws = abi.SmpcWeightSets(1, table.ctypes.data, idx.ctypes.data)
    unseen, n_log = np.zeros(B, np.int32), np.zeros((B, 10), np.int32)
    seen_log = np.zeros((B, 10, R - 1 + 5, 5))
    neg = np.arange(B, dtype=np.int32) - 1
    ident = np.arange(B, dtype=np.int32)
    L = _lib.lib()

    def call(over=None, fields=None, null_pc=False, use_crowd=True, use_scene=True, orca=None, w=None, episode=io):
        pc = abi.perception_params(**(over or {}))
        pc.unseen_personal_ticks = unseen.ctypes.data
        for f, v in (fields or {}).items():
            setattr(pc, f, v)
        c0 = a.opt.launch_count()
        rc = L.smpc_run_perceived_episodes(a.opt._h, C.byref(episode), C.byref(crowd) if use_crowd else None,
                                           C.byref(scene) if use_scene else None, None if w is None else C.byref(w),
                                           None if orca is None else C.byref(orca), None if null_pc else C.byref(pc))
        if rc != 0:
            assert a.opt.launch_count() == c0
        return rc

    try:
        first = tick(a)
        assert call(null_pc=True) == ARG
        for f, bad in (("max_range", (0.0, -1.0, np.nan)), ("occluder_radius", (-0.1, np.nan, np.inf)),
                       ("occluding_cost", (-1, 256)), ("detect_prob", (-0.1, 1.5, np.nan)),
                       ("pos_noise", (-0.1, np.nan, np.inf)), ("vel_noise", (-0.1, np.nan, np.inf))):
            for v in bad:
                assert call(over={f: v}) == ARG, (f, v)
        assert call(fields=dict(unseen_personal_ticks=None)) == ARG
        assert call(fields=dict(seen_log=seen_log.ctypes.data)) == ARG
        assert call(fields=dict(n_seen_log=n_log.ctypes.data)) == ARG
        assert call(fields=dict(stream_index=neg.ctypes.data)) == ARG
        assert call(use_crowd=False) == ARG  # a scene without a crowd
        assert call(use_crowd=False, use_scene=False, orca=abi.orca_params()) == ARG  # ORCA without a crowd
        assert call(orca=abi.orca_params(max_neighbors=0)) == ARG
        assert call(w=abi.SmpcWeightSets(0, table.ctypes.data, idx.ctypes.data)) == ARG
        assert call(use_crowd=False, use_scene=False, episode=wio) == ARG  # L = 65
        # the same blocks with valid parameters run, and leave the warm-start memory of optimize_batch alone
        assert call() == 0
        assert call(w=ws, orca=abi.orca_params(), over=NEUTRAL,
                    fields=dict(seen_log=seen_log.ctypes.data, n_seen_log=n_log.ctypes.data,
                                stream_index=ident.ctypes.data)) == 0
        second = tick(a)
        want = [tick(b), tick(b)]
        for k in ("cmds", "path", "optimized", "n_out", "termination", "cost_final"):
            assert np.array_equal(first[k], want[0][k]) and np.array_equal(second[k], want[1][k]), k
    finally:
        a.close()
        b.close()
