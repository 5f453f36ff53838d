"""GPU tests of the tracked episode entry smpc_run_tracked_episodes (FleetOptimizer.run_episodes / run_crowd_episodes /
run_shared_episodes with perception=... and tracker=...): the pass-through tracker on standing people computes what
smpc_run_perceived_episodes computes, bit for bit; with the default tracker every tick is replayed through the numpy
tracker of tests/tracker_ref.py and the public path (filter_people_fov, optimize_batch); a hand-built scene checks
coasting, confirmation and latency."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from tests import episode_ref as ref
from tests import perception_ref as pref
from tests import shared_ref as sref
from tests import tracker_ref as tref

pytestmark = pytest.mark.gpu

A = 3
ARG = -1
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
CROWD_OUT = METRICS + ("people_disturbance",)
LOGS = ("pose_log", "cmd_log", "optimized_log")
PERCEIVED = ("unseen_personal_ticks", "seen_log", "n_seen_log")
TRACKED = PERCEIVED + ("untracked_personal_ticks", "track_rows", "mean_track_pos_error", "mean_track_vel_error",
                       "track_id_log")
SENSOR = dict(vel_noise=0.0)  # the default sensor, reporting positions only


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


def _same(a, b, keys):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k


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


def test_pass_through_on_standing_people_is_the_perceived_entry():
    T = 60
    s = sc.episodes(8, 6, ticks=T, n_maps=2, seed=11)
    s["people"][..., 2:] = 0.0  # standing people
    exact = dict(pos_noise=0.0, vel_noise=0.0)  # occlusion, range and missed detections stay on
    fleet = _fleet(s["params"], 8)
    try:
        c0 = fleet.opt.launch_count()
        a = _run(fleet, s, T, perception=exact)
        c1 = fleet.opt.launch_count()
        b = _run(fleet, s, T, perception=exact, tracker=abi.TRACKER_PASS_THROUGH)
        c2 = fleet.opt.launch_count()
    finally:
        fleet.close()
    _same(a, b, METRICS + LOGS + PERCEIVED)
    assert c2 - c1 == c1 - c0
    assert np.array_equal(b["untracked_personal_ticks"], b["unseen_personal_ticks"])
    ran = np.arange(T)[None, :] < b["ticks"][:, None]
    assert (b["n_seen_log"] < s["n_people"][:, None])[ran].any()  # the sensor dropped rows
    rows = b["track_rows"]
    assert rows.sum() == b["n_seen_log"].sum()
    assert np.all(b["mean_track_pos_error"][rows > 0] == 0.0) and np.all(b["mean_track_vel_error"][rows > 0] == 0.0)
    ids = b["track_id_log"]
    n = b["n_seen_log"]
    L = ids.shape[2]
    past = np.arange(L)[None, None, :] >= n[..., None]
    assert np.all(ids[past] == -1) and np.all(ids[~past] >= 0)
    assert np.all(np.diff(ids, axis=2)[~past[..., 1:]] > 0)  # in list order


@pytest.mark.parametrize("kind", ["cv", "sfm1", "sfm4", "orca", "shared2", "shared3"])
def test_default_tracker_replays_through_the_numpy_tracker_and_the_public_path(kind):
    T = 60
    s = _scenes(kind, T)
    R = s.get("robots_per_scene", 1)
    p, dt_c = s["params"], s["control_period"]
    B = s["pose"].shape[0]
    K = s["people"].shape[1]
    pprm = dict(pref.DEFAULTS, **SENSOR)
    d = tref.DEFAULTS["latency_ticks"]
    trackers = [tref.RobotTracker(K + R if R > 1 else K, tref.DEFAULTS, dt_c) for _ in range(B)]
    fleet, replay = _fleet(p, B), _fleet(p, B)
    cos, sin = _device_trig()
    try:
        got = _run(fleet, s, T, perception=SENSOR, tracker={}, **_kw(kind))
        pl, cl, ol, ticks = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"]
        sl, nsl, il = got["seen_log"], got["n_seen_log"], got["track_id_log"]
        assert sl.shape == (B, T, R - 1 + K, 5) and nsl.shape == (B, T) and il.shape == (B, T, R - 1 + K)
        assert not nsl[:, :d].any()
        H, W = s["costmaps"].shape[1:]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
        sums = dict(unseen=np.zeros(B, np.int32), untracked=np.zeros(B, np.int32), rows=np.zeros(B, np.int32),
                    pos=np.zeros(B), vel=np.zeros(B))
        coasted = 0
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
            want = tref.tracked_all(trackers, lists, n_list, pk, act, k, pprm, s["costmaps"], s["costmap_origin"],
                                    s["costmap_resolution"], s["costmap_index"], R=R, K=K)
            assert np.array_equal(nsl[:, k], want["n_seen"]), k
            assert np.array_equal(il[:, k], want["ids"]), k
            assert np.abs(sl[:, k] - want["seen"]).max() <= 1e-12, k
            sums["unseen"] += want["missed"]
            sums["untracked"] += want["untracked"]
            sums["rows"] += want["rows"]
            sums["pos"] += want["pos_err"]
            sums["vel"] += want["vel_err"]
            if k >= d:
                coasted += sum(int(tr.misses > 0 and tr.hits >= tref.DEFAULTS["confirm_hits"]) for tr in
                               (t for b in np.flatnonzero(act) for t in trackers[b].tracks))
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
        assert np.array_equal(got["unseen_personal_ticks"], sums["unseen"])
        assert np.array_equal(got["untracked_personal_ticks"], sums["untracked"])
        assert np.array_equal(got["track_rows"], sums["rows"])
        some = sums["rows"] > 0
        assert some.any()
        for key, ref_sum in (("mean_track_pos_error", sums["pos"]), ("mean_track_vel_error", sums["vel"])):
            assert np.allclose(got[key][some] * sums["rows"][some], ref_sum[some], rtol=1e-9, atol=1e-12), key
            assert np.all(np.isnan(got[key][~some])), key
        assert coasted > 0  # some published track coasted through a miss
    finally:
        fleet.close()
        replay.close()


def _crossing(T):
    """Two robots driving +x along y = 2 from x = 1, each with one person crossing the corridor at x = 6, walking +y at
    0.5 m/s from y = 0.9, and a lethal bar at x = 5, y in [1.6, 2.4] (a costmap of its own) between them: the person
    is seen, hidden behind the bar, and seen again."""
    s = sc.episodes(2, 1, ticks=T, seed=3)
    s["pose"][:, 1:] = [2.0, 0.0]
    s["people"][:, 0] = [6.0, 0.9, 0.0, 0.5, 0.0]
    s["n_people"][:] = 1
    res = s["costmap_resolution"]
    bar = s["costmaps"][0].copy()
    inside = slice(int(round(0.4 / res)), int(round(3.6 / res)))
    bar[inside] = 0  # the corridor without the scenario's box
    bar[int(round(1.6 / res)):int(round(2.4 / res)), int(round(5.0 / res))] = 254
    M = s["costmaps"].shape[0]
    s["costmaps"] = np.concatenate([s["costmaps"], bar[None]])
    s["costmap_origin"] = np.zeros((M + 1, 2))
    s["costmap_index"] = np.full(2, M, np.int32)
    return s


def test_coasting_confirmation_latency_and_blindness_in_a_crossing():
    T, hits = 80, 3
    s = _crossing(T)
    exact = dict(detect_prob=1.0, pos_noise=0.0, vel_noise=0.0)
    trk = dict(confirm_hits=hits, latency_ticks=0)
    fleet = _fleet(s["params"], 2)
    try:
        coast = _run(fleet, s, T, perception=exact, tracker=dict(trk, max_coast_ticks=64))
        drop = _run(fleet, s, T, perception=exact, tracker=dict(trk, max_coast_ticks=0))
        late = _run(fleet, s, T, perception=exact, tracker=dict(trk, max_coast_ticks=64, latency_ticks=5))
        blind = _run(fleet, s, T, perception=dict(exact, detect_prob=0.0), tracker={})
    finally:
        fleet.close()
    for r in (coast, drop):
        # the sensor's view from the robot's logged poses: seen, hidden behind the bar, seen again
        vis = np.array([pref.perceive(ref.people_at(s["people"][:1], k * s["control_period"])[0], r["pose_log"][0, k],
                                      k, 0, dict(pref.NEUTRAL, occluding_cost=254), s["costmaps"][-1],
                                      s["costmap_origin"][-1], s["costmap_resolution"])[1][0] for k in range(T)])
        h0 = int(np.argmin(vis))  # the first hidden tick
        h1 = h0 + int(np.argmax(vis[h0:]))  # the first tick seen again
        assert vis[:h0].all() and h0 >= hits and h1 - h0 >= 10 and vis[h1:h1 + hits].all() and h1 + hits < T, (h0, h1)
        assert r["ticks"][0] == T
        n = r["n_seen_log"][0]
        assert not n[:hits - 1].any() and n[hits - 1:h0].all()  # published from the third detection on
        if r is coast:
            assert n[h0:h1].all()  # coasting through the hidden stretch
            assert r["untracked_personal_ticks"][0] == 0
        else:
            assert not n[h0:h1 + hits - 1].any() and n[h1 + hits - 1]  # gone at once, back after three detections
        assert np.all(r["track_id_log"][0, n > 0, 0] == 0)
    nl = late["n_seen_log"]
    assert not nl[:, :5].any() and nl[:, 5:].any()  # nothing before the first list arrives, 5 ticks late
    assert late["mean_track_pos_error"][0] > coast["mean_track_pos_error"][0]  # the truth moved on meanwhile
    assert not blind["n_seen_log"].any() and not blind["seen_log"].any() and np.all(blind["track_id_log"] == -1)
    assert np.all(blind["track_rows"] == 0) and np.all(np.isnan(blind["mean_track_pos_error"]))


def test_seeds_streams_and_early_stop():
    B0, T = 6, 40
    s = sc.crowd_episodes(B0, 5, seed=8, ticks=T, substeps=2)
    p = s["params"]
    fleet = _fleet(p, B0)
    try:
        x, y = _run(fleet, s, T, perception=SENSOR, tracker={}), _run(fleet, s, T, perception=SENSOR, tracker={})
        z = _run(fleet, s, T, perception=dict(SENSOR, seed=1), tracker={})
        per = _run(fleet, s, T, perception=SENSOR)
    finally:
        fleet.close()
    _same(x, y, CROWD_OUT + LOGS + TRACKED)
    assert not np.array_equal(x["seen_log"], z["seen_log"])
    assert np.array_equal(x["unseen_personal_ticks"], per["unseen_personal_ticks"])  # the same detections
    # copies of the scenes under an identity weight table with one stream per scene see the same detections and tracks
    t = sc.tile_scenes(s, 2)
    row = abi.weight_row(p)
    fw = _fleet(p, 2 * B0)
    try:
        got = _run(fw, t, T, weights=(np.stack([row, row]), np.repeat(np.arange(2), B0).astype(np.int32)),
                   perception=dict(SENSOR, stream_index=np.arange(2 * B0) % B0), tracker={})
    finally:
        fw.close()
    for k in CROWD_OUT + LOGS + TRACKED:
        assert np.array_equal(got[k][:B0], got[k][B0:], equal_nan=True), k
        assert np.array_equal(got[k][:B0], x[k], equal_nan=True), k
    # an early stop gives the results of the run that ends at the last arrival tick
    e = sc.episodes(8, 2, ticks=400, seed=5, path_length=1.2)
    e["pose"][:, 1] = 2.0
    fe = _fleet(e["params"], 8)
    try:
        long = _run(fe, e, 400, perception=SENSOR, tracker={})
        last = int(long["ticks"].max())
        assert last < 400 - 16
        short = _run(fe, e, last, perception=SENSOR, tracker={})
    finally:
        fe.close()
    _same(long, short, METRICS + ("unseen_personal_ticks", "untracked_personal_ticks", "track_rows",
                                  "mean_track_pos_error", "mean_track_vel_error"))
    for k in ("cmd_log", "optimized_log", "seen_log", "n_seen_log", "track_id_log"):
        assert np.array_equal(long[k][:, :last], short[k]), k
    assert not long["n_seen_log"][:, last:].any() and np.all(long["track_id_log"][:, last:] == -1)


@pytest.mark.parametrize("kind,per_tick", [("cv", 13), ("sfm1", 14), ("shared2", 16)])
def test_launches_per_tick(kind, per_tick):
    s = _scenes(kind, 3)
    fleet = _fleet(s["params"], s["pose"].shape[0])
    try:
        counts = {}
        for T in (1, 3):
            c0 = fleet.opt.launch_count()
            _run(fleet, s, T, want_logs=False, perception=SENSOR, tracker={})
            counts[T] = fleet.opt.launch_count() - c0
    finally:
        fleet.close()
    assert counts[1] == per_tick and counts[3] == 3 * per_tick, counts


def test_python_arguments():
    s = _scenes("cv", 3)
    fleet = _fleet(s["params"], s["pose"].shape[0])
    try:
        with pytest.raises(ValueError, match="perception"):
            _run(fleet, s, 3, tracker={})
        with pytest.raises(ValueError, match="vel_noise"):
            _run(fleet, s, 3, perception={}, tracker={})
        with pytest.raises(TypeError):
            _run(fleet, s, 3, perception=SENSOR, tracker=dict(latency=1))
        r = _run(fleet, s, 3, want_logs=False, perception=SENSOR, tracker=abi.tracker_params(latency_ticks=0))
        assert "track_id_log" not in r and "seen_log" not in r and r["track_rows"].shape == (s["pose"].shape[0],)
    finally:
        fleet.close()


def test_tracked_argument_errors_launch_nothing_and_leave_the_fleet_state():
    S, R = 3, 2
    B = S * R
    T = 10
    sh = sc.shared_episodes(S, R, 5, ticks=T, seed=4)
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
                                       ticks=T, robots_per_scene=R)
    goals = np.ascontiguousarray(sh["goals"])
    vdes = np.ascontiguousarray(sh["desired_speed"])
    dist, rmin, rint = np.zeros(B), np.zeros(B), np.zeros(B, np.int32)
    crowd = abi.SmpcCrowdIo(goals.ctypes.data, vdes.ctypes.data, 1, dist.ctypes.data, None)
    scene = abi.SmpcSceneIo(R, rmin.ctypes.data, rint.ctypes.data)
    table = abi.weight_row(p)[None].copy()
    idx = np.zeros(B, np.int32)
    ws = abi.SmpcWeightSets(1, table.ctypes.data, idx.ctypes.data)
    L = R - 1 + 5
    unseen, n_log, seen_log = np.zeros(B, np.int32), np.zeros((B, T), np.int32), np.zeros((B, T, L, 5))
    untracked, rows, pos, vel = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B), np.zeros(B)
    id_log = np.zeros((B, T, L), np.int32)
    lib = _lib.lib()

    def call(pover=None, tover=None, tfields=None, pfields=None, null_pc=False, null_tk=False, use_crowd=True,
             orca=None, w=None):
        pc = abi.perception_params(**dict(SENSOR, **(pover or {})))
        pc.unseen_personal_ticks = unseen.ctypes.data
        for f, v in (pfields or {}).items():
            setattr(pc, f, v)
        tk = abi.tracker_params(**(tover or {}))
        tk.untracked_personal_ticks, tk.track_rows = untracked.ctypes.data, rows.ctypes.data
        tk.track_pos_err, tk.track_vel_err = pos.ctypes.data, vel.ctypes.data
        for f, v in (tfields or {}).items():
            setattr(tk, f, v)
        c0 = a.opt.launch_count()
        rc = lib.smpc_run_tracked_episodes(a.opt._h, C.byref(io), C.byref(crowd) if use_crowd else None,
                                           C.byref(scene), None if w is None else C.byref(w),
                                           None if orca is None else C.byref(orca), None if null_pc else C.byref(pc),
                                           None if null_tk else C.byref(tk))
        if rc != 0:
            assert a.opt.launch_count() == c0
        return rc

    logs_on = dict(seen_log=seen_log.ctypes.data, n_seen_log=n_log.ctypes.data)
    try:
        first = tick(a)
        assert call(null_pc=True) == ARG
        assert call(null_tk=True) == ARG
        for f, bad in (("accel_noise", (-0.1, np.nan, np.inf)), ("meas_noise", (0.0, -0.1, np.nan, np.inf)),
                       ("init_vel_std", (0.0, np.nan, np.inf)), ("confirm_hits", (0, 17)),
                       ("max_coast_ticks", (-1, 65)), ("latency_ticks", (-1, 17))):
            for v in bad:
                assert call(tover={f: v}) == ARG, (f, v)
        assert call(pover=dict(vel_noise=0.1)) == ARG
        for f in ("untracked_personal_ticks", "track_rows", "track_pos_err", "track_vel_err"):
            assert call(tfields={f: None}) == ARG, f
        assert call(tfields=dict(track_id_log=id_log.ctypes.data)) == ARG  # without seen_log
        assert call(pfields=logs_on) == ARG  # seen_log without track_id_log
        assert call(pover=dict(detect_prob=1.5)) == ARG  # what run_perceived_episodes rejects
        assert call(pfields=dict(unseen_personal_ticks=None)) == ARG
        assert call(use_crowd=False) == ARG
        assert call(orca=abi.orca_params(max_neighbors=0)) == ARG
        assert call(w=abi.SmpcWeightSets(0, table.ctypes.data, idx.ctypes.data)) == ARG
        # the same blocks with valid parameters run, and leave the warm-start memory of optimize_batch alone
        assert call() == 0
        assert call(w=ws, orca=abi.orca_params(), pfields=logs_on, tfields=dict(track_id_log=id_log.ctypes.data)) == 0
        assert n_log[:, :2].sum() == 0 and np.all(id_log[:, :2] == -1)
        second = tick(a)
        want = [tick(b), tick(b)]
        for k in ("cmds", "path", "optimized", "n_out", "termination", "cost_final"):
            assert np.array_equal(first[k], want[0][k]) and np.array_equal(second[k], want[1][k]), k
    finally:
        a.close()
        b.close()
