"""GPU tests of the local-costmap episode entry smpc_run_local_costmap_episodes (FleetOptimizer.run_episodes /
run_crowd_episodes / run_shared_episodes with local_costmap=...): every logged window is the numpy build of
tests/local_costmap_ref.py from the logged pose and the true people of its tick, every tick replays through the public
path (trajectorize_batch, filter_people_fov and optimize_batch on the logged windows), a person ahead stays out of the
controller's input until the window reaches them, and a marked person pushes the robot away through the obstacle
critic alone."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from tests import episode_ref as ref
from tests import local_costmap_ref as lref
from tests import shared_ref as sref

pytestmark = pytest.mark.gpu

A = 3
ARG = -1
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
LOGS = ("pose_log", "cmd_log", "optimized_log")
LOCAL = ("marked_rows", "local_costmap_log", "local_origin_log")
SENSOR = dict(vel_noise=0.0)  # the default sensor, reporting positions only (what the tracker needs)


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


def _static(s, b):
    m = s["costmap_index"][b]
    return s["costmaps"][m], s["costmap_origin"][m]


def _check_builds(s, got, prm, lists_at):
    """Every build's window, origin and the marked_rows sums against the numpy build from the logged pose and
    lists_at(k) = (rows [B][L][5], n [B]) of build tick k; builds after an episode is done are zero with NaN origins."""
    B, n = s["pose"].shape[0], prm["update_period_ticks"]
    sten, hw, _ = lref.stencil(prm, s["costmap_resolution"])
    wl, ol, ticks = got["local_costmap_log"], got["local_origin_log"], got["ticks"]
    marked = np.zeros(B, np.int32)
    for j in range(wl.shape[1]):
        k = j * n
        rows, n_rows = lists_at(k)
        for b in range(B):
            if k >= ticks[b]:
                assert not wl[b, j].any() and np.all(np.isnan(ol[b, j])), (b, j)
                continue
            static, origin = _static(s, b)
            win, org, m = lref.build(static, origin, s["costmap_resolution"], got["pose_log"][b, k], rows[b],
                                     n_rows[b], prm, sten, hw)
            assert np.array_equal(ol[b, j], org), (b, j)
            assert np.array_equal(wl[b, j], win), (b, j, np.argwhere(wl[b, j] != win)[:5])
            marked[b] += m
    assert np.array_equal(got["marked_rows"], marked)
    return marked


def test_static_crop_without_people():
    T = 40
    s = sc.episodes(8, 6, ticks=T, n_maps=2, seed=11)
    prm = dict(lref.DEFAULTS, mark_people=0, update_period_ticks=3)
    fleet = _fleet(s["params"], 8)
    try:
        got = _run(fleet, s, T, local_costmap=prm)
    finally:
        fleet.close()
    assert got["local_costmap_log"].shape == (8, 14, 80, 80) and got["local_origin_log"].shape == (8, 14, 2)
    _check_builds(s, got, prm, lambda k: (np.zeros((8, 0, 5)), np.zeros(8, np.int32)))
    assert np.all(got["marked_rows"] == 0)
    assert (got["local_origin_log"][:, 0, 0] < 0.0).all()  # the first windows stick out of the map's end


# period 4 without a sensor and period 1 with the sensor and the tracker, for every scene kind
@pytest.mark.parametrize("kind", ["cv", "sfm1", "sfm4", "orca", "shared2", "shared3"])
@pytest.mark.parametrize("period,tracked", [(4, False), (1, True)])
def test_windows_byte_for_byte_and_replay_through_the_public_path(kind, period, tracked):
    T = 40
    s = _scenes(kind, T)
    R = s.get("robots_per_scene", 1)
    p, dt_c, res = s["params"], s["control_period"], s["costmap_resolution"]
    B = s["pose"].shape[0]
    prm = dict(lref.DEFAULTS, update_period_ticks=period)
    extra = dict(perception=SENSOR, tracker={}) if tracked else {}
    fleet, replay = _fleet(p, B), _fleet(p, B)
    cos, sin = _device_trig()
    try:
        got = _run(fleet, s, T, local_costmap=prm, **extra, **_kw(kind))
        pl, cl, ol, ticks = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"]
        speeds = np.empty((T, B, 2))  # the measured speed of every tick, for the scene views
        speeds[0] = s["speed"]
        for k in range(1, T):
            speeds[k] = np.where((ticks > k - 1)[:, None], cl[:, k - 1], speeds[k - 1])

        def lists_at(k):
            if kind == "cv":
                return ref.people_at(s["people"], k * dt_c), s["n_people"]
            if R == 1:
                return got["people_log"][:, k], s["n_people"]
            return sref.scene_views(pl[:, k], speeds[k], ticks > k, got["people_log"][:, k], s["n_people"], R,
                                    cos=cos, sin=sin)

        marked = _check_builds(s, got, prm, lists_at)
        assert marked.sum() > 0
        sy, sx = prm["size_y"], prm["size_x"]
        windows = [np.ascontiguousarray(got["local_costmap_log"][:, j]) for j in range(got["local_costmap_log"].shape[1])]
        origins = [np.nan_to_num(got["local_origin_log"][:, j]) for j in range(len(windows))]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
        for k in range(T):
            pk = pl[:, k]
            act = ~done
            if tracked:
                rows, n_rows = got["seen_log"][:, k], got["n_seen_log"][:, k]
            else:
                rows, n_rows = lists_at(k)
            j = k // period
            poses, cmds3, n_steps = replay.trajectorize_batch(s["global_path"], pk)
            cmds = np.ascontiguousarray(cmds3[:, :, [0, 2]])
            fp, fn = replay.filter_people_fov(rows, n_rows, pk, origins[j], sx, sy, res)
            n_poses = np.where(done, 0, n_steps + 1).astype(np.int32)
            r = replay.optimize_batch(poses, cmds, fp, fn, speed, windows[j], origins[j], res, s["od"],
                                      n_poses=n_poses, want_people_proj=False)
            cmd = r["cmds"][:, 0]
            assert np.array_equal(cl[act, k], cmd[act]), k
            assert np.array_equal(ol[act, k], r["optimized"][act]), k
            speed[act] = cmd[act]
            done |= ticks == k + 1
    finally:
        fleet.close()
        replay.close()


def test_a_person_ahead_is_unseen_until_the_window_reaches_them():
    T = 80
    s = sc.episodes(2, 1, ticks=T, seed=3)
    s["pose"][:, 1:] = [2.0, 0.0]
    s["people"][:, 0] = [4.02, 2.0, 0.0, 0.0, 0.0]  # standing 3 m ahead on the path, in static cell column 80
    nobody = dict(s, n_people=np.zeros(2, np.int32))
    prm = dict(lref.DEFAULTS, mark_people=0)
    fleet = _fleet(s["params"], 2)
    try:
        win = _run(fleet, s, T, local_costmap=prm)
        alone = _run(fleet, nobody, T, local_costmap=prm)
        full = _run(fleet, s, T)
        seen = np.array([fleet.filter_people_fov(s["people"], s["n_people"], win["pose_log"][:, k],
                                                 win["local_origin_log"][:, k // prm["update_period_ticks"]],
                                                 80, 80, s["costmap_resolution"])[1] for k in range(T)]).T
    finally:
        fleet.close()
    enter = int(np.argmax(seen[0] > 0))
    org = win["local_origin_log"][0, np.arange(T) // prm["update_period_ticks"], 0]
    inside = (s["people"][0, 0, 0] - org) / s["costmap_resolution"] < 80
    assert enter > 8 and not seen[0, :enter].any() and not inside[:enter].any() and inside[enter], (seen[0], inside)
    # the controller's input is the empty list until then: what it computes alone in the corridor
    assert np.array_equal(win["cmd_log"][:, :enter], alone["cmd_log"][:, :enter])
    assert not np.array_equal(win["cmd_log"], alone["cmd_log"])
    assert not np.array_equal(full["cmd_log"][:, :enter], alone["cmd_log"][:, :enter])  # the whole map shows them


# The obstacle critic as the only people term: the social-work, agent-angle and proxemics weights are 0 and the
# obstacle weight is 1.0, about 8x the benchmark's 0.13, so that a marked person is a clear obstacle next to the path.
OBSTACLE_ONLY = dict(socialwork_w=0.0, agent_angle_w=0.0, proxemics_w=0.0, obstacle_w=1.0)


def test_a_marked_person_beside_the_path_is_avoided_by_the_obstacle_critic():
    T = 120
    s = sc.episodes(4, 1, ticks=T, seed=3)
    s["pose"][:, 1:] = [2.0, 0.0]
    s["people"][:, 0] = [3.5, 2.45, 0.0, 0.0, 0.0]  # standing 0.45 m beside the path
    row = abi.weight_row(s["params"])
    for k, v in OBSTACLE_ONLY.items():
        row[abi.WEIGHT_NAMES.index(k)] = v
    w = (row[None], np.zeros(4, np.int32))
    fleet = _fleet(s["params"], 4)
    try:
        off = _run(fleet, s, T, weights=w, local_costmap=dict(mark_people=0))
        on = _run(fleet, s, T, weights=w, local_costmap={})
    finally:
        fleet.close()
    assert np.all(on["marked_rows"] > 0) and np.all(off["marked_rows"] == 0)
    assert np.all(on["min_person_dist"] > off["min_person_dist"]), (on["min_person_dist"], off["min_person_dist"])


@pytest.mark.parametrize("kind", ["cv", "sfm1", "shared2"])
def test_launches_per_tick_add_one_on_build_ticks(kind):
    s = _scenes(kind, 9)
    fleet = _fleet(s["params"], s["pose"].shape[0])
    try:
        for extra in ({}, dict(perception=SENSOR, tracker={})):
            counts = {}
            for T in (1, 5, 9):
                for local in (None, dict(update_period_ticks=4)):
                    c0 = fleet.opt.launch_count()
                    _run(fleet, s, T, want_logs=False, local_costmap=local, **extra)
                    counts[T, local is None] = fleet.opt.launch_count() - c0
            for T, builds in ((1, 1), (5, 2), (9, 3)):
                assert counts[T, False] == counts[T, True] + builds, (extra, counts)
    finally:
        fleet.close()


def test_determinism_early_stop_and_tiled_copies():
    B0, T = 6, 40
    s = sc.crowd_episodes(B0, 5, seed=8, ticks=T, substeps=2)
    p = s["params"]
    fleet = _fleet(p, B0)
    try:
        x, y = _run(fleet, s, T, local_costmap={}), _run(fleet, s, T, local_costmap={})
    finally:
        fleet.close()
    _same(x, y, METRICS + LOGS + LOCAL + ("people_disturbance",))
    # copies of the scenes under an identity weight table compute the same windows and commands
    t = sc.tile_scenes(s, 2)
    row = abi.weight_row(p)
    fw = _fleet(p, 2 * B0)
    try:
        got = _run(fw, t, T, weights=(np.stack([row, row]), np.repeat(np.arange(2), B0).astype(np.int32)),
                   local_costmap={})
    finally:
        fw.close()
    for k in METRICS + LOGS + LOCAL:
        assert np.array_equal(got[k][:B0], got[k][B0:], equal_nan=True), k
        assert np.array_equal(got[k][:B0], x[k], equal_nan=True), k
    # an early stop gives the results of the run that ends at the last arrival tick
    e = sc.episodes(8, 2, ticks=400, seed=5, path_length=1.2)
    e["pose"][:, 1] = 2.0
    fe = _fleet(e["params"], 8)
    try:
        long = _run(fe, e, 400, local_costmap={})
        last = int(long["ticks"].max())
        assert last < 400 - 16
        short = _run(fe, e, last, local_costmap={})
    finally:
        fe.close()
    _same(long, short, METRICS + ("marked_rows",))
    nb = -(-last // 4)
    assert np.array_equal(long["local_costmap_log"][:, :nb], short["local_costmap_log"])
    assert np.array_equal(long["local_origin_log"][:, :nb], short["local_origin_log"], equal_nan=True)
    assert not long["local_costmap_log"][:, nb:].any() and np.all(np.isnan(long["local_origin_log"][:, nb:]))


def test_python_arguments():
    s = _scenes("cv", 3)
    fleet = _fleet(s["params"], s["pose"].shape[0])
    try:
        with pytest.raises(ValueError, match="size"):
            _run(fleet, s, 3, local_costmap=dict(size=40))
        with pytest.raises(ValueError, match="perception"):
            _run(fleet, s, 3, tracker={}, local_costmap={})
        r = _run(fleet, s, 3, want_logs=False, local_costmap=abi.local_costmap_params(size_x=41, size_y=33))
        assert "local_costmap_log" not in r and r["marked_rows"].shape == (s["pose"].shape[0],)
        r = _run(fleet, s, 3, local_costmap=dict(size_x=41, size_y=33, update_period_ticks=2))
        assert r["local_costmap_log"].shape == (8, 2, 33, 41)  # an odd-sized window: byte stores
    finally:
        fleet.close()


def test_local_costmap_argument_errors_launch_nothing_and_leave_the_fleet_state():
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
    marked = np.zeros(B, np.int32)
    wlog, olog = np.zeros((B, 3, 80, 80), np.uint8), np.zeros((B, 3, 2))
    unseen = np.zeros(B, np.int32)
    lib = _lib.lib()

    def call(lover=None, lfields=None, null_lc=False, use_crowd=True, use_scene=True, orca=None, w=None, pc=None,
             tk=None):
        lc = abi.local_costmap_params(**(lover or {}))
        lc.marked_rows = marked.ctypes.data
        for f, v in (lfields or {}).items():
            setattr(lc, f, v)
        c0 = a.opt.launch_count()
        rc = lib.smpc_run_local_costmap_episodes(a.opt._h, C.byref(io), C.byref(crowd) if use_crowd else None,
                                                 C.byref(scene) if use_scene else None,
                                                 None if w is None else C.byref(w),
                                                 None if orca is None else C.byref(orca),
                                                 None if pc is None else C.byref(pc),
                                                 None if tk is None else C.byref(tk), None if null_lc else C.byref(lc))
        if rc != 0:
            assert a.opt.launch_count() == c0
        return rc

    def perception(**over):
        pc = abi.perception_params(**dict(SENSOR, **over))
        pc.unseen_personal_ticks = unseen.ctypes.data
        return pc

    try:
        first = tick(a)
        assert call(null_lc=True) == ARG
        for f, bad in (("size_x", (7, 257)), ("size_y", (0, 300)), ("update_period_ticks", (0, 21)),
                       ("mark_people", (-1, 2)), ("agent_radius", (-0.1, np.nan, np.inf)),
                       ("inscribed_radius", (-0.1, np.nan)), ("cost_scaling_factor", (0.0, -1.0, np.nan, np.inf)),
                       ("inflation_radius", (np.nan, np.inf, 2.0))):
            for v in bad:
                assert call(lover={f: v}) == ARG, (f, v)
        assert call(lover=dict(inscribed_radius=0.3, inflation_radius=0.2)) == ARG
        assert call(lfields=dict(marked_rows=None)) == ARG
        assert call(lfields=dict(costmap_log=wlog.ctypes.data)) == ARG
        assert call(lfields=dict(origin_log=olog.ctypes.data)) == ARG
        assert call(tk=abi.tracker_params()) == ARG  # a tracker without perception
        assert call(pc=perception(detect_prob=1.5)) == ARG  # what the perceived entry rejects
        assert call(pc=perception(vel_noise=0.1), tk=abi.tracker_params()) == ARG  # what the tracked entry rejects
        assert call(use_crowd=False) == ARG  # a scene without a crowd
        assert call(orca=abi.orca_params(max_neighbors=0)) == ARG
        assert call(w=abi.SmpcWeightSets(0, table.ctypes.data, idx.ctypes.data)) == ARG
        # the same blocks with valid parameters run, and leave the warm-start memory of optimize_batch alone
        assert call() == 0
        ws = abi.SmpcWeightSets(1, table.ctypes.data, idx.ctypes.data)
        assert call(w=ws, orca=abi.orca_params(), lfields=dict(costmap_log=wlog.ctypes.data,
                                                                origin_log=olog.ctypes.data)) == 0
        assert wlog[:, 0].any() and np.isfinite(olog[:, 0]).all()
        second = tick(a)
        want = [tick(b), tick(b)]
        for k in ("cmds", "path", "optimized", "n_out", "termination", "cost_final"):
            assert np.array_equal(first[k], want[0][k]) and np.array_equal(second[k], want[1][k]), k
    finally:
        a.close()
        b.close()
