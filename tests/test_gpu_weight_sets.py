"""GPU tests of per-robot critic weights (smpc_optimize_batch_weighted, smpc_run_weighted_episodes; the `weights=`
keyword of FleetOptimizer): a robot under row p of the table computes bit for bit what it computes on a handle whose
params carry row p, in fleet ticks and in every episode kind; launch counts are the unweighted entries'; invalid
tables are rejected before anything is launched."""
import ctypes as C

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from nav2_social_mpc_controller_b200.optimizer import weight_sets
from tests import episode_ref as ref
from tests import shared_ref as sref

pytestmark = pytest.mark.gpu

A = 3
ARG, UNSUP = -1, -3
METRICS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks", "collision_ticks",
           "not_optimized_ticks", "cmd_variation")
LOGS = ("pose_log", "cmd_log", "optimized_log")
CROWD_OUT = METRICS + LOGS + ("people_disturbance", "people_log")
SHARED_OUT = CROWD_OUT + ("robot_min_dist", "robot_intimate_ticks")
TICK_OUT = ("cmds", "path", "optimized", "n_out", "termination", "iterations", "cost_initial", "cost_final",
            "people_proj")
ROW3 = dict(proxemics_w=40.0, obstacle_w=0.3, velocity_feasibility_w=1.5)


def _fleet(p, B):
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    return FleetOptimizer(p, n_robots=B, n_agents=A)


def _args(s, **kw):
    a = {k: v for k, v in s.items() if k not in ("params", "ticks")}
    a.update(kw)
    return a


def _tick_scenes(B, seed, **overrides):
    """Fleet tick inputs: corridor scenes with 5 people each (the first A go to the optimizer) and trajectorizer seeds."""
    s = sc.episodes(B, 5, seed=seed, ticks=20, **overrides)
    poses, cmds = sc.pure_pursuit_seed(s["global_path"], s["pose"], s["params"])
    people = np.ascontiguousarray(s["people"][:, :A])
    return s, poses, cmds, people, np.full(B, A, np.int32)


def _tick(fleet, inputs, sel, weights=None):
    s, poses, cmds, people, n_people = inputs
    return fleet.optimize_batch(poses[sel], cmds[sel], people[sel], n_people[sel], s["speed"][sel], s["costmaps"],
                                s["costmap_origin"], s["costmap_resolution"], s["od"],
                                costmap_index=s["costmap_index"][sel], weights=weights)


def _device_trig():
    """cos / sin from the device's math library, which the scene view kernel uses."""
    import torch

    def f(fn):
        return lambda x: fn(torch.as_tensor(np.asarray(x, dtype=np.float64), device="cuda")).cpu().numpy()
    return f(torch.cos), f(torch.sin)


# 3 blocks: the 4-warp CTAs of the fleet tick's shape; 9 blocks (block length 2, horizon 18): the one-warp kernels
@pytest.mark.parametrize("blocks", [{}, dict(parameter_block_length=2)], ids=["nb3", "nb9"])
def test_fleet_tick_mixed_sets_equal_each_sets_own_tick(blocks):
    B = 12
    inputs = _tick_scenes(B, 21, **blocks)
    base = inputs[0]["params"]
    rows = [sc.make_params("obst_only", **blocks), sc.make_params("soc_work_obst", **blocks),
            sc.make_params("soc_work_obst", **blocks, **ROW3)]
    table = weight_sets(rows, base)
    idx = np.random.default_rng(5).permutation(np.arange(B) % 3).astype(np.int32)
    fw = _fleet(base, B)
    try:
        got = [_tick(fw, inputs, np.arange(B), (table, idx)) for _ in range(2)]  # tick 2 starts from tick 1's memory
    finally:
        fw.close()
    for p in range(3):
        sel = np.nonzero(idx == p)[0]
        fp = _fleet(rows[p], sel.size)
        try:
            want = [_tick(fp, inputs, sel) for _ in range(2)]
        finally:
            fp.close()
        for t in range(2):
            for k in TICK_OUT:
                assert np.array_equal(got[t][k][sel], want[t][k]), (p, t, k)
    assert got[0]["iterations"].max() > 0


def test_identity_table_is_the_unweighted_call():
    B = 8
    inputs = _tick_scenes(B, 22)
    p = inputs[0]["params"]
    ident = (abi.weight_row(p)[None], np.zeros(B, np.int32))
    a, b = _fleet(p, B), _fleet(p, B)
    try:
        for t in range(2):
            ra, rb = _tick(a, inputs, np.arange(B)), _tick(b, inputs, np.arange(B), ident)
            for k in TICK_OUT:
                assert np.array_equal(ra[k], rb[k]), (t, k)
        e = sc.episodes(B, 4, seed=3, ticks=40)
        x, y = (a.run_episodes(ticks=40, want_logs=True, weights=w, **_args(e)) for w in (None, ident))
        for k in METRICS + LOGS:
            assert np.array_equal(x[k], y[k]), k
        c = sc.crowd_episodes(B, 5, seed=4, ticks=40, substeps=2)
        x, y = (a.run_crowd_episodes(ticks=40, want_logs=True, weights=w, **_args(c)) for w in (None, ident))
        for k in CROWD_OUT:
            assert np.array_equal(x[k], y[k]), k
        sh = sc.shared_episodes(4, 2, 5, seed=6, ticks=40)
        x, y = (a.run_shared_episodes(ticks=40, want_logs=True, weights=w, **_args(sh)) for w in (None, ident))
        for k in SHARED_OUT:
            assert np.array_equal(x[k], y[k]), k
    finally:
        a.close()
        b.close()


def _mixed_episodes(kind, B0, T, seed, substeps=1):
    """P = 2 copies of B0 scenes (episode p * B0 + i = scene i) under obst_only (p = 0) and soc_work_obst (p = 1)."""
    s = (sc.episodes(B0, 4, seed=seed, ticks=T) if kind == "plain"
         else sc.crowd_episodes(B0, 5, seed=seed, ticks=T, substeps=substeps))
    rows = [sc.make_params("obst_only"), sc.make_params("soc_work_obst")]
    table = weight_sets(rows, s["params"])
    return s, rows, table, sc.tile_scenes(s, 2), np.repeat(np.arange(2), B0).astype(np.int32)


@pytest.mark.parametrize("kind,substeps", [("plain", 1), ("crowd", 1), ("crowd", 4)])
def test_episodes_mixed_sets_equal_each_sets_own_run(kind, substeps):
    B0, T = 6, 60
    s, rows, table, tiled, idx = _mixed_episodes(kind, B0, T, 8, substeps)
    run = "run_episodes" if kind == "plain" else "run_crowd_episodes"
    out = METRICS + LOGS if kind == "plain" else CROWD_OUT
    fw = _fleet(s["params"], 2 * B0)
    try:
        got = getattr(fw, run)(ticks=T, want_logs=True, weights=(table, idx), **_args(tiled))
    finally:
        fw.close()
    for p in range(2):
        fp = _fleet(rows[p], B0)
        try:  # s passes its explicit costmap_index: with NULL, episode b would use map b % M of the subset
            want = getattr(fp, run)(ticks=T, want_logs=True, **_args(s))
        finally:
            fp.close()
        for k in out:
            assert np.array_equal(got[k][p * B0:(p + 1) * B0], want[k]), (p, k)


def test_sets_change_behaviour():
    B0, T = 8, 40
    s, rows, table, tiled, idx = _mixed_episodes("crowd", B0, T, 12)
    fw = _fleet(s["params"], 2 * B0)
    try:
        got = fw.run_crowd_episodes(ticks=T, want_logs=True, weights=(table, idx), **_args(tiled))
    finally:
        fw.close()
    cl = got["cmd_log"]
    assert any(not np.array_equal(cl[i], cl[B0 + i]) for i in range(B0))


@pytest.mark.parametrize("R", [2, 3])
def test_shared_scenes_with_mixed_sets_replay_through_weighted_ticks(R):
    S, T = 4, 50
    s = sc.shared_episodes(S, R, 6, seed=15 + R, ticks=T)
    p, B, dt_c = s["params"], S * R, s["control_period"]
    table = weight_sets([sc.make_params("obst_only"), sc.make_params("soc_work_obst")], p)
    idx = (np.arange(B) % 2).astype(np.int32)  # both sets in every scene
    fleet, replay = _fleet(p, B), _fleet(p, B)
    cos, sin = _device_trig()
    try:
        got = fleet.run_shared_episodes(ticks=T, want_logs=True, weights=(table, idx), **_args(s))
        pl, cl, ol, ticks, ppl = got["pose_log"], got["cmd_log"], got["optimized_log"], got["ticks"], got["people_log"]
        H, W = s["costmaps"].shape[1:]
        speed = s["speed"].copy()
        done = np.zeros(B, bool)
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
                                      n_poses=n_poses, want_people_proj=False, weights=(table, idx))
            cmd = r["cmds"][:, 0]
            assert np.array_equal(cl[act, k], cmd[act]), k
            assert np.array_equal(ol[act, k], r["optimized"][act]), k
            want = ref.euler_step(pk[act], cl[act, k], dt_c)
            assert np.abs(pl[act, k + 1] - want).max() <= 1e-12, k
            speed[act] = cmd[act]
            done |= ticks == k + 1
        assert ol.any()
    finally:
        fleet.close()
        replay.close()


def test_launches_per_tick_match_the_unweighted_entries():
    B = 8
    inputs = _tick_scenes(B, 23)
    p = inputs[0]["params"]
    table = weight_sets([sc.make_params("obst_only"), p], p)
    idx = (np.arange(B) % 2).astype(np.int32)
    fleet = _fleet(p, B)

    def count(fn):
        c0 = fleet.opt.launch_count()
        fn()
        return fleet.opt.launch_count() - c0
    try:
        for w in (None, (table, idx)):  # warm both: the first tick of a fleet shape allocates
            _tick(fleet, inputs, np.arange(B), w)
        assert count(lambda: _tick(fleet, inputs, np.arange(B), (table, idx))) == \
            count(lambda: _tick(fleet, inputs, np.arange(B)))
        e = sc.episodes(B, 4, seed=3, ticks=3)
        c = sc.crowd_episodes(B, 5, seed=4, ticks=3)
        sh = sc.shared_episodes(4, 2, 5, seed=6, ticks=3)
        for name, s, per_tick in (("run_episodes", e, 12), ("run_crowd_episodes", c, 13),
                                  ("run_shared_episodes", sh, 15)):
            for T in (1, 3):
                plain = count(lambda: getattr(fleet, name)(ticks=T, **_args(s)))
                weighted = count(lambda: getattr(fleet, name)(ticks=T, weights=(table, idx), **_args(s)))
                assert weighted == plain == per_tick * T, (name, T, weighted, plain)
    finally:
        fleet.close()


def _bad_tables(P, B):
    """(name, smpc_weight_sets or None, arrays kept alive) for every invalid table of include/smpc.h."""
    good = np.ones((P, 9))
    idx = np.zeros(B, np.int32)
    out = [("NULL", None, ())]

    def ws(n, t, i):
        return abi.SmpcWeightSets(n, None if t is None else t.ctypes.data, None if i is None else i.ctypes.data)
    out.append(("n_sets 0", ws(0, good, idx), (good, idx)))
    out.append(("weights NULL", ws(P, None, idx), (idx,)))
    out.append(("set_index NULL", ws(P, good, None), (good,)))
    for v in (P, -1):
        i = idx.copy()
        i[B - 1] = v
        out.append((f"index {v}", ws(P, good, i), (good, i)))
    for v in (np.nan, np.inf, -np.inf):
        t = good.copy()
        t[P - 1, 5] = v
        out.append((f"weight {v}", ws(P, t, idx), (t, idx)))
    return out


def test_argument_errors_launch_nothing_and_leave_the_fleet_state(monkeypatch):
    B, P = 6, 2
    inputs = _tick_scenes(B, 24)
    p = inputs[0]["params"]
    table = weight_sets([sc.make_params("obst_only"), p], p)
    good = (table, (np.arange(B) % P).astype(np.int32))
    L = _lib.lib()
    real_tick, real_eps = L.smpc_optimize_batch_weighted, L.smpc_run_weighted_episodes

    def with_table(w):  # the keyword builds a valid table; the C entry gets w instead
        ref_w = None if w is None else C.byref(w)
        monkeypatch.setattr(L, "smpc_optimize_batch_weighted", lambda h, io, _: real_tick(h, io, ref_w))
        monkeypatch.setattr(L, "smpc_run_weighted_episodes", lambda h, io, cr, sc_, _: real_eps(h, io, cr, sc_, ref_w))

    def code_of(fleet, fn):
        c0 = fleet.opt.launch_count()
        with pytest.raises(_lib.SmpcError) as e:
            fn()
        assert fleet.opt.launch_count() == c0
        return e.value.code

    a, b = _fleet(p, B), _fleet(p, B)
    e = sc.episodes(B, 4, seed=3, ticks=5)
    c = sc.crowd_episodes(B, 5, seed=4, ticks=5)
    sh = sc.shared_episodes(3, 2, 5, seed=6, ticks=5)
    try:
        first = _tick(a, inputs, np.arange(B), good)
        for name, w, keep in _bad_tables(P, B):
            with_table(w)
            assert code_of(a, lambda: _tick(a, inputs, np.arange(B), good)) == ARG, name
            assert code_of(a, lambda: a.run_episodes(ticks=5, weights=good, **_args(e))) == ARG, name
            assert code_of(a, lambda: a.run_crowd_episodes(ticks=5, weights=good, **_args(c))) == ARG, name
            assert code_of(a, lambda: a.run_shared_episodes(ticks=5, weights=good, **_args(sh))) == ARG, name
            monkeypatch.undo()
        # a scene needs a crowd
        io, out, logs, keep = a.episode_io(**{k: v for k, v in _args(sh).items()
                                              if k not in ("goals", "desired_speed", "substeps", "robots_per_scene")},
                                           ticks=5, robots_per_scene=2)
        rmin, rint = np.zeros(B), np.zeros(B, np.int32)
        scene = abi.SmpcSceneIo(2, rmin.ctypes.data, rint.ctypes.data)
        idx = np.ascontiguousarray(good[1])
        w = abi.SmpcWeightSets(P, table.ctypes.data, idx.ctypes.data)
        c0 = a.opt.launch_count()
        assert L.smpc_run_weighted_episodes(a.opt._h, C.byref(io), None, C.byref(scene), C.byref(w)) == ARG
        assert a.opt.launch_count() == c0
        # the fleet state is untouched: the next tick equals that of a fleet that never saw the errors
        second = _tick(a, inputs, np.arange(B), good)
        want = [_tick(b, inputs, np.arange(B), good) for _ in range(2)]
        for k in TICK_OUT:
            assert np.array_equal(first[k], want[0][k]) and np.array_equal(second[k], want[1][k]), k
    finally:
        a.close()
        b.close()
    omni = _fleet(sc.make_params("soc_work_obst", omni_solve=1), B)
    try:
        assert code_of(omni, lambda: _tick(omni, inputs, np.arange(B), good)) == UNSUP
        assert code_of(omni, lambda: omni.run_episodes(ticks=5, weights=good, **_args(e))) == UNSUP
    finally:
        omni.close()
