"""CPU tests of the people tracker of smpc_run_tracked_episodes: its parameter block mirrors include/smpc.h, and the numpy
restatement the GPU tests compare with (tests/tracker_ref.py) is a constant-velocity Kalman filter that reaches the
Riccati steady state, follows a straight walk, coasts linearly, confirms, coasts and ends tracks as the header says,
and delivers its lists latency ticks late."""
import os
import re

import numpy as np
import pytest
import scipy.linalg

from nav2_social_mpc_controller_b200 import _lib, abi
from tests import perception_ref as pref
from tests import tracker_ref as tref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = 0.05


def test_tracker_struct_field_order_defaults_and_entry_match_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_tracker \{(.*?)\} smpc_tracker;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [d.strip().split()[-1].lstrip("*") for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in abi.SmpcTracker._fields_]
    assert re.search(r"int smpc_run_tracked_episodes\(smpc_handle\* h, smpc_episode_io\* io,", hdr)
    assert "smpc_run_tracked_episodes" in _lib.EXPORTED_SYMBOLS
    t = abi.tracker_params()
    assert {f: getattr(t, f) for f in tref.DEFAULTS} == tref.DEFAULTS
    assert not (t.untracked_personal_ticks or t.track_rows or t.track_pos_err or t.track_vel_err or t.track_id_log)
    assert abi.tracker_params(latency_ticks=5).latency_ticks == 5
    assert abi.TRACKER_PASS_THROUGH == tref.PASS_THROUGH
    with pytest.raises(TypeError):
        abi.tracker_params(latency=3)


def _walk(n, p0=(1.0, -2.0), v=(0.7, -0.4), prm=None, detect=None):
    """A track of a noise-free constant-velocity walk; detect(k) False: a miss at tick k. Returns the track and the
    per-tick (p, v) estimates."""
    prm = dict(tref.DEFAULTS, **(prm or {}))
    tr = tref.Track()
    est = []
    for k in range(n):
        z = (p0[0] + v[0] * k * DT, p0[1] + v[1] * k * DT)
        tr.step(z if detect is None or detect(k) else None, prm, DT)
        est.append((list(tr.p), list(tr.v)))
    return tr, est


@pytest.mark.parametrize("accel,meas", [(0.5, 0.05), (2.0, 0.02), (0.1, 0.3)])
def test_steady_state_covariance_is_the_riccati_solution(accel, meas):
    prm = dict(accel_noise=accel, meas_noise=meas)
    tr, _ = _walk(3000, prm=prm)
    F = np.array([[1.0, DT], [0.0, 1.0]])
    H = np.array([[1.0, 0.0]])
    q = tref.noise_terms(accel, DT)
    Q = np.array([[q[0], q[1]], [q[1], q[2]]])
    Rm = np.array([[meas * meas]])
    prior = scipy.linalg.solve_discrete_are(F.T, H.T, Q, Rm)  # the predicted covariance of the steady state
    post = prior - prior @ H.T @ np.linalg.inv(H @ prior @ H.T + Rm) @ H @ prior
    got = np.array([[tr.pp, tr.pv], [tr.pv, tr.vv]])
    assert np.allclose(got, post, rtol=1e-12, atol=0.0), (got, post)
    tr.predict(DT, q)
    assert np.allclose([[tr.pp, tr.pv], [tr.pv, tr.vv]], prior, rtol=1e-12, atol=0.0)


def test_noise_free_walk_velocity_converges():
    v = (0.7, -0.4)
    _, est = _walk(200, v=v)
    err = [np.hypot(e[1][0] - v[0], e[1][1] - v[1]) for e in est]
    assert err[0] == pytest.approx(np.hypot(*v))  # a new track starts at rest
    assert max(err[80:]) < 1e-6  # 4 s after the first detection with the default parameters
    assert err[5] > 1e-2 and max(err[40:60]) > 1e-6  # and not long before: the estimate lags and rings


def test_coasting_extrapolates_linearly():
    tr, est = _walk(200, v=(0.7, -0.4), prm=dict(max_coast_ticks=64), detect=lambda k: k < 150)
    p, v = est[149]
    for k in range(150, 200):
        m = k - 149
        assert est[k][1] == v  # the velocity is held
        assert np.allclose(est[k][0], [p[0] + m * DT * v[0], p[1] + m * DT * v[1]], rtol=0, atol=1e-12)
    assert tr.hits > 0 and tr.misses == 50


def _life(seq, confirm=3, coast=2):
    """Published flag and hits after each tick of a scripted detection sequence (1 detected, 0 missed)."""
    prm = dict(tref.DEFAULTS, confirm_hits=confirm, max_coast_ticks=coast)
    tr = tref.Track()
    pub, hits = [], []
    for k, d in enumerate(seq):
        tr.step((0.1 * k, 0.0) if d else None, prm, DT)
        pub.append(tr.published(prm))
        hits.append(tr.hits)
    return pub, hits


def test_confirm_coast_and_death():
    # confirmed at the third detection, coasts through two misses, dies at the third
    pub, hits = _life([1, 1, 1, 0, 0, 0, 1, 1, 1, 1])
    assert pub == [False, False, True, True, True, False, False, False, True, True]
    assert hits == [1, 2, 3, 3, 3, 0, 1, 2, 3, 4]  # re-born after the death, re-confirmed after 3 detections
    # a miss before confirmation keeps the hits; a detection resets the misses
    pub, hits = _life([1, 0, 1, 0, 0, 1, 0, 0, 0])
    assert pub == [False, False, False, False, False, True, True, True, False]
    # max_coast_ticks 0: the first miss ends the track; confirm 1: the first detection publishes
    pub, hits = _life([1, 0, 1, 1, 0], confirm=1, coast=0)
    assert pub == [True, False, True, True, False] and hits == [1, 0, 1, 2, 0]
    # hits saturate at 16
    _, hits = _life([1] * 40, confirm=16)
    assert max(hits) == tref.MAX_HITS and hits[-1] == tref.MAX_HITS
    # no detection, no track
    pub, hits = _life([0, 0, 0])
    assert pub == [False] * 3 and hits == [0] * 3


def test_pass_through_publishes_the_detections():
    prm = dict(tref.DEFAULTS, **tref.PASS_THROUGH)
    rt = tref.RobotTracker(3, prm, DT)
    z = [(1.0, 2.0), None, (3.0, -1.5)]
    for k in range(4):  # standing people: the estimate stays on the detection, the velocity at 0
        rows, ids = rt.tick([0, 1, 2], z)
        assert ids.tolist() == [0, 2]
        assert rows.tolist() == [[1.0, 2.0, 0.0, 0.0, 0.0], [3.0, -1.5, 0.0, 0.0, 0.0]]


@pytest.mark.parametrize("d", [0, 1, 2, 5])
def test_latency_delivers_the_list_of_tick_k_minus_d(d):
    prm = dict(tref.DEFAULTS, **dict(tref.PASS_THROUGH, latency_ticks=d))
    rt = tref.RobotTracker(2, prm, DT)
    published = []
    for k in range(12):
        z = [(float(k), 0.0) if k % 3 else None, (0.0, float(k))]  # person 0 missed every third tick
        rows, ids = rt.tick([0, 1], z)
        published.append(rt.history[k])
        if k < d:
            assert rows.shape == (0, 5) and ids.size == 0
        else:
            want_rows, want_ids = published[k - d]
            assert np.array_equal(rows, want_rows) and np.array_equal(ids, want_ids)


def test_tracked_all_counts_untracked_people_and_errors():
    # one robot at the origin, two standing people within 1.2 m; the default sensor parameters without noise or drops
    pprm = dict(pref.NEUTRAL)
    prm = dict(tref.DEFAULTS, confirm_hits=2, latency_ticks=1)
    lists = np.array([[[0.5, 0.0, 0.0, 0.0, 0.0], [0.0, 0.8, 0.3, 0.0, 0.0]]])
    rt = [tref.RobotTracker(2, prm, DT)]
    cm = np.zeros((1, 4, 4), np.uint8)
    got = [tref.tracked_all(rt, lists, [2], np.zeros((1, 3)), [True], k, pprm, cm, np.zeros((1, 2)), 0.05)
           for k in range(4)]
    assert [int(g["n_seen"][0]) for g in got] == [0, 0, 2, 2]  # confirmed at tick 1, delivered a tick later
    assert [bool(g["untracked"][0]) for g in got] == [True, True, False, False]
    assert not any(g["missed"][0] for g in got)
    assert got[2]["ids"][0].tolist() == [0, 1]
    assert got[2]["pos_err"][0] == 0.0  # standing still, measured exactly
    assert got[2]["vel_err"][0] == pytest.approx(0.3)  # person 1 walks at 0.3 m/s; the position does not show it
