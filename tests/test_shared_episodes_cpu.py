"""CPU tests of the shared-scene episode entry (smpc_run_shared_episodes): its argument block mirrors include/smpc.h,
the numpy crowd step with one robot is the one-robot reference, and the generated shared scenes keep their rules."""
import os
import re

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import abi, scenarios as sc
from tests import crowd_ref as cref
from tests import shared_ref as sref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_scene_io_field_order_matches_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_scene_io \{(.*?)\} smpc_scene_io;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [d.strip().split()[-1].lstrip("*") for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in abi.SmpcSceneIo._fields_]
    assert re.search(r"int smpc_run_shared_episodes\(smpc_handle\* h, smpc_episode_io\* io, const smpc_crowd_io\* crowd,"
                     r"\s+const smpc_scene_io\* scene\);", hdr)


@pytest.mark.parametrize("substeps", [1, 3])
def test_one_robot_crowd_step_is_the_crowd_reference(substeps):
    s = sc.crowd_episodes(4, 7, seed=3)
    od = cref.od_of(s["od"])
    for b in range(4):
        flags = np.ones(7, bool)
        flags[b] = False
        cmd = [0.4, 0.1]
        want = cref.crowd_step(s["people"][b], flags, s["goals"][b], s["desired_speed"][b], s["pose"][b], cmd, od,
                               0.05, substeps, near_eps=1e-9)
        got = sref.crowd_step(s["people"][b], flags, s["goals"][b], s["desired_speed"][b], s["pose"][b:b + 1], [cmd],
                              [True], od, 0.05, substeps, near_eps=1e-9)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and np.array_equal(got[3], want[3])
        assert got[2].shape == (1,) and got[2][0] == want[2]


def test_finished_robot_stands_still_and_a_second_robot_adds_its_force():
    s = sc.crowd_episodes(1, 3, seed=4)
    od = cref.od_of(s["od"])
    args = (s["people"][0], np.ones(3, bool), s["goals"][0], s["desired_speed"][0])
    far = [100.0, 100.0, 0.0]
    alone = sref.crowd_step(*args, [s["pose"][0], far], [[0.5, 0.0], [0.8, 0.0]], [True, False], od, 0.05, 2)
    parked = cref.crowd_step(*args, far, [0.0, 0.0], od, 0.05, 2)
    # the finished robot's force is that of a robot standing at its pose: compare against the pair in either order
    both = sref.crowd_step(*args, [far, s["pose"][0]], [[0.0, 0.0], [0.5, 0.0]], [False, True], od, 0.05, 2)
    assert np.allclose(alone[0], both[0], rtol=0, atol=1e-15)
    assert alone[2][0] == both[2][1] and alone[2][1] == both[2][0]
    assert alone[2][1] < 1e-50 and parked[2] < 1e-50


@pytest.mark.parametrize("S,R,K,seed", [(32, 2, 20, 6), (16, 3, 9, 1), (16, 4, 12, 2), (8, 1, 5, 3), (4, 4, 0, 5)])
def test_shared_scenes_keep_spacing_clearance_and_margins(S, R, K, seed):
    s = sc.shared_episodes(S, R, K, seed=seed, ticks=200)
    again = sc.shared_episodes(S, R, K, seed=seed, ticks=200)
    for k, v in s.items():
        if k not in ("params", "od"):
            assert np.array_equal(np.asarray(v), np.asarray(again[k])), k
    B = S * R
    p = s["params"]
    assert s["global_path"].shape[0] == B and s["pose"].shape == (B, 3) and s["speed"].shape == (B, 2)
    assert s["people"].shape == (S, K, 5) and s["goals"].shape == (S, K, 2) and s["n_people"].shape == (S,)
    assert s["costmap_index"].shape == (B,) and s["robots_per_scene"] == R
    assert np.all(s["costmap_index"].reshape(S, R) == s["costmap_index"][::R, None])
    gp, pose = s["global_path"], s["pose"]
    assert np.array_equal(gp[:, 0], pose[:, :2])
    fwd = np.arange(B) % R % 2 == 0
    assert np.all((gp[fwd, -1, 0] > gp[fwd, 0, 0])) and np.all(gp[~fwd, -1, 0] < gp[~fwd, 0, 0])
    assert np.all(np.abs(gp[..., 1] - 2.0) <= sc.SHARED_LATERAL) and np.all(gp[..., 1] == gp[:, :1, 1])
    od = s["od"]
    margin = sc.EPISODE_MARGIN + 0.5 * sc.f32(p.max_time)
    assert gp[..., 0].min() >= margin - 1e-9 and gp[..., 0].max() <= od["width"] * od["resolution"] - margin + 1e-9
    res = s["costmap_resolution"]
    start = pose[:, :2].reshape(S, R, 2)
    for c in range(S):
        d = np.hypot(start[c, :, None, 0] - start[c, None, :, 0], start[c, :, None, 1] - start[c, None, :, 1])
        d[np.arange(R), np.arange(R)] = np.inf
        assert d.min() >= sc.SHARED_SPACING
        f = np.arange(R) % 2 == 0
        for same in (f, ~f):
            xs = np.sort(start[c, same, 0])
            assert np.all(np.diff(xs) >= sc.SHARED_STAGGER - 1e-9)
        cm = s["costmaps"][s["costmap_index"][c * R]]
        ly, lx = np.nonzero(cm >= 253)
        cx, cy = (lx + 0.5) * res, (ly + 0.5) * res
        for r in range(R):
            assert np.hypot(cx - start[c, r, 0], cy - start[c, r, 1]).min() >= sc.CROWD_CLEARANCE
            if K:
                ppl = s["people"][c, :, :2]
                assert np.hypot(ppl[:, 0] - start[c, r, 0], ppl[:, 1] - start[c, r, 1]).min() >= sc.CROWD_CLEARANCE


def test_too_many_robots_for_the_corridor_are_refused():
    with pytest.raises(ValueError):
        sc.shared_episodes(2, 8, 4)
