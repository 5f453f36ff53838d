"""CPU tests of the closed-loop episode entry (smpc_run_episodes): its argument block mirrors include/smpc.h, the numpy
world / metric reference the GPU tests compare with agrees with hand-computed cases, and the episode scenes keep every
person inside the obstacle-distance grid for the whole run (a person outside it makes the reference throw)."""
import math
import os
import re

import numpy as np

from nav2_social_mpc_controller_b200 import abi, scenarios as sc
from tests import episode_ref as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_episode_io_field_order_matches_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_episode_io \{(.*?)\} smpc_episode_io;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [re.sub(r"\[.*\]", "", d.strip().split()[-1].lstrip("*")) for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in abi.SmpcEpisodeIo._fields_]
    assert abi.SMPC_ABI_VERSION == 4
    assert re.search(r"#define SMPC_ABI_VERSION 4\b", hdr)


def test_euler_step_and_people_by_hand():
    # straight ahead at 0.5 m/s for 0.1 s, then a quarter turn in place
    p1 = ref.euler_step([1.0, 2.0, 0.0], [0.5, 0.0], 0.1)
    assert np.allclose(p1, [1.05, 2.0, 0.0], atol=1e-15)
    p2 = ref.euler_step([0.0, 0.0, math.pi / 2], [1.0, 0.0], 0.5)
    assert abs(p2[0]) < 1e-15 and p2[1] == 0.5 and abs(p2[2] - math.pi / 2) < 1e-15
    p3 = ref.euler_step([0.0, 0.0, 3.0], [0.0, 2.0], 0.1)  # yaw wraps through setRPY / getYaw
    assert np.isclose(p3[2], 3.2 - 2 * math.pi, atol=1e-14)
    ppl = ref.people_at(np.array([[1.0, 1.0, 0.5, -0.25, 0.1]]), 2.0)
    assert ppl.tolist() == [[2.0, 0.5, 0.5, -0.25, 0.1]]


def test_metrics_from_logs_by_hand():
    # one episode, three ticks along +x at 0.5 m/s (dt 0.1), a person standing at (1.1, 0.5), goal at x = 1.2
    dt = 0.1
    pose_log = np.array([[[1.0, 0.0, 0.0], [1.05, 0.0, 0.0], [1.1, 0.0, 0.0], [1.2, 0.0, 0.0]]])
    cmd_log = np.array([[[0.5, 0.0], [0.5, 0.2], [0.3, 0.0]]])
    opt_log = np.array([[True, False, True]])
    people = np.array([[[1.1, 0.5, 0.0, 0.0, 0.0]]])
    gpath = np.array([[[1.0, 0.0], [1.2, 0.0]]])
    cm = np.zeros((1, 10, 40), np.uint8)
    cm[0, 0, 22] = 254  # the cell under (1.1, 0.0) at 0.05 m
    m = ref.metrics_from_logs(pose_log, cmd_log, opt_log, [3], people, [1], gpath, cm, np.zeros((1, 2)), 0.05, None,
                              dt, 0.02)
    assert np.isclose(m["path_length"][0], 0.2, atol=1e-12)
    assert np.isclose(m["min_person_dist"][0], 0.5, atol=1e-12)  # at tick 1 the robot is right below the person
    assert m["intimate_ticks"][0] == 0 and m["personal_ticks"][0] == 3
    assert m["collision_ticks"][0] == 1 and m["not_optimized_ticks"][0] == 1
    assert np.isclose(m["cmd_variation"][0], 0.2 + 0.2 + 0.2, atol=1e-12)
    assert m["reached"][0] and m["goal_first"][0] == 2
    # no people: +inf and no proximity counts; off the map reads as lethal
    m = ref.metrics_from_logs(pose_log - [5.0, 0.0, 0.0], cmd_log, opt_log, [3], people, [0], gpath, cm,
                              np.zeros((1, 2)), 0.05, None, dt, 0.02)
    assert m["min_person_dist"][0] == np.inf and m["personal_ticks"][0] == 0
    assert m["collision_ticks"][0] == 3 and not m["reached"][0]


def test_episode_scenes_keep_people_inside_the_obstacle_grid():
    for B, K, T in ((64, 20, 200), (8, 6, 60), (3, 1, 400)):
        s = sc.episodes(B, K, ticks=T, seed=B)
        od, p = s["od"], s["params"]
        horizon = T * s["control_period"] + sc.f32(p.max_time)
        t = np.linspace(0.0, horizon, 241)
        ppl = s["people"]
        x = ppl[:, :, 0, None] + ppl[:, :, 2, None] * t
        y = ppl[:, :, 1, None] + ppl[:, :, 3, None] * t
        W, H = od["width"] * od["resolution"], od["height"] * od["resolution"]
        m = sc.EPISODE_MARGIN - 1e-9
        assert x.min() >= m and y.min() >= m and x.max() <= W - m and y.max() <= H - m, (B, K, T)
        v = np.hypot(ppl[:, :, 2], ppl[:, :, 3])
        assert v.min() >= 0.3 - 1e-12 and v.max() <= 1.2 + 1e-12
        assert np.all(s["n_people"] == K)
        # the robot starts in free space of its corridor and its path ends inside the map
        cms = s["costmaps"]
        for b in range(B):
            cm = cms[s["costmap_index"][b]]
            assert ref.cell_cost(cm, (0.0, 0.0), 0.05, *s["pose"][b, :2]) < 253
        assert s["global_path"][:, -1, 0].max() < W
