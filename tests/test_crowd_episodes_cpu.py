"""CPU tests of the reactive-crowd episode entry (smpc_run_crowd_episodes): its argument block mirrors include/smpc.h,
the numpy crowd reference the GPU tests compare with behaves as the social force model should in hand-built cases, and
the generated crowd scenes keep the spacing, margins and speeds they promise."""
import math
import os
import re

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import abi, scenarios as sc
from tests import crowd_ref as cref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _open_od(w=400, h=400, res=0.05):
    """A grid whose nearest-obstacle index is out of range everywhere: no obstacle force."""
    return dict(width=w, height=h, resolution=res, origin_x=0.0, origin_y=0.0,
                indexes=np.full(w * h, w * h, dtype=np.uint32))


FAR_ROBOT = ([100.0, 100.0, 0.0], [0.0, 0.0])


def test_crowd_io_field_order_matches_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_crowd_io \{(.*?)\} smpc_crowd_io;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [re.sub(r"\[.*\]", "", d.strip().split()[-1].lstrip("*")) for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in abi.SmpcCrowdIo._fields_]
    assert re.search(r"int smpc_run_crowd_episodes\(smpc_handle\* h, smpc_episode_io\* io, const smpc_crowd_io\* crowd\);",
                     hdr)


def test_lone_person_reaches_its_goal_clears_it_and_brakes():
    od = _open_od()
    p = np.array([[2.0, 2.0, 0.0, 0.0, 0.0]])
    goal, vdes, flag = np.array([[6.0, 2.0]]), np.array([0.8]), np.array([True])
    speeds, cleared_at = [], None
    for k in range(200):
        p, flag, dist = cref.crowd_step(p, flag, goal, vdes, *FAR_ROBOT, od, 0.05, 2)
        assert dist < 1e-50  # the robot is 140 m away
        speeds.append(math.hypot(p[0, 2], p[0, 3]))
        if not flag[0] and cleared_at is None:
            cleared_at = k
    assert 0.8 - 1e-6 < max(speeds) <= 0.8 + 1e-15  # accelerates to the desired speed and no further
    assert cleared_at is not None and abs(p[0, 1] - 2.0) < 1e-12
    assert math.hypot(p[0, 0] - 6.0, p[0, 1] - 2.0) < 0.25 + 0.8 * 0.5 + 1e-9  # braking: v decays over 0.5 s
    assert speeds[cleared_at + 20] < 0.2 * speeds[cleared_at]  # -v / 0.5 for 1 s: e^-2
    assert speeds[-1] < 1e-3


def test_mirrored_people_get_mirrored_forces():
    od = _open_od()
    # two people mirrored about y = 2, walking toward each other's side
    p = np.array([[2.0, 1.6, 0.5, 0.3, 0.0], [2.0, 2.4, 0.5, -0.3, 0.0]])
    goals = np.array([[5.0, 1.0], [5.0, 3.0]])
    vdes = np.array([0.9, 0.9])
    q, flags, _ = cref.crowd_step(p, [True, True], goals, vdes, *FAR_ROBOT, od, 0.05, 1)
    assert q[0, 0] == pytest.approx(q[1, 0], abs=1e-14) and q[0, 2] == pytest.approx(q[1, 2], abs=1e-14)
    assert q[0, 1] - 2.0 == pytest.approx(2.0 - q[1, 1], abs=1e-14)
    assert q[0, 3] == pytest.approx(-q[1, 3], abs=1e-14)
    assert q[0, 4] == pytest.approx(-q[1, 4], abs=1e-12)
    # they repel each other: less closing speed than without the other
    alone, _, _ = cref.crowd_step(p[:1], [True], goals[:1], vdes[:1], *FAR_ROBOT, od, 0.05, 1)
    assert q[0, 3] < alone[0, 3]


def test_person_next_to_the_robot_is_pushed_away_and_the_disturbance_is_the_robot_force():
    od = _open_od()
    p = np.array([[3.0, 2.4, 0.0, 0.0, 0.0]])  # standing 0.4 m left of the robot's track
    robot_pose, robot_cmd = [2.6, 2.0, 0.0], [0.5, 0.0]
    q, _, dist = cref.crowd_step(p, [False], [[3.0, 2.4]], [1.0], robot_pose, robot_cmd, od, 0.05, 1)
    assert q[0, 1] > 2.4 and q[0, 3] > 0.0  # away from the robot's side
    # one substep: the disturbance is |F(robot -> person)| dt_s, and with no goal, obstacle or other person the force
    # on the person is that pair force plus braking (zero at rest): velocity = F dt_s
    f = np.array([q[0, 2], q[0, 3]]) / 0.05
    assert dist == pytest.approx(np.linalg.norm(f) * 0.05, rel=1e-12)
    assert dist > 0.0


def test_obstacle_cell_outside_the_grid_is_none():
    od = _open_od(w=10, h=10)
    od["indexes"] = np.zeros(100, dtype=np.uint32)  # nearest obstacle: cell (0, 0)
    assert cref.obstacle_cell([-0.01, 0.2], od) is None and cref.obstacle_cell([0.2, 0.6], od) is None
    c = cref.obstacle_cell([0.2, 0.3], od)
    assert c == pytest.approx([0.0, 0.0], abs=1e-15)


@pytest.mark.parametrize("B,K,seed", [(64, 20, 6), (16, 9, 1), (8, 0, 2)])
def test_crowd_scenes_keep_spacing_margins_and_speeds(B, K, seed):
    s = sc.crowd_episodes(B, K, seed=seed, ticks=200)
    p = s["params"]
    assert s["people"].shape == (B, K, 5) and s["goals"].shape == (B, K, 2) and s["desired_speed"].shape == (B, K)
    assert np.all(s["n_people"] == K) and s["substeps"] == 1 and s["ticks"] == 200
    if K == 0:
        return
    start, goal, vdes = s["people"][..., :2], s["goals"], s["desired_speed"]
    assert np.all((vdes >= 0.3) & (vdes <= 1.2))
    v = s["people"][..., 2:4]
    assert np.allclose(np.linalg.norm(v, axis=-1), vdes, rtol=1e-12)
    dg = goal - start
    assert np.allclose(v / vdes[..., None], dg / np.linalg.norm(dg, axis=-1, keepdims=True), atol=1e-12)
    # starts: from the robot, from each other, from lethal cells
    pose = s["pose"]
    assert np.hypot(start[..., 0] - pose[:, None, 0], start[..., 1] - pose[:, None, 1]).min() >= sc.CROWD_CLEARANCE
    d = np.hypot(start[:, :, None, 0] - start[:, None, :, 0], start[:, :, None, 1] - start[:, None, :, 1])
    d[:, np.arange(K), np.arange(K)] = np.inf
    assert d.min() >= sc.CROWD_SPACING
    res = s["costmap_resolution"]
    for b in range(B):
        cm = s["costmaps"][s["costmap_index"][b]]
        ly, lx = np.nonzero(cm >= 253)
        cx, cy = (lx + 0.5) * res, (ly + 0.5) * res
        for i in range(K):
            assert np.hypot(cx - start[b, i, 0], cy - start[b, i, 1]).min() >= sc.CROWD_CLEARANCE
    # goals: away from the grid's ends by the margin the controller's projection needs, inside the corridor
    od = s["od"]
    margin = sc.EPISODE_MARGIN + 0.5 * sc.f32(p.max_time)
    assert goal[..., 0].min() >= margin - 1e-12 and goal[..., 0].max() <= od["width"] * od["resolution"] - margin + 1e-12
    assert goal[..., 1].min() >= 1.0 - 1e-12 and goal[..., 1].max() <= 3.0 + 1e-12
    # the three kinds of walker
    kind = np.arange(K) % 3
    assert np.all(goal[:, kind == 0, 0] < start[:, kind == 0, 0])  # oncoming: toward the robot's start end
    assert np.all(goal[:, kind == 1, 0] > start[:, kind == 1, 0])  # same direction: to the far end
    assert np.all(np.sign(goal[:, kind == 2, 1] - 2.0) == -np.sign(start[:, kind == 2, 1] - 2.0))  # across
