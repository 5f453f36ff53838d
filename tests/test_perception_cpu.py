"""CPU tests of the perception stage of smpc_run_perceived_episodes: its parameter block mirrors include/smpc.h, and the
numpy restatement the GPU tests compare with (tests/perception_ref.py) draws Random123's Philox numbers, walks the
costmap through every cell the line of sight crosses and occludes as the header says."""
import math
import os
import re

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi
from tests import perception_ref as pref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_perception_struct_field_order_defaults_and_entry_match_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_perception \{(.*?)\} smpc_perception;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [d.strip().split()[-1].lstrip("*") for d in body.split(";") if d.strip()]
    assert fields == [f[0] for f in abi.SmpcPerception._fields_]
    assert re.search(r"int smpc_run_perceived_episodes\(smpc_handle\* h, smpc_episode_io\* io,", hdr)
    assert "smpc_run_perceived_episodes" in _lib.EXPORTED_SYMBOLS
    p = abi.perception_params()
    assert {f: getattr(p, f) for f in pref.DEFAULTS} == pref.DEFAULTS
    assert not p.stream_index and not p.unseen_personal_ticks and not p.seen_log and not p.n_seen_log
    assert abi.perception_params(detect_prob=0.5).detect_prob == 0.5
    assert {f: getattr(abi.perception_params(**abi.PERCEPTION_NEUTRAL), f) for f in pref.NEUTRAL} == pref.NEUTRAL
    with pytest.raises(TypeError):
        abi.perception_params(range=3.0)


def test_philox_matches_the_random123_known_answers():
    hexed = lambda c, k: ["%08x" % w for w in pref.philox(c, k)]  # noqa: E731
    assert hexed([0, 0, 0, 0], [0, 0]) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    assert hexed([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert hexed([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]
    assert pref.key_of(0x0123456789ABCDEF) == (0x89ABCDEF, 0x01234567)


def test_uniform_end_points():
    assert pref.uniform(0, 0) == 2.0 ** -53
    assert pref.uniform(0xFFFFFFFF, 0xFFFFFFFF) == 1.0
    assert pref.uniform(0, 0x7FF) == 2.0 ** -53  # the low 11 bits of the second word are dropped
    assert pref.uniform(0, 0x800) == 2.0 ** -52


def test_box_muller_moments():
    n = 20000
    z = np.array([pref.normals(pref.draw(7, k, 3, 5, 0)) for k in range(n // 2)]).ravel()
    se = 1.0 / math.sqrt(n)
    assert abs(z.mean()) < 5 * se
    assert abs(z.var() - 1.0) < 5 * math.sqrt(2.0) * se
    assert abs(np.mean(z ** 4) - 3.0) < 5 * math.sqrt(96.0) * se
    assert abs(np.corrcoef(z[0::2], z[1::2])[0, 1]) < 5 * math.sqrt(2.0) * se
    u = np.array([pref.uniform(*pref.draw(7, k, 3, 5, 2)[:2]) for k in range(n)])
    assert abs(u.mean() - 0.5) < 5 * math.sqrt(1.0 / 12.0) * se
    # the detection, position and velocity draws of one agent and tick are distinct blocks
    assert len({tuple(pref.draw(7, 0, 3, 5, d)) for d in range(3)}) == 3


def _sampled_cells(g0, g1, n=20001):
    t = np.linspace(0.0, 1.0, n)[1:-1]
    x = g0[0] + t * (g1[0] - g0[0])
    y = g0[1] + t * (g1[1] - g0[1])
    return set(zip(np.floor(x).astype(int).tolist(), np.floor(y).astype(int).tolist()))


@pytest.mark.parametrize("octant", range(8))
def test_walk_visits_every_cell_the_segment_crosses(octant):
    rng = np.random.default_rng(octant)
    for _ in range(40):
        g0 = rng.uniform(20.0, 30.0, 2)
        ang = (octant + rng.uniform(0.02, 0.98)) * math.pi / 4.0
        g1 = g0 + rng.uniform(0.5, 15.0) * np.array([math.cos(ang), math.sin(ang)])
        _check_walk(tuple(g0), tuple(g1))
    for d in ((7.0, 0.0), (-7.0, 0.0), (0.0, 7.0), (0.0, -7.0)):  # axis-aligned rays
        g0 = (20.3, 40.6)
        _check_walk(g0, (g0[0] + d[0], g0[1] + d[1]))


def _check_walk(g0, g1):
    cells = pref.walk(g0, g1)
    c0 = (math.floor(g0[0]), math.floor(g0[1]))
    c1 = (math.floor(g1[0]), math.floor(g1[1]))
    assert len(cells) == max(abs(c1[0] - c0[0]) + abs(c1[1] - c0[1]) - 1, 0)
    assert c0 not in cells and c1 not in cells
    path = [c0] + cells + [c1] if c0 != c1 else [c0]
    for a, b in zip(path, path[1:]):  # 4-connected, one axis per step
        assert abs(a[0] - b[0]) + abs(a[1] - b[1]) == 1
    assert _sampled_cells(g0, g1) - {c0, c1} <= set(cells)


def test_wall_across_a_ray_blocks_it():
    res, origin = 0.05, (-1.0, 2.0)
    cm = np.zeros((100, 120), np.uint8)
    cm[:, 60] = 254  # a wall across the map at x = origin + 3.0 m
    world = lambda gx, gy: (origin[0] + gx * res, origin[1] + gy * res)  # noqa: E731
    a, b = world(20.5, 30.5), world(90.2, 41.7)
    assert pref.wall_between(cm, origin, res, a, b, 254)
    assert pref.wall_between(cm, origin, res, b, a, 254)
    assert not pref.wall_between(cm, origin, res, a, b, 255)  # cost below the threshold
    assert not pref.wall_between(cm, origin, res, a, world(55.0, 31.0), 254)  # stops short of the wall
    assert not pref.wall_between(cm, origin, res, a, world(60.5, 31.0), 254)  # the row's own cell does not block
    assert not pref.wall_between(cm, origin, res, world(60.5, 31.5), world(90.2, 31.7), 254)  # nor the robot's
    # cells outside the map do not block: a ray around the map's edge
    assert not pref.wall_between(cm, origin, res, world(20.5, -5.5), world(90.5, -5.5), 1)


def test_occlusion_geometry():
    r = 0.25
    target = (4.0, 0.0)
    assert pref.occluded([target, (2.0, 0.1)], 0, r)  # on the line
    assert not pref.occluded([target, (2.0, 0.3)], 0, r)  # beside it, beyond the radius
    assert not pref.occluded([target, (5.0, 0.0)], 0, r)  # behind the target
    assert not pref.occluded([target, (-1.0, 0.0)], 0, r)  # behind the robot (t < 0)
    assert not pref.occluded([target, target], 0, r) and not pref.occluded([target, target], 1, r)  # equal distances
    assert not pref.occluded([target, (2.0, 0.0)], 0, 0.0)  # radius 0: nobody occludes
    # through the stage: two people in line, the farther one is hidden; a robot row does not count as a missed person
    prm = dict(pref.NEUTRAL, occluder_radius=r)
    rows = np.array([[1.0, 0.0, 0, 0, 0], [0.5, 0.0, 0, 0, 0], [0.0, 3.0, 0, 0, 0]])
    seen, vis, missed = pref.perceive(rows, (0.0, 0.0, 0.0), 0, 0, prm)
    assert vis.tolist() == [False, True, True] and missed
    seen, vis, missed = pref.perceive(rows, (0.0, 0.0, 0.0), 0, 0, prm, R=2, K=2)
    assert vis.tolist() == [False, True, True] and not missed  # row 0 is the other robot


def test_neutral_parameters_return_the_list_unchanged_and_in_order():
    rng = np.random.default_rng(3)
    rows = rng.normal(size=(40, 5)) * 4.0
    rows[5, :2] = rows[9, :2]  # coincident people
    rows[7, 2] = -0.0
    seen, vis, missed = pref.perceive(rows, (0.3, -0.2, 1.0), 12, 4, pref.NEUTRAL, np.zeros((4, 4), np.uint8),
                                      (0.0, 0.0), 0.05)
    assert vis.all() and not missed
    assert seen.tobytes() == rows.tobytes()


def test_range_and_detection():
    rows = np.array([[3.0, 4.0, 0, 0, 0], [0.0, 5.000001, 0, 0, 0], [1.0, 0.0, 0, 0, 0]])
    seen, vis, missed = pref.perceive(rows, (0.0, 0.0, 0.0), 0, 0, dict(pref.NEUTRAL, max_range=5.0))
    assert vis.tolist() == [True, False, True] and not missed
    seen, vis, missed = pref.perceive(rows, (0.0, 0.0, 0.0), 0, 0, dict(pref.NEUTRAL, detect_prob=0.0))
    assert seen.shape == (0, 5) and missed
    # a draw decides detection: the same seed, tick, stream and agent always decide alike
    p = dict(pref.NEUTRAL, detect_prob=0.5, seed=11)
    a = [pref.perceive(rows, (0.0, 0.0, 0.0), k, 2, p)[1] for k in range(64)]
    b = [pref.perceive(rows, (0.0, 0.0, 0.0), k, 2, p)[1] for k in range(64)]
    assert np.array_equal(a, b) and 0.3 < np.mean(a) < 0.7
