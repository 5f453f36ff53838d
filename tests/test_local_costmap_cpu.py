"""CPU tests of the rolling local costmap of smpc_run_local_costmap_episodes: its parameter block mirrors include/smpc.h,
the library's stencil (smpc_local_costmap_stencil) is the numpy one of tests/local_costmap_ref.py and has Nav2's
inflation properties, the window is placed around the robot's cell at odd and even sizes, and the numpy splat is the
inflation of the union of the people's lethal discs."""
import os
import re

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, fleet
from tests import local_costmap_ref as lref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RES = 0.05
# (overrides, resolution): the defaults, an inscribed band, whole-cell radii, a steep and a flat decay, a point agent,
# another resolution and the largest stencil that fits
STENCILS = [
    ({}, RES),
    (dict(inscribed_radius=0.1), RES),
    (dict(agent_radius=0.2, inscribed_radius=0.05, inflation_radius=0.4), RES),
    (dict(cost_scaling_factor=10.0, inflation_radius=1.0), RES),
    (dict(cost_scaling_factor=0.5), RES),
    (dict(agent_radius=0.0, inflation_radius=0.3), RES),
    (dict(agent_radius=0.3, inscribed_radius=0.3, inflation_radius=0.8), 0.1),
    (dict(agent_radius=0.5, inflation_radius=1.1), RES),
]


def _lib_stencil(over, res):
    return fleet.local_costmap_stencil(res, over)


def test_local_costmap_struct_defaults_and_entries_match_header():
    hdr = open(os.path.join(ROOT, "include", "smpc.h")).read()
    body = re.search(r"typedef struct smpc_local_costmap \{(.*?)\} smpc_local_costmap;", hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [n.strip().lstrip("*") for d in body.split(";") if d.strip()
              for n in re.sub(r"^\s*\w+\*?\s+", "", d.strip()).split(",")]
    assert fields == [f[0] for f in abi.SmpcLocalCostmap._fields_]
    assert re.search(r"int smpc_run_local_costmap_episodes\(smpc_handle\* h, smpc_episode_io\* io,", hdr)
    assert re.search(r"int smpc_local_costmap_stencil\(const smpc_local_costmap\* local, double resolution,", hdr)
    for sym in ("smpc_run_local_costmap_episodes", "smpc_local_costmap_stencil"):
        assert sym in _lib.EXPORTED_SYMBOLS
    lc = abi.local_costmap_params()
    assert {f: getattr(lc, f) for f in lref.DEFAULTS} == lref.DEFAULTS == abi.LOCAL_COSTMAP_DEFAULTS
    assert not (lc.marked_rows or lc.costmap_log or lc.origin_log)
    assert abi.local_costmap_params(size_x=41).size_x == 41
    with pytest.raises(ValueError, match="size"):
        abi.local_costmap_params(size=41)


@pytest.mark.parametrize("over,res", STENCILS)
def test_library_stencil_is_the_numpy_stencil(over, res):
    prm = dict(lref.DEFAULTS, **over)
    want, hw, raw = lref.stencil(prm, res)
    got = _lib_stencil(over, res)
    assert got.shape == want.shape and hw <= lref.MAX_HALF
    diff = got != want
    # a cell may differ only where the unrounded 252 exp(...) lies within 1e-9 of an integer (libm vs numpy exp)
    near = np.abs(raw - np.round(raw)) <= 1e-9
    assert not (diff & ~near).any(), np.argwhere(diff & ~near)
    assert not diff.any(), "a near-integer cost rounded differently"  # none did on these parameters


def test_stencil_has_nav2_inflation_properties():
    for over, res in STENCILS:
        prm = dict(lref.DEFAULTS, **over)
        s = _lib_stencil(over, res).astype(int)
        hw = s.shape[0] // 2
        assert s[hw, hw] == 254
        for t in (s, s.T, s[::-1], s[:, ::-1]):  # 8-fold symmetry
            assert np.array_equal(t, s)
        assert (s[0] > 0).any() or (s[:, 0] > 0).any()  # the half-width is the smallest that holds the support
        dy, dx = np.mgrid[-hw:hw + 1, -hw:hw + 1]
        d_centre = np.hypot(dx, dy) * res
        rho = prm["agent_radius"]
        beyond = d_centre > rho + prm["inflation_radius"] + res  # farther than the disc plus the inflation radius
        assert not s[beyond].any()
        assert (s == 253).any() == (prm["inscribed_radius"] > 0)  # every inscribed radius here reaches a cell
        # non-increasing along the rays from the centre (axes and diagonals)
        for ray in (s[hw, hw:], s[hw:, hw], np.diag(s)[hw:], np.diag(s[::-1])[hw:]):
            assert np.all(np.diff(ray) <= 0)


def test_whole_cell_radii_are_inclusive():
    # agent radius of exactly 2 cells: (2, 0) is lethal, (2, 1) is not
    s = _lib_stencil(dict(agent_radius=0.1, inflation_radius=0.1, cost_scaling_factor=1.0), RES)
    hw = s.shape[0] // 2
    assert s[hw, hw + 2] == 254 and s[hw + 1, hw + 2] < 254
    # inflation radius of exactly 2 cells: (4, 0) is 2 cells from the disc and inflated, (5, 0) is not
    assert s[hw, hw + 4] > 0 and hw == 4
    # inscribed radius of exactly 1 cell: the first ring outside the disc is 253
    s = _lib_stencil(dict(agent_radius=0.1, inscribed_radius=0.05, inflation_radius=0.2), RES)
    hw = s.shape[0] // 2
    assert s[hw, hw + 3] == 253 and s[hw, hw + 4] < 253


def test_out_of_range_stencils_are_rejected():
    for over in (dict(inflation_radius=1.6), dict(agent_radius=1.7), dict(size_x=7), dict(size_y=257),
                 dict(update_period_ticks=0), dict(update_period_ticks=21), dict(mark_people=2),
                 dict(agent_radius=np.nan), dict(inscribed_radius=-0.1), dict(cost_scaling_factor=0.0),
                 dict(cost_scaling_factor=np.inf), dict(inflation_radius=np.nan),
                 dict(inscribed_radius=0.3, inflation_radius=0.2)):
        with pytest.raises(_lib.SmpcError):
            _lib_stencil(over, RES)
        prm = dict(lref.DEFAULTS, **over)
        if "inflation_radius" in over and np.isfinite(over["inflation_radius"]) and "inscribed_radius" not in over:
            assert lref.stencil(prm, RES)[1] > lref.MAX_HALF
    with pytest.raises(_lib.SmpcError):
        _lib_stencil({}, 0.0)
    assert _lib_stencil(dict(inflation_radius=1.35), RES).shape[0] <= 2 * lref.MAX_HALF + 1


@pytest.mark.parametrize("sx,sy", [(80, 80), (81, 79), (8, 9), (256, 255)])
def test_placement_centres_the_robot_cell(sx, sy):
    rng = np.random.default_rng(sx * 1000 + sy)
    origin = np.array([-1.3, 0.45])
    for _ in range(200):
        x, y = rng.uniform(-5.0, 15.0), rng.uniform(-5.0, 10.0)
        c0x, c0y, org = lref.placement(x, y, origin, RES, sx, sy)
        cx, cy = lref.static_cell(x, y, origin, RES)
        assert cx - c0x == sx // 2 and cy - c0y == sy // 2  # the centre cell; odd: the middle, even: right of middle
        assert org[0] == origin[0] + c0x * RES and org[1] == origin[1] + c0y * RES
        assert abs((x - org[0]) / RES - (sx // 2 + 0.5)) <= 0.5 + 1e-9  # the robot lies in that cell of the window
    # a window hanging over the map's corner keeps the map's bytes where they exist and zeros elsewhere
    static = rng.integers(1, 255, (30, 40), dtype=np.uint8)
    win = lref.crop(static, -3, 25, sx, sy)
    assert np.array_equal(win[:5, 3:3 + min(40, sx - 3)], static[25:, :min(40, sx - 3)])
    assert not win[:, :3].any() and not win[5:].any()


def test_numpy_splat_is_the_inflation_of_the_union_of_discs():
    rng = np.random.default_rng(5)
    for trial in range(12):
        over = STENCILS[trial % len(STENCILS)][0]
        prm = dict(lref.DEFAULTS, **over)
        sten, hw, _ = lref.stencil(prm, RES)
        sx, sy = int(rng.integers(20, 50)), int(rng.integers(20, 50))
        cells = [(int(rng.integers(0, sx)), int(rng.integers(0, sy))) for _ in range(int(rng.integers(1, 6)))]
        got = lref.splat(np.zeros((sy, sx), np.uint8), cells, sten, hw)
        assert np.array_equal(got, lref.inflate_brute(sx, sy, cells, prm, RES)), (trial, cells)


def test_build_marks_only_rows_inside_the_window():
    prm = dict(lref.DEFAULTS, size_x=20, size_y=20)
    sten, hw, _ = lref.stencil(prm, RES)
    static = np.zeros((80, 240), np.uint8)
    static[:6] = 254
    pose = np.array([2.0, 2.0, 0.0])
    rows = np.array([[2.3, 2.0], [2.0 + 0.51, 2.0], [2.0 + 0.45, 2.0], [np.nan, 2.0], [-3.0, 2.0]])
    win, org, n = lref.build(static, np.zeros(2), RES, pose, rows, len(rows), prm, sten, hw)
    assert n == 2  # 0.51 m ahead is in the next window's cell column 20, outside; NaN and far rows are not marked
    assert org[0] == 0.0 + 30 * RES and org[1] == 0.0 + 30 * RES
    off, _, _ = lref.build(static, np.zeros(2), RES, pose, rows, len(rows), dict(prm, mark_people=0), sten, hw)
    assert np.array_equal(off, lref.crop(static, 30, 30, 20, 20)) and (win >= off).all() and (win > off).any()
