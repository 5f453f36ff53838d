"""numpy restatement of the rolling local costmap of smpc_run_local_costmap_episodes (include/smpc.h): the window's
placement at whole static cells, the inflation stencil (Nav2's InflationLayer::computeCost on a disc of lethal cells)
and the splat of the people's cells. The GPU tests compare every logged window with it byte for byte."""
import math

import numpy as np

DEFAULTS = dict(size_x=80, size_y=80, update_period_ticks=4, mark_people=1, agent_radius=0.25, inscribed_radius=0.0,
                cost_scaling_factor=3.0, inflation_radius=0.55)
MAX_HALF = 32


def stencil(prm, res):
    """(stencil uint8 [2 hw + 1][2 hw + 1] with row dy + hw and column dx + hw, hw, raw) for the parameters prm at
    resolution res; raw is the unrounded 252 exp(...) of the same cells (NaN where the cost is not that branch).
    Computed on a grid of half-width MAX_HALF + 1: hw > MAX_HALF means the entry rejects prm."""
    H = MAX_HALF + 1
    r = np.arange(-H, H + 1)
    dy, dx = np.meshgrid(r, r, indexing="ij")
    rho = prm["agent_radius"] / res + 1e-9
    lethal = (dx * dx + dy * dy).astype(np.float64) <= rho * rho
    lx, ly = dx[lethal], dy[lethal]
    d2 = np.min((dx[..., None] - lx) ** 2 + (dy[..., None] - ly) ** 2, axis=-1)
    d = np.sqrt(d2.astype(np.float64))
    ins, csf = prm["inscribed_radius"], prm["cost_scaling_factor"]
    raw = 252.0 * np.exp(-csf * (d * res - ins))
    band = d * res <= ins + 1e-9
    inflated = ~band & (d <= prm["inflation_radius"] / res + 1e-9)
    cost = np.where(band, 253, np.where(inflated, np.floor(raw), 0)).astype(np.int64)
    cost[lethal] = 254
    raw = np.where(inflated & ~lethal, raw, np.nan)
    nz = cost > 0
    hw = int(np.max(np.maximum(np.abs(dx), np.abs(dy))[nz]))
    sl = slice(H - hw, H + hw + 1)
    return cost[sl, sl].astype(np.uint8), hw, raw[sl, sl]


def static_cell(x, y, origin, res):
    """The floor rule of the placement and the people layer: (cx, cy) as floats (NaN stays NaN)."""
    return np.floor((x - origin[0]) / res), np.floor((y - origin[1]) / res)


def placement(x, y, origin, res, sx, sy):
    """(c0x, c0y, window origin) of a robot at (x, y) on a static map with this origin: its static cell is the window's
    centre cell (C integer division of the size), and the origin is one multiply then add per axis."""
    cx, cy = static_cell(x, y, origin, res)
    c0x, c0y = int(cx) - sx // 2, int(cy) - sy // 2
    return c0x, c0y, np.array([origin[0] + c0x * res, origin[1] + c0y * res])


def crop(static, c0x, c0y, sx, sy):
    """[sy][sx] window of the static map starting at static cell (c0x, c0y), 0 outside the map."""
    H, W = static.shape
    out = np.zeros((sy, sx), np.uint8)
    x0, x1 = max(c0x, 0), min(c0x + sx, W)
    y0, y1 = max(c0y, 0), min(c0y + sy, H)
    if x0 < x1 and y0 < y1:
        out[y0 - c0y:y1 - c0y, x0 - c0x:x1 - c0x] = static[y0:y1, x0:x1]
    return out


def splat(window, cells, sten, hw):
    """Max the stencil into window (in place) centred on every (wx, wy) window cell of `cells`."""
    sy, sx = window.shape
    for wx, wy in cells:
        x0, x1 = max(wx - hw, 0), min(wx + hw + 1, sx)
        y0, y1 = max(wy - hw, 0), min(wy + hw + 1, sy)
        if x0 < x1 and y0 < y1:
            np.maximum(window[y0:y1, x0:x1], sten[y0 - wy + hw:y1 - wy + hw, x0 - wx + hw:x1 - wx + hw],
                       out=window[y0:y1, x0:x1])
    return window


def marked_cells(rows, n, origin, res, c0x, c0y, sx, sy):
    """The window cells of the first n rows [.][>= 2] whose static cell lies inside the window."""
    out = []
    for j in range(n):
        cx, cy = static_cell(rows[j, 0], rows[j, 1], origin, res)
        fx, fy = cx - c0x, cy - c0y
        if 0.0 <= fx < sx and 0.0 <= fy < sy:
            out.append((int(fx), int(fy)))
    return out


def build(static, origin, res, pose, rows, n, prm, sten, hw):
    """One build of a robot's window: (window uint8 [sy][sx], window origin [2], rows marked)."""
    sx, sy = prm["size_x"], prm["size_y"]
    c0x, c0y, org = placement(pose[0], pose[1], origin, res, sx, sy)
    win = crop(static, c0x, c0y, sx, sy)
    cells = marked_cells(rows, n, origin, res, c0x, c0y, sx, sy) if prm["mark_people"] else []
    return splat(win, cells, sten, hw), org, len(cells)


def inflate_brute(sx, sy, cells, prm, res):
    """Nav2's inflation of a window with no static cost and the lethal discs of `cells` (window cells, possibly near its
    edge), by the distance of every cell to the nearest lethal cell of the union, lethal cells outside the window
    included: [sy][sx] uint8."""
    rho = prm["agent_radius"] / res + 1e-9
    R = int(math.floor(rho))
    lethal = set()
    for wx, wy in cells:
        for dy in range(-R, R + 1):
            for dx in range(-R, R + 1):
                if dx * dx + dy * dy <= rho * rho:
                    lethal.add((wx + dx, wy + dy))
    out = np.zeros((sy, sx), np.uint8)
    if not lethal:
        return out
    L = np.array(sorted(lethal), dtype=np.float64)
    ys, xs = np.mgrid[0:sy, 0:sx]
    d = np.sqrt(np.min((xs[..., None] - L[:, 0]) ** 2 + (ys[..., None] - L[:, 1]) ** 2, axis=-1))
    ins, csf = prm["inscribed_radius"], prm["cost_scaling_factor"]
    cost = np.where(d * res <= ins + 1e-9, 253,
                    np.where(d <= prm["inflation_radius"] / res + 1e-9,
                             np.floor(252.0 * np.exp(-csf * (d * res - ins))), 0))
    cost = np.where(d == 0.0, 254, cost)
    return cost.astype(np.uint8)
