"""numpy restatement of the perception stage of smpc_run_perceived_episodes (include/smpc.h, csrc/smpc_perception.cu),
operation for operation: Philox4x32-10, the 53-bit uniform, Box-Muller, the Amanatides-Woo walk over the costmap, the
occlusion test and the order-preserving compaction. The visibility decision uses only IEEE-rounded + - * / sqrt (the
kernel is compiled without FMA contraction), so it is reproduced exactly; the noise goes through log / cos / sin and
may differ from the device in the last bits."""
from __future__ import annotations

import math

import numpy as np

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF
PERSONAL = 1.2
DEFAULTS = dict(max_range=8.0, occluder_radius=0.25, occluding_cost=254, detect_prob=0.95, pos_noise=0.05,
                vel_noise=0.1, seed=0)
NEUTRAL = dict(max_range=math.inf, occluder_radius=0.0, occluding_cost=0, detect_prob=1.0, pos_noise=0.0,
               vel_noise=0.0, seed=0)


def philox(counter, key):
    """Philox4x32-10 of a 4-word counter under a 2-word key (Random123's philox4x32, 10 rounds): 4 words."""
    c = [int(x) & MASK for x in counter]
    k = [int(x) & MASK for x in key]
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & MASK, p1 & MASK, ((p0 >> 32) ^ c[3] ^ k[1]) & MASK, p0 & MASK]
        k = [(k[0] + W0) & MASK, (k[1] + W1) & MASK]
    return c


def uniform(a, b):
    """Two words -> a uniform in (0, 1]: ((a << 21) + (b >> 11) + 1) 2^-53."""
    return float((int(a) << 21) + (int(b) >> 11) + 1) * 2.0 ** -53


def normals(words):
    """Two standard normals from one Philox block by Box-Muller."""
    r = math.sqrt(-2.0 * math.log(uniform(words[0], words[1])))
    ang = 2.0 * math.pi * uniform(words[2], words[3])
    return r * math.cos(ang), r * math.sin(ang)


def key_of(seed):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return seed & MASK, seed >> 32


def draw(seed, k, stream, agent, d):
    """The Philox block of draw d (0: position pair, 1: velocity pair, 2: detection) of an agent at tick k."""
    return philox((k, stream, agent, d), key_of(seed))


def walk(g0, g1):
    """The cells strictly between the cell of g0 and the cell of g1 (grid units) that the kernel's Amanatides-Woo walk
    visits, in order: x steps when tmx <= tmy, never past the end index on an axis."""
    cx, cy = math.floor(g0[0]), math.floor(g0[1])
    ex, ey = math.floor(g1[0]), math.floor(g1[1])
    nx, ny = abs(ex - cx), abs(ey - cy)
    sx = 1 if ex > cx else -1
    sy = 1 if ey > cy else -1
    ax, ay = abs(g1[0] - g0[0]), abs(g1[1] - g0[1])
    tmx = tmy = tdx = tdy = math.inf
    if nx > 0:
        tmx = ((cx + 1) - g0[0] if sx > 0 else g0[0] - cx) / ax
        tdx = 1.0 / ax
    if ny > 0:
        tmy = ((cy + 1) - g0[1] if sy > 0 else g0[1] - cy) / ay
        tdy = 1.0 / ay
    cells = []
    for _ in range(nx + ny - 1):
        if ny == 0 or (nx > 0 and tmx <= tmy):
            cx += sx
            tmx += tdx
            nx -= 1
        else:
            cy += sy
            tmy += tdy
            ny -= 1
        cells.append((cx, cy))
    return cells


def wall_between(costmap, origin, res, a, b, occluding_cost):
    """True when a cell of costmap [H][W] strictly between the cells of world points a and b has cost >= occluding_cost
    (cells outside the map do not block)."""
    H, W = costmap.shape
    g0 = ((a[0] - origin[0]) / res, (a[1] - origin[1]) / res)
    g1 = ((b[0] - origin[0]) / res, (b[1] - origin[1]) / res)
    for cx, cy in walk(g0, g1):
        if 0 <= cx < W and 0 <= cy < H and costmap[cy, cx] >= occluding_cost:
            return True
    return False


def occluded(offsets, j, radius):
    """True when a row i != j of offsets [n][2] (p_i - robot) strictly closer than row j lies within `radius` of the
    segment robot -> p_j, strictly inside it (0 < t < 1)."""
    ex, ey = float(offsets[j][0]), float(offsets[j][1])
    d2 = ex * ex + ey * ey
    r2 = radius * radius
    for i in range(len(offsets)):
        fx, fy = float(offsets[i][0]), float(offsets[i][1])
        if not fx * fx + fy * fy < d2:
            continue
        t = (fx * ex + fy * ey) / d2
        if not (0.0 < t < 1.0):
            continue
        gx, gy = fx - t * ex, fy - t * ey
        if gx * gx + gy * gy < r2:
            return True
    return False


def agent_ids(n, R, K, me):
    """Agent id of each of the n rows of robot `me`'s list: the other robots of the scene (K + their index) first when
    R > 1, then the people's scene slots."""
    others = [r for r in range(R) if r != me][: R - 1] if R > 1 else []
    return [K + others[j] if j < R - 1 else j - (R - 1) for j in range(n)]


def perceive(rows, pose, k, stream, prm, costmap=None, origin=None, res=None, R=1, K=None, me=0):
    """The stage for one robot at tick k: rows [n][5] (its list, true state), pose (x, y, ...). Returns (seen [m][5],
    visible [n] bool, missed) with missed = a person (not a robot) within 1.2 m went unreported."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 5)
    n = rows.shape[0]
    K = n - (R - 1) if K is None else K
    rx, ry = float(pose[0]), float(pose[1])
    offs = [(float(rows[j, 0]) - rx, float(rows[j, 1]) - ry) for j in range(n)]
    ids = agent_ids(n, R, K, me)
    vis = np.zeros(n, bool)
    missed = False
    for j in range(n):
        dx, dy = offs[j]
        dist = math.sqrt(dx * dx + dy * dy)
        v = dist <= prm["max_range"]
        if v and prm["detect_prob"] < 1.0:
            w = draw(prm["seed"], k, stream, ids[j], 2)
            v = uniform(w[0], w[1]) <= prm["detect_prob"]
        if v and prm["occluder_radius"] > 0.0:
            v = not occluded(offs, j, prm["occluder_radius"])
        if v and prm["occluding_cost"] > 0:
            v = not wall_between(costmap, origin, res, (rx, ry), (float(rows[j, 0]), float(rows[j, 1])),
                                 prm["occluding_cost"])
        vis[j] = v
        if not v and j >= R - 1 and dist < PERSONAL:
            missed = True
    seen = []
    for j in np.flatnonzero(vis):
        row = rows[j].copy()
        if prm["pos_noise"] > 0.0:
            n0, n1 = normals(draw(prm["seed"], k, stream, ids[j], 0))
            row[0] = row[0] + prm["pos_noise"] * n0
            row[1] = row[1] + prm["pos_noise"] * n1
        if prm["vel_noise"] > 0.0:
            n0, n1 = normals(draw(prm["seed"], k, stream, ids[j], 1))
            row[2] = row[2] + prm["vel_noise"] * n0
            row[3] = row[3] + prm["vel_noise"] * n1
        seen.append(row)
    return np.array(seen).reshape(-1, 5), vis, missed


def perceive_all(lists, n_list, poses, active, k, prm, costmaps, origins, res, costmap_index=None, R=1, K=None,
                 stream_index=None):
    """The stage for every robot at tick k: lists [B][L][5], n_list [B], poses [B][3], active [B]. Returns
    (seen [B][L][5] with zero rows after n, n_seen [B], missed [B]); inactive robots report nothing."""
    B, L = lists.shape[0], lists.shape[1]
    K = L - (R - 1) if K is None else K
    seen = np.zeros((B, L, 5))
    n_seen = np.zeros(B, np.int32)
    missed = np.zeros(B, bool)
    for b in range(B):
        if not active[b]:
            continue
        mi = int(costmap_index[b]) if costmap_index is not None else b % costmaps.shape[0]
        stream = int(stream_index[b]) if stream_index is not None else b
        rows, _, miss = perceive(lists[b, : int(n_list[b])], poses[b], k, stream, prm, costmaps[mi], origins[mi], res,
                                 R=R, K=K, me=b % R)
        seen[b, : rows.shape[0]] = rows
        n_seen[b] = rows.shape[0]
        missed[b] = miss
    return seen, n_seen, missed
