"""numpy restatement of the people tracker of smpc_run_tracked_episodes (include/smpc.h, csrc/smpc_tracker.cu) on top of
the detections of tests/perception_ref.py: one constant-velocity Kalman track per agent id with the kernel's
operation order (its header comment), confirmation, coasting, death, and the latency ring. Every product and sum is an
IEEE-rounded double operation in the kernel's order, so the filter matches the device bit for bit wherever the
measurements do; the position noise goes through log / cos / sin and may differ from the device in the last bits."""
from __future__ import annotations

import math

import numpy as np

from tests import perception_ref as pref

DEFAULTS = dict(accel_noise=0.5, meas_noise=0.05, init_vel_std=1.0, confirm_hits=3, max_coast_ticks=10,
                latency_ticks=2)
PASS_THROUGH = dict(confirm_hits=1, max_coast_ticks=0, latency_ticks=0)
MAX_HITS = 16
PERSONAL = pref.PERSONAL


def noise_terms(accel_noise, dt):
    """(q_pp, q_pv, q_vv) of the white-acceleration model over dt, in the kernel's order."""
    a2 = accel_noise * accel_noise
    dt2 = dt * dt
    return a2 * dt2 * dt2 / 4.0, a2 * dt2 * dt / 2.0, a2 * dt2


class Track:
    """One id's track: position, velocity, the per-axis covariance (pp, pv, vv) both axes share, hits (0: no track)
    and misses."""

    def __init__(self):
        self.p = [0.0, 0.0]
        self.v = [0.0, 0.0]
        self.pp = self.pv = self.vv = 0.0
        self.hits = self.misses = 0

    def predict(self, dt, q):
        self.p = [self.p[0] + dt * self.v[0], self.p[1] + dt * self.v[1]]
        pp, pv, vv = self.pp, self.pv, self.vv
        self.pp = pp + 2.0 * dt * pv + dt * dt * vv + q[0]
        self.pv = pv + dt * vv + q[1]
        self.vv = vv + q[2]

    def update(self, z, r2):
        pp, pv, vv = self.pp, self.pv, self.vv
        S = pp + r2
        k0, k1 = pp / S, pv / S
        for c in range(2):
            i = float(z[c]) - self.p[c]
            self.p[c] = self.p[c] + k0 * i
            self.v[c] = self.v[c] + k1 * i
        self.vv = vv - k1 * pv
        self.pv = pv - k0 * pv
        self.pp = pp - k0 * pp

    def step(self, z, prm, dt):
        """One tick: z the detected position, or None for a miss."""
        r2 = prm["meas_noise"] * prm["meas_noise"]
        if self.hits > 0:
            self.predict(dt, noise_terms(prm["accel_noise"], dt))
        if z is not None:
            if self.hits == 0:
                self.p = [float(z[0]), float(z[1])]
                self.v = [0.0, 0.0]
                self.pp, self.pv, self.vv = r2, 0.0, prm["init_vel_std"] * prm["init_vel_std"]
                self.hits = 1
            else:
                self.update(z, r2)
                self.hits = min(self.hits + 1, MAX_HITS)
            self.misses = 0
        elif self.hits > 0:
            self.misses += 1
            if self.misses > prm["max_coast_ticks"]:
                self.hits = self.misses = 0

    def published(self, prm):
        return self.hits >= prm["confirm_hits"]

    def row(self):
        return [self.p[0], self.p[1], self.v[0], self.v[1], 0.0]


class RobotTracker:
    """The tracks of one robot (ids 0..M-1) and the lists it published, for the latency."""

    def __init__(self, M, prm, dt):
        self.prm, self.dt = dict(prm), dt
        self.tracks = [Track() for _ in range(M)]
        self.history = []  # published (rows [m][5], ids [m]) per tick the robot ran

    def tick(self, ids, z):
        """One tick the robot runs: ids [n] of its list's rows in order, z [n] their detections (None: missed).
        Publishes (rows, ids) in list order and returns what the FOV filter receives: the list of latency ticks ago,
        empty before."""
        rows, out = [], []
        for i, zi in zip(ids, z):
            tr = self.tracks[i]
            tr.step(zi, self.prm, self.dt)
            if tr.published(self.prm):
                rows.append(tr.row())
                out.append(i)
        self.history.append((np.array(rows).reshape(-1, 5), np.array(out, np.int64)))
        k, d = len(self.history) - 1, self.prm["latency_ticks"]
        return self.history[k - d] if k >= d else (np.zeros((0, 5)), np.zeros(0, np.int64))


def tracked_all(trackers, lists, n_list, poses, active, k, pprm, costmaps, origins, res, costmap_index=None, R=1,
                K=None, stream_index=None):
    """Tick k of every robot b with trackers[b] (RobotTracker, M = K + R in shared scenes, else K): the detections of
    perception_ref.perceive under pprm (vel_noise 0), the tracker step, and what the FOV filter receives. Returns a
    dict of seen [B][L][5] (zero rows past n), n_seen [B], ids [B][L] (-1 past n), missed [B] (a person within 1.2 m
    not detected), untracked [B] (a person within 1.2 m not delivered), rows [B], pos_err [B], vel_err [B]; inactive
    robots deliver nothing and their tracks freeze."""
    B, L = lists.shape[0], lists.shape[1]
    K = L - (R - 1) if K is None else K
    out = dict(seen=np.zeros((B, L, 5)), n_seen=np.zeros(B, np.int32), ids=np.full((B, L), -1, np.int32),
               missed=np.zeros(B, bool), untracked=np.zeros(B, bool), rows=np.zeros(B, np.int32),
               pos_err=np.zeros(B), vel_err=np.zeros(B))
    for b in range(B):
        if not active[b]:
            continue
        n = int(n_list[b])
        rows_in = np.asarray(lists[b, :n], dtype=np.float64)
        mi = int(costmap_index[b]) if costmap_index is not None else b % costmaps.shape[0]
        stream = int(stream_index[b]) if stream_index is not None else b
        me = b % R
        seen, vis, miss = pref.perceive(rows_in, poses[b], k, stream, pprm, costmaps[mi], origins[mi], res, R=R, K=K,
                                        me=me)
        ids = pref.agent_ids(n, R, K, me)
        z = [None] * n
        for r, j in enumerate(np.flatnonzero(vis)):
            z[j] = seen[r, :2]
        rows, got = trackers[b].tick(ids, z)
        m = rows.shape[0]
        out["seen"][b, :m] = rows
        out["n_seen"][b] = m
        out["ids"][b, :m] = got
        out["missed"][b] = miss
        people = set()
        for row, i in zip(rows, got):
            if i >= K:
                continue  # a robot
            people.add(int(i))
            t = rows_in[i + R - 1]
            out["rows"][b] += 1
            out["pos_err"][b] += math.sqrt((row[0] - t[0]) ** 2 + (row[1] - t[1]) ** 2)
            out["vel_err"][b] += math.sqrt((row[2] - t[2]) ** 2 + (row[3] - t[3]) ** 2)
        rx, ry = float(poses[b][0]), float(poses[b][1])
        for j in range(R - 1, n):
            dx, dy = float(rows_in[j, 0]) - rx, float(rows_in[j, 1]) - ry
            if math.sqrt(dx * dx + dy * dy) < PERSONAL and (j - (R - 1)) not in people:
                out["untracked"][b] = True
    return out
