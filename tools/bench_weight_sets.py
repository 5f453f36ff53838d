#!/usr/bin/env python
"""Per-robot critic weights on one GPU: P controller tunings on the same reactive-crowd scenes, three arms alternating
within one run:
  weighted  one FleetOptimizer.run_crowd_episodes(weights=...) call over B = P * B0 episodes: scenarios.crowd_episodes
            (B0, K) tiled P times (scenarios.tile_scenes), episode p * B0 + i = scene i under set p;
  per_set   P unweighted calls of B0 episodes, each on a handle whose params carry set p (explicit costmap_index, so
            every scene keeps its map);
  plain     one unweighted call over the B tiled episodes on the weighted arm's handle: the cost of the weighted kernel.
Per arm: robot ticks/s, ms per tick, kernel launches per tick (smpc_launch_count). Per set: the outcome means of the
weighted arm. The weighted arm must equal the per_set arm bit for bit in every metric; the script exits non-zero when
it does not. The card's name and power limit are read in the same run. Writes one JSON (stdout and --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nav2_social_mpc_controller_b200 import scenarios as sc  # noqa: E402
from nav2_social_mpc_controller_b200.fleet import FleetOptimizer  # noqa: E402
from nav2_social_mpc_controller_b200.optimizer import weight_sets  # noqa: E402
from tools.bench_episodes import _args, _card  # noqa: E402

OUTCOMES = ("reached", "ticks", "min_person_dist", "intimate_ticks", "people_disturbance", "path_length")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", default="obst_only,soc_work_obst", help="scenarios.PARAM_SETS names, one per set")
    ap.add_argument("--scenes", type=int, default=8192, help="B0 scenes per set")
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--substeps", type=int, default=1)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm, alternating the arms")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_weight_sets.py needs a CUDA device")
    names = a.sets.split(",")
    P, B0, T = len(names), a.scenes, a.ticks
    B = P * B0
    s = sc.crowd_episodes(B0, a.people, ticks=T, substeps=a.substeps, param_set=names[-1])
    rows = [sc.make_params(n) for n in names]
    table = weight_sets(rows, s["params"])
    idx = np.repeat(np.arange(P), B0).astype(np.int32)
    tiled = sc.tile_scenes(s, P)
    base = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
    own = [FleetOptimizer(r, n_robots=B0, n_agents=3) for r in rows]

    def weighted(T_):
        return [base.run_crowd_episodes(ticks=T_, weights=(table, idx), **_args(tiled))]

    def per_set(T_):
        return [fl.run_crowd_episodes(ticks=T_, **_args(s)) for fl in own]

    def plain(T_):
        return [base.run_crowd_episodes(ticks=T_, **_args(tiled))]

    arms = {"weighted": weighted, "per_set": per_set, "plain": plain}
    for fn in arms.values():  # warm-up: module loads, allocations of this shape
        fn(3)
    times = {n: [] for n in arms}
    launches, last = {}, {}
    for _ in range(a.reps):
        for name, fn in arms.items():
            c0 = base.opt.launch_count() + sum(fl.opt.launch_count() for fl in own)
            t0 = time.perf_counter()
            last[name] = fn(T)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
            launches[name] = base.opt.launch_count() + sum(fl.opt.launch_count() for fl in own) - c0
    base.close()
    for fl in own:
        fl.close()
    w = last["weighted"][0]
    split = {k: np.concatenate([r[k] for r in last["per_set"]]) for k in w}
    mismatch = [k for k in w if not np.array_equal(w[k], split[k])]
    result = {"card": _card(), "sets": names, "scenes_per_set": B0, "episodes": B, "people": a.people, "agents": 3,
              "ticks": T, "substeps": a.substeps, "control_period_s": 0.05,
              "timing": "wall clock of the whole arm, ending in a device synchronise; best of the reps",
              "weighted_equals_per_set_bit_for_bit": not mismatch, "mismatched_metrics": mismatch, "arms": {}}
    for name in arms:
        ticks_run = int(max(int(np.max(r["ticks"])) for r in last[name]))
        best = min(times[name])
        result["arms"][name] = {"robot_ticks_per_s": B * ticks_run / best, "ms_per_tick": 1e3 * best / ticks_run,
                                "ticks_run": ticks_run, "launches_per_tick": launches[name] / ticks_run,
                                "runs_s": [round(t, 4) for t in times[name]]}
    arms_out = result["arms"]
    arms_out["weighted"]["ms_per_tick_over_plain"] = arms_out["weighted"]["ms_per_tick"] / arms_out["plain"]["ms_per_tick"]
    arms_out["weighted"]["ms_per_tick_over_per_set"] = (arms_out["weighted"]["ms_per_tick"] /
                                                        arms_out["per_set"]["ms_per_tick"])
    result["outcome_means_by_set"] = {
        n: {k: float(np.mean(w[k][p * B0:(p + 1) * B0].astype(np.float64))) for k in OUTCOMES}
        for p, n in enumerate(names)}
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    if mismatch:
        raise SystemExit(f"weighted and per-set runs differ in {mismatch}")


if __name__ == "__main__":
    main()
