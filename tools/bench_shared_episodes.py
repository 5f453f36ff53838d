#!/usr/bin/env python
"""Closed-loop episodes in shared scenes on one GPU, alternating the arms within one run at each B:
  shared_R<R>  FleetOptimizer.run_shared_episodes on scenarios.shared_episodes(B / R, R, K) scenes: R robots per scene
               share one reactive crowd and see each other as people;
  crowd        FleetOptimizer.run_crowd_episodes on scenarios.crowd_episodes(B, K) scenes (one robot per scene).
The scenes differ, so the comparison is one of speed only. Per arm and B: robot ticks/s, ms per tick, kernel launches
per tick (smpc_launch_count) and the outcome summary (reached fraction, the robot_min_dist distribution, the share of
episodes with robot_intimate_ticks > 0). The scene view kernel moves B * (K + R - 1) * 40 bytes per tick in each
direction; that figure is reported beside the time. The card's name and power limit are read in the same run. Writes
one JSON (stdout and --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nav2_social_mpc_controller_b200 import scenarios as sc  # noqa: E402
from nav2_social_mpc_controller_b200.fleet import FleetOptimizer  # noqa: E402
from tools.bench_crowd_episodes import crowd_summary  # noqa: E402
from tools.bench_episodes import _args, _card  # noqa: E402


def shared_summary(r):
    out = crowd_summary(r)
    d = r["robot_min_dist"]
    fin = d[np.isfinite(d)]
    out.update(robot_min_dist_m=({"min": float(fin.min()), "p05": float(np.percentile(fin, 5)),
                                  "p50": float(np.percentile(fin, 50)), "p95": float(np.percentile(fin, 95))}
                                 if fin.size else None),
               episodes_with_robot_intimate_ticks=float(np.mean(r["robot_intimate_ticks"] > 0)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,4096,16384")
    ap.add_argument("--robots", default="1,2,4", help="robots per scene of the shared arms")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--substeps", type=int, default=1)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_shared_episodes.py needs a CUDA device")
    K = a.people
    result = {"card": _card(), "ticks": a.ticks, "people": K, "agents": 3, "substeps": a.substeps,
              "param_set": "soc_work_obst", "control_period_s": 0.05,
              "timing": "wall clock of the whole run, ending in a device synchronise; best of the reps",
              "note": "the arms run different scenes: a speed comparison only", "sizes": {}}
    for B in [int(x) for x in a.sizes.split(",")]:
        scenes = {"crowd": sc.crowd_episodes(B, K, ticks=a.ticks, substeps=a.substeps)}
        for R in [int(x) for x in a.robots.split(",")]:
            scenes[f"shared_R{R}"] = sc.shared_episodes(B // R, R, K, ticks=a.ticks, substeps=a.substeps)
        fl = FleetOptimizer(scenes["crowd"]["params"], n_robots=B, n_agents=3)

        def arm(name):
            s = _args(scenes[name])
            if name == "crowd":
                return lambda T: fl.run_crowd_episodes(ticks=T, **s)
            return lambda T: fl.run_shared_episodes(ticks=T, **s)
        arms = {n: arm(n) for n in scenes}
        for fn in arms.values():  # warm-up: module loads, allocations of this shape
            fn(3)
        times = {n: [] for n in arms}
        launches = {n: 0 for n in arms}
        last = {}
        for _ in range(a.reps):
            for name, fn in arms.items():
                c0 = fl.opt.launch_count()
                t0 = time.perf_counter()
                last[name] = fn(a.ticks)
                torch.cuda.synchronize()
                times[name].append(time.perf_counter() - t0)
                launches[name] = fl.opt.launch_count() - c0
        fl.close()
        entry = {}
        for name in arms:
            ticks_run = int(np.max(last[name]["ticks"]))
            best = min(times[name])
            e = {"robot_ticks_per_s": B * ticks_run / best, "ms_per_tick": 1e3 * best / ticks_run,
                 "ticks_run": ticks_run, "launches_per_tick": launches[name] / ticks_run,
                 "runs_s": [round(t, 4) for t in times[name]],
                 "outcome": crowd_summary(last[name]) if name == "crowd" else shared_summary(last[name])}
            if name != "crowd":
                R = scenes[name]["robots_per_scene"]
                e["scene_view_bytes_per_tick"] = 2 * B * (K + R - 1) * 40
            entry[name] = e
        for name in arms:
            if name != "crowd":
                entry[name]["ms_per_tick_over_crowd"] = entry[name]["ms_per_tick"] / entry["crowd"]["ms_per_tick"]
        result["sizes"][str(B)] = entry
        print(json.dumps({str(B): entry}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
