#!/usr/bin/env python
"""Closed-loop episodes with a reactive crowd on one GPU, alternating two arms within one run:
  crowd      FleetOptimizer.run_crowd_episodes on scenarios.crowd_episodes scenes (people walk to goals under the
             social force model and react to the robot; 13 launches per tick);
  episodes   FleetOptimizer.run_episodes on scenarios.episodes scenes of the same B and K (constant-velocity people).
The scenes differ, so the comparison is one of speed only. Per arm and B: robot ticks/s, ms per tick, kernel launches
per tick (smpc_launch_count) and the outcome summary. With --profile a separate run under torch.profiler (CUDA
activities, trace written under --trace-dir) gives the time of smpc_crowd_step_kernel per tick and its share of all
kernel time of the tick. The card's name and power limit are read in the same run. Writes one JSON (stdout and
--out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nav2_social_mpc_controller_b200 import scenarios as sc  # noqa: E402
from nav2_social_mpc_controller_b200.fleet import FleetOptimizer  # noqa: E402
from tools.bench_episodes import _args, _card, summary  # noqa: E402


def crowd_summary(r):
    out = summary(r)
    out.update(min_person_dist_min_m=float(np.min(r["min_person_dist"])),
               episodes_within_1cm_of_a_person=float(np.mean(r["min_person_dist"] < 0.01)),
               mean_people_disturbance=float(np.mean(r["people_disturbance"])),
               p95_people_disturbance=float(np.percentile(r["people_disturbance"], 95)))
    return out


def profile_crowd(B, K, T, trace_dir):
    """One run_crowd_episodes under torch.profiler: smpc_crowd_step_kernel time per tick and share of kernel time."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    s = sc.crowd_episodes(B, K, ticks=T)
    fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
    args = _args(s)
    fl.run_crowd_episodes(ticks=3, **args)  # warm-up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fl.run_crowd_episodes(ticks=T, **args)
        torch.cuda.synchronize()
    fl.close()
    os.makedirs(trace_dir, exist_ok=True)
    trace = os.path.join(trace_dir, f"crowd_episodes_B{B}.pt.trace.json")
    prof.export_chrome_trace(trace)
    ticks_run = int(np.max(r["ticks"]))
    total_us, crowd_us, crowd_n = 0.0, 0.0, 0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0:
            continue
        if "Memcpy" in e.key or "Memset" in e.key:
            continue
        total_us += t
        if "smpc_crowd_step_kernel" in e.key:
            crowd_us += t
            crowd_n += e.count
    return {"B": B, "ticks_run": ticks_run, "crowd_step_launches": crowd_n,
            "crowd_step_ms_per_tick": crowd_us / 1e3 / ticks_run, "kernel_ms_per_tick": total_us / 1e3 / ticks_run,
            "crowd_step_share_of_kernel_time": crowd_us / total_us if total_us else None,
            "trace": os.path.basename(trace)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,64,4096,16384")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--substeps", type=int, default=1)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--profile", type=int, default=0, help="B of a separate profiled crowd run (0: none)")
    ap.add_argument("--trace-dir", default="profiles_run")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_crowd_episodes.py needs a CUDA device")
    result = {"card": _card(), "ticks": a.ticks, "people": a.people, "agents": 3, "substeps": a.substeps,
              "param_set": "soc_work_obst", "control_period_s": 0.05,
              "timing": "wall clock of the whole run, ending in a device synchronise; best of the reps",
              "note": "the arms run different scenes (reactive vs constant-velocity people): a speed comparison only",
              "sizes": {}}
    for B in [int(x) for x in a.sizes.split(",")]:
        sc_crowd = sc.crowd_episodes(B, a.people, ticks=a.ticks, substeps=a.substeps)
        sc_cv = sc.episodes(B, a.people, ticks=a.ticks)
        fl = FleetOptimizer(sc_crowd["params"], n_robots=B, n_agents=3)
        arms = {"crowd": lambda T: fl.run_crowd_episodes(ticks=T, **_args(sc_crowd)),
                "episodes": lambda T: fl.run_episodes(ticks=T, **_args(sc_cv))}
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
            entry[name] = {"robot_ticks_per_s": B * ticks_run / best, "ms_per_tick": 1e3 * best / ticks_run,
                           "ticks_run": ticks_run, "launches_per_tick": launches[name] / ticks_run,
                           "runs_s": [round(t, 4) for t in times[name]],
                           "outcome": crowd_summary(last[name]) if name == "crowd" else summary(last[name])}
        entry["crowd_ms_per_tick_over_episodes"] = entry["crowd"]["ms_per_tick"] / entry["episodes"]["ms_per_tick"]
        result["sizes"][str(B)] = entry
        print(json.dumps({str(B): entry}), flush=True)
    if a.profile:
        result["profile"] = profile_crowd(a.profile, a.people, a.ticks, a.trace_dir)
        print(json.dumps({"profile": result["profile"]}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
