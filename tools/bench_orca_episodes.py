#!/usr/bin/env python
"""Closed-loop episodes with an ORCA crowd against the lightsfm crowd on one GPU, alternating the two arms on the same
scenes within one run:
  orca       run_crowd_episodes / run_shared_episodes with orca=abi.orca_params() (smpc_run_orca_episodes);
  lightsfm   the same entry without orca (the social force crowd the controller's projection also uses).
Scenes: scenarios.crowd_episodes (R = 1) or scenarios.shared_episodes (R = 2), K people, T ticks. Per arm, B and R:
robot ticks/s, ms and kernel launches per tick, and the outcomes side by side (reached fraction, intimate and personal
ticks, the 5th percentile of the nearest person distance, collisions): the point of the ORCA crowd is how the
controller fares against people it does not predict. With --profile a separate run under torch.profiler (CUDA
activities, trace under --trace-dir) gives each crowd kernel's ms per tick and its share of all kernel time. The
card's name and power limit are read in the same run. Writes one JSON (stdout and --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nav2_social_mpc_controller_b200 import abi, scenarios as sc  # noqa: E402
from nav2_social_mpc_controller_b200.fleet import FleetOptimizer  # noqa: E402
from tools.bench_episodes import _args, _card  # noqa: E402

KERNELS = {"orca": "smpc_orca_step_kernel", "lightsfm": "smpc_crowd_step_kernel"}


def scenes(B, R, K, T, substeps):
    if R == 1:
        return sc.crowd_episodes(B, K, ticks=T, substeps=substeps)
    return sc.shared_episodes(B // R, R, K, ticks=T, substeps=substeps)


def arm(fl, s, name):
    fn = fl.run_crowd_episodes if "robots_per_scene" not in s else fl.run_shared_episodes
    orca = abi.orca_params() if name == "orca" else None
    return lambda T: fn(ticks=T, orca=orca, **_args(s))


def outcome(r):
    return {"reached_fraction": float(np.mean(r["reached"])),
            "mean_intimate_ticks": float(np.mean(r["intimate_ticks"])),
            "mean_personal_ticks": float(np.mean(r["personal_ticks"])),
            "p5_min_person_dist_m": float(np.percentile(r["min_person_dist"], 5)),
            "episodes_with_collision": float(np.mean(r["collision_ticks"] > 0)),
            "mean_collision_ticks": float(np.mean(r["collision_ticks"])),
            "mean_people_disturbance": float(np.mean(r["people_disturbance"]))}


def profile(B, R, K, T, substeps, trace_dir):
    """One run per arm under torch.profiler: the crowd kernel's time per tick and share of kernel time."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    s = scenes(B, R, K, T, substeps)
    fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
    out = {}
    for name in KERNELS:
        fn = arm(fl, s, name)
        fn(3)  # warm-up
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            r = fn(T)
            torch.cuda.synchronize()
        os.makedirs(trace_dir, exist_ok=True)
        trace = os.path.join(trace_dir, f"{name}_episodes_B{B}_R{R}.pt.trace.json")
        prof.export_chrome_trace(trace)
        ticks_run = int(np.max(r["ticks"]))
        total_us, crowd_us = 0.0, 0.0
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t <= 0 or "Memcpy" in e.key or "Memset" in e.key:
                continue
            total_us += t
            if KERNELS[name] in e.key:
                crowd_us += t
        out[name] = {"ticks_run": ticks_run, "crowd_kernel": KERNELS[name],
                     "crowd_kernel_ms_per_tick": crowd_us / 1e3 / ticks_run,
                     "kernel_ms_per_tick": total_us / 1e3 / ticks_run,
                     "crowd_kernel_share_of_kernel_time": crowd_us / total_us if total_us else None,
                     "trace": os.path.basename(trace)}
    fl.close()
    return {"B": B, "R": R, **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="64,4096,16384")
    ap.add_argument("--robots", default="1,2", help="robots per scene")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--substeps", type=int, default=1)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--profile", type=int, default=0, help="B of a separate profiled run per R (0: none)")
    ap.add_argument("--trace-dir", default="profiles_run")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_orca_episodes.py needs a CUDA device")
    result = {"card": _card(), "ticks": a.ticks, "people": a.people, "agents": 3, "substeps": a.substeps,
              "param_set": "soc_work_obst", "control_period_s": 0.05, "orca": dict(abi.ORCA_DEFAULTS),
              "timing": "wall clock of the whole run, ending in a device synchronise; best of the reps",
              "runs": {}}
    for R in [int(x) for x in a.robots.split(",")]:
        for B in [int(x) for x in a.sizes.split(",")]:
            s = scenes(B, R, a.people, a.ticks, a.substeps)
            fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
            arms = {name: arm(fl, s, name) for name in KERNELS}
            for fn in arms.values():  # warm-up: module loads, allocations of this shape
                fn(3)
            times = {n: [] for n in arms}
            launches, last = {}, {}
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
                               "runs_s": [round(t, 4) for t in times[name]], "outcome": outcome(last[name])}
            entry["orca_ms_per_tick_over_lightsfm"] = entry["orca"]["ms_per_tick"] / entry["lightsfm"]["ms_per_tick"]
            key = f"B{B}_R{R}"
            result["runs"][key] = entry
            print(json.dumps({key: entry}), flush=True)
        if a.profile:
            result.setdefault("profile", {})[f"R{R}"] = profile(a.profile, R, a.people, a.ticks, a.substeps,
                                                                 a.trace_dir)
            print(json.dumps({"profile": result["profile"][f"R{R}"]}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
