#!/usr/bin/env python
"""Closed-loop episodes with a rolling local costmap against the static map on one GPU, alternating three arms on the
same scenes within one run:
  static     no local costmap (smpc_run_crowd_episodes / smpc_run_orca_episodes / smpc_run_shared_episodes): the FOV
             filter and the fleet tick read the whole static corridor map;
  window0    local_costmap=dict(mark_people=0) (smpc_run_local_costmap_episodes): an 80 x 80 window around each robot,
             rebuilt every 4 ticks, with the static layer only;
  window     local_costmap=abi.local_costmap_params(): the same window with the people marked and inflated.
Scenes: scenarios.crowd_episodes (R = 1) or scenarios.shared_episodes (R = 2), K people, T ticks, in the lightsfm and
the ORCA crowd. Per crowd, arm, B and R: robot ticks/s, ms and kernel launches per tick. With --profile a separate run
under torch.profiler (CUDA activities, trace under --trace-dir) gives per arm the window kernel's ms per tick and share
of kernel time and the solve kernel's ms per tick: the solve reads B distinct windows instead of a few shared maps.
With --outcome-scenes the obst_only and soc_work_obst critic weights run as a weight table on the same scenes
(scenarios.tile_scenes) for --outcome-ticks ticks, per crowd and arm: intimate and personal ticks, the 5th percentile
of the nearest person distance, collision episodes, reached and mean marked_rows. The card's name and power limit are
read in the same run. Writes one JSON (stdout and --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nav2_social_mpc_controller_b200 import abi, scenarios as sc  # noqa: E402
from nav2_social_mpc_controller_b200.fleet import FleetOptimizer  # noqa: E402
from nav2_social_mpc_controller_b200.optimizer import weight_sets  # noqa: E402
from tools.bench_episodes import _args, _card  # noqa: E402

ARMS = {"static": {}, "window0": dict(local_costmap=dict(mark_people=0)), "window": dict(local_costmap={})}
WINDOW_KERNEL, SOLVE_KERNEL = "smpc_local_costmap_kernel", "smpc_solve_kernel"
TUNINGS = ("obst_only", "soc_work_obst")


def scenes(B, R, K, T):
    if R == 1:
        return sc.crowd_episodes(B, K, ticks=T)
    return sc.shared_episodes(B // R, R, K, ticks=T)


def arm(fl, s, crowd, name, **kw):
    fn = fl.run_crowd_episodes if "robots_per_scene" not in s else fl.run_shared_episodes
    orca = abi.orca_params() if crowd == "orca" else None
    return lambda T: fn(ticks=T, orca=orca, want_logs=False, **ARMS[name], **kw, **_args(s))


def outcome(r, sel):
    out = {"reached_fraction": float(np.mean(r["reached"][sel])),
           "mean_intimate_ticks": float(np.mean(r["intimate_ticks"][sel])),
           "mean_personal_ticks": float(np.mean(r["personal_ticks"][sel])),
           "p5_min_person_dist_m": float(np.percentile(r["min_person_dist"][sel], 5)),
           "episodes_with_collision": float(np.mean(r["collision_ticks"][sel] > 0))}
    if "marked_rows" in r:
        out["mean_marked_rows"] = float(np.mean(r["marked_rows"][sel]))
    return out


def profile(B, K, T, trace_dir):
    """One run per crowd and arm under torch.profiler: the window kernel's and the solve kernel's time per tick, and
    the window kernel's share of kernel time."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    s = scenes(B, 1, K, T)
    fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
    out = {}
    for crowd in ("lightsfm", "orca"):
        for name in ARMS:
            fn = arm(fl, s, crowd, name)
            fn(3)  # warm-up
            torch.cuda.synchronize()
            with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
                r = fn(T)
                torch.cuda.synchronize()
            os.makedirs(trace_dir, exist_ok=True)
            trace = os.path.join(trace_dir, f"local_costmap_{crowd}_{name}_B{B}.pt.trace.json")
            prof.export_chrome_trace(trace)
            ticks_run = int(np.max(r["ticks"]))
            total_us, window_us, solve_us = 0.0, 0.0, 0.0
            for e in prof.key_averages():
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                if t <= 0 or "Memcpy" in e.key or "Memset" in e.key:
                    continue
                total_us += t
                if WINDOW_KERNEL in e.key:
                    window_us += t
                if SOLVE_KERNEL in e.key:
                    solve_us += t
            out[f"{crowd}_{name}"] = {"ticks_run": ticks_run, "window_kernel_ms_per_tick": window_us / 1e3 / ticks_run,
                                      "window_share_of_kernel_time": window_us / total_us if total_us else None,
                                      "solve_kernel_ms_per_tick": solve_us / 1e3 / ticks_run,
                                      "kernel_ms_per_tick": total_us / 1e3 / ticks_run,
                                      "trace": os.path.basename(trace)}
    fl.close()
    return {"B": B, "R": 1, **out}


def outcomes(B0, K, T, crowds):
    """obst_only against soc_work_obst as a weight table on the same B0 scenes, per crowd and arm."""
    base = sc.make_params("soc_work_obst")
    table = weight_sets([sc.make_params(n) for n in TUNINGS], base)
    s = sc.tile_scenes(sc.crowd_episodes(B0, K, ticks=T), len(TUNINGS))
    B = B0 * len(TUNINGS)
    idx = np.repeat(np.arange(len(TUNINGS)), B0).astype(np.int32)
    fl = FleetOptimizer(base, n_robots=B, n_agents=3)
    out = {}
    for crowd in crowds:
        for name in ARMS:
            r = arm(fl, s, crowd, name, weights=(table, idx))(T)
            out[f"{crowd}_{name}"] = {t: outcome(r, idx == i) for i, t in enumerate(TUNINGS)}
            print(json.dumps({f"outcome_{crowd}_{name}": out[f"{crowd}_{name}"]}), flush=True)
    fl.close()
    return {"scenes": B0, "ticks": T, **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="64x1,4096x1,16384x1,64x2,4096x2,16384x2", help="B x robots per scene")
    ap.add_argument("--crowds", default="lightsfm,orca")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--profile", type=int, default=0, help="B of a separate profiled run per crowd and arm (0: none)")
    ap.add_argument("--trace-dir", default="profiles_run")
    ap.add_argument("--outcome-scenes", type=int, default=0, help="scenes of the tuning comparison (0: none)")
    ap.add_argument("--outcome-ticks", type=int, default=400, help="ticks of the tuning comparison")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_local_costmap_episodes.py needs a CUDA device")
    result = {"card": _card(), "ticks": a.ticks, "people": a.people, "agents": 3, "param_set": "soc_work_obst",
              "control_period_s": 0.05, "local_costmap": dict(abi.LOCAL_COSTMAP_DEFAULTS),
              "timing": "wall clock of the whole run without logs, ending in a device synchronise; best of the reps",
              "runs": {}}
    crowds = a.crowds.split(",")
    for crowd in crowds:
        for cfg in a.configs.split(","):
            B, R = (int(x) for x in cfg.split("x"))
            s = scenes(B, R, a.people, a.ticks)
            fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
            arms = {name: arm(fl, s, crowd, name) for name in ARMS}
            for fn in arms.values():  # warm-up: module loads, allocations of this shape
                fn(3)
            times = {n: [] for n in arms}
            launches, ticks_run = {}, {}
            for _ in range(a.reps):
                for name, fn in arms.items():
                    c0 = fl.opt.launch_count()
                    t0 = time.perf_counter()
                    r = fn(a.ticks)
                    torch.cuda.synchronize()
                    times[name].append(time.perf_counter() - t0)
                    launches[name] = fl.opt.launch_count() - c0
                    ticks_run[name] = int(np.max(r["ticks"]))
            fl.close()
            entry = {}
            for name in arms:
                best = min(times[name])
                entry[name] = {"robot_ticks_per_s": B * ticks_run[name] / best,
                               "ms_per_tick": 1e3 * best / ticks_run[name], "ticks_run": ticks_run[name],
                               "launches_per_tick": launches[name] / ticks_run[name],
                               "runs_s": [round(t, 4) for t in times[name]]}
            entry["window_ms_per_tick_over_static"] = entry["window"]["ms_per_tick"] / entry["static"]["ms_per_tick"]
            key = f"{crowd}_B{B}_R{R}"
            result["runs"][key] = entry
            print(json.dumps({key: entry}), flush=True)
    if a.profile:
        result["profile"] = profile(a.profile, a.people, a.ticks, a.trace_dir)
        print(json.dumps({"profile": result["profile"]}), flush=True)
    if a.outcome_scenes:
        result["outcomes"] = outcomes(a.outcome_scenes, a.people, a.outcome_ticks, crowds)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
