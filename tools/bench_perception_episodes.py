#!/usr/bin/env python
"""Closed-loop episodes with sensor-limited perception against perfect perception on one GPU, alternating the two arms
on the same scenes within one run:
  default    perception=abi.perception_params() (smpc_run_perceived_episodes): 8 m range, occlusion by walls and
             people, 95 % detection, noisy tracks;
  neutral    perception with the neutral parameters: the same entry computing what the entry without perception
             computes, plus the stage's launch.
Scenes: scenarios.crowd_episodes (R = 1) or scenarios.shared_episodes (R = 2), K people, T ticks, in the lightsfm and
the ORCA crowd. Per crowd, arm, B and R: robot ticks/s, ms and kernel launches per tick, and the outcomes side by side
(intimate and personal ticks, the 5th percentile of the nearest person distance, collisions, unseen_personal_ticks,
the mean list length the FOV filter received). With --profile a separate run under torch.profiler (CUDA activities,
trace under --trace-dir) gives the perception kernel's ms per tick and its share of all kernel time. The card's name
and power limit are read in the same run. Writes one JSON (stdout and --out)."""
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

KERNEL = "smpc_perception_kernel"
ARMS = {"default": {}, "neutral": dict(abi.PERCEPTION_NEUTRAL)}


def scenes(B, R, K, T):
    if R == 1:
        return sc.crowd_episodes(B, K, ticks=T)
    return sc.shared_episodes(B // R, R, K, ticks=T)


def arm(fl, s, crowd, name):
    fn = fl.run_crowd_episodes if "robots_per_scene" not in s else fl.run_shared_episodes
    orca = abi.orca_params() if crowd == "orca" else None
    return lambda T, want_logs=False: fn(ticks=T, orca=orca, perception=ARMS[name], want_logs=want_logs, **_args(s))


def outcome(r):
    ran = np.arange(r["n_seen_log"].shape[1])[None, :] < r["ticks"][:, None]
    return {"reached_fraction": float(np.mean(r["reached"])),
            "mean_intimate_ticks": float(np.mean(r["intimate_ticks"])),
            "mean_personal_ticks": float(np.mean(r["personal_ticks"])),
            "p5_min_person_dist_m": float(np.percentile(r["min_person_dist"], 5)),
            "episodes_with_collision": float(np.mean(r["collision_ticks"] > 0)),
            "mean_collision_ticks": float(np.mean(r["collision_ticks"])),
            "mean_unseen_personal_ticks": float(np.mean(r["unseen_personal_ticks"])),
            "mean_reported_list_length": float(r["n_seen_log"][ran].mean())}


def profile(B, K, T, trace_dir):
    """One run per crowd with the default perception under torch.profiler: the perception kernel's time per tick and
    share of kernel time."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    s = scenes(B, 1, K, T)
    fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
    out = {}
    for crowd in ("lightsfm", "orca"):
        fn = arm(fl, s, crowd, "default")
        fn(3)  # warm-up
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            r = fn(T)
            torch.cuda.synchronize()
        os.makedirs(trace_dir, exist_ok=True)
        trace = os.path.join(trace_dir, f"perception_{crowd}_B{B}.pt.trace.json")
        prof.export_chrome_trace(trace)
        ticks_run = int(np.max(r["ticks"]))
        total_us, stage_us = 0.0, 0.0
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t <= 0 or "Memcpy" in e.key or "Memset" in e.key:
                continue
            total_us += t
            if KERNEL in e.key:
                stage_us += t
        out[crowd] = {"ticks_run": ticks_run, "perception_kernel_ms_per_tick": stage_us / 1e3 / ticks_run,
                      "kernel_ms_per_tick": total_us / 1e3 / ticks_run,
                      "perception_share_of_kernel_time": stage_us / total_us if total_us else None,
                      "trace": os.path.basename(trace)}
    fl.close()
    return {"B": B, "R": 1, **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="64x1,4096x1,16384x1,16384x2", help="B x robots per scene")
    ap.add_argument("--crowds", default="lightsfm,orca")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--profile", type=int, default=0, help="B of a separate profiled run per crowd (0: none)")
    ap.add_argument("--trace-dir", default="profiles_run")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_perception_episodes.py needs a CUDA device")
    result = {"card": _card(), "ticks": a.ticks, "people": a.people, "agents": 3, "param_set": "soc_work_obst",
              "control_period_s": 0.05, "perception": dict(abi.PERCEPTION_DEFAULTS),
              "timing": "wall clock of the whole run without logs, ending in a device synchronise; best of the reps",
              "outcomes": "from one more run per arm with every log on", "runs": {}}
    for crowd in a.crowds.split(","):
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
            entry = {}
            for name, fn in arms.items():
                best = min(times[name])
                entry[name] = {"robot_ticks_per_s": B * ticks_run[name] / best,
                               "ms_per_tick": 1e3 * best / ticks_run[name], "ticks_run": ticks_run[name],
                               "launches_per_tick": launches[name] / ticks_run[name],
                               "runs_s": [round(t, 4) for t in times[name]], "outcome": outcome(fn(a.ticks, True))}
            fl.close()
            entry["default_ms_per_tick_over_neutral"] = entry["default"]["ms_per_tick"] / entry["neutral"]["ms_per_tick"]
            key = f"{crowd}_B{B}_R{R}"
            result["runs"][key] = entry
            print(json.dumps({key: entry}), flush=True)
    if a.profile:
        result["profile"] = profile(a.profile, a.people, a.ticks, a.trace_dir)
        print(json.dumps({"profile": result["profile"]}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
