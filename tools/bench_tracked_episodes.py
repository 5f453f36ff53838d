#!/usr/bin/env python
"""Closed-loop episodes with a people tracker against white-noise tracks on one GPU, alternating the two arms on the
same scenes within one run:
  white      perception=abi.perception_params() (smpc_run_perceived_episodes): the default sensor, whose velocities
             are the true ones plus fresh white noise every tick;
  tracked    the default sensor with vel_noise=0 followed by tracker=abi.tracker_params() (smpc_run_tracked_episodes):
             velocities estimated by a constant-velocity Kalman filter, 3 detections to confirm, 10 coasted misses,
             2 ticks of latency.
Scenes: scenarios.crowd_episodes (R = 1) or scenarios.shared_episodes (R = 2), K people, T ticks, in the lightsfm and
the ORCA crowd. Per crowd, arm, B and R: robot ticks/s, ms and kernel launches per tick, and the outcomes side by side
(intimate and personal ticks, the 5th percentile of the nearest person distance, collisions, unseen and untracked
personal ticks, the mean track errors). With --profile a separate run under torch.profiler (CUDA activities, trace
under --trace-dir) gives the perception and tracker kernels' ms per tick and share of all kernel time. The card's
name and power limit are read in the same run. Writes one JSON (stdout and --out)."""
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

KERNELS = {"white": "smpc_perception_kernel", "tracked": "smpc_tracked_perception_kernel"}
ARMS = {"white": dict(perception={}), "tracked": dict(perception=dict(vel_noise=0.0), tracker={})}


def scenes(B, R, K, T):
    if R == 1:
        return sc.crowd_episodes(B, K, ticks=T)
    return sc.shared_episodes(B // R, R, K, ticks=T)


def arm(fl, s, crowd, name):
    fn = fl.run_crowd_episodes if "robots_per_scene" not in s else fl.run_shared_episodes
    orca = abi.orca_params() if crowd == "orca" else None
    return lambda T: fn(ticks=T, orca=orca, want_logs=False, **ARMS[name], **_args(s))


def outcome(r):
    out = {"reached_fraction": float(np.mean(r["reached"])),
           "mean_intimate_ticks": float(np.mean(r["intimate_ticks"])),
           "mean_personal_ticks": float(np.mean(r["personal_ticks"])),
           "p5_min_person_dist_m": float(np.percentile(r["min_person_dist"], 5)),
           "episodes_with_collision": float(np.mean(r["collision_ticks"] > 0)),
           "mean_collision_ticks": float(np.mean(r["collision_ticks"])),
           "mean_unseen_personal_ticks": float(np.mean(r["unseen_personal_ticks"]))}
    if "track_rows" in r:
        rows = r["track_rows"]
        some = rows > 0
        out.update(mean_untracked_personal_ticks=float(np.mean(r["untracked_personal_ticks"])),
                   mean_track_rows_per_tick=float(rows.sum() / r["ticks"].sum()),
                   mean_track_pos_error_m=float((r["mean_track_pos_error"][some] * rows[some]).sum() / rows.sum()),
                   mean_track_vel_error_mps=float((r["mean_track_vel_error"][some] * rows[some]).sum() / rows.sum()))
    return out


def profile(B, K, T, trace_dir):
    """One run per crowd and arm under torch.profiler: the perception (white) or tracked perception (tracked) kernel's
    time per tick and share of kernel time."""
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
            trace = os.path.join(trace_dir, f"tracked_{crowd}_{name}_B{B}.pt.trace.json")
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
                if KERNELS[name] in e.key:
                    stage_us += t
            out[f"{crowd}_{name}"] = {"kernel": KERNELS[name], "ticks_run": ticks_run,
                                      "stage_kernel_ms_per_tick": stage_us / 1e3 / ticks_run,
                                      "kernel_ms_per_tick": total_us / 1e3 / ticks_run,
                                      "stage_share_of_kernel_time": stage_us / total_us if total_us else None,
                                      "trace": os.path.basename(trace)}
    fl.close()
    return {"B": B, "R": 1, **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="64x1,4096x1,16384x1,64x2,4096x2,16384x2", help="B x robots per scene")
    ap.add_argument("--crowds", default="lightsfm,orca")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--profile", type=int, default=0, help="B of a separate profiled run per crowd and arm (0: none)")
    ap.add_argument("--trace-dir", default="profiles_run")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_tracked_episodes.py needs a CUDA device")
    result = {"card": _card(), "ticks": a.ticks, "people": a.people, "agents": 3, "param_set": "soc_work_obst",
              "control_period_s": 0.05, "perception": dict(abi.PERCEPTION_DEFAULTS),
              "tracker": dict(abi.TRACKER_DEFAULTS),
              "timing": "wall clock of the whole run without logs, ending in a device synchronise; best of the reps",
              "outcomes": "from the last timed run of each arm", "runs": {}}
    for crowd in a.crowds.split(","):
        for cfg in a.configs.split(","):
            B, R = (int(x) for x in cfg.split("x"))
            s = scenes(B, R, a.people, a.ticks)
            fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
            arms = {name: arm(fl, s, crowd, name) for name in ARMS}
            for fn in arms.values():  # warm-up: module loads, allocations of this shape
                fn(3)
            times = {n: [] for n in arms}
            launches, ticks_run, last = {}, {}, {}
            for _ in range(a.reps):
                for name, fn in arms.items():
                    c0 = fl.opt.launch_count()
                    t0 = time.perf_counter()
                    r = fn(a.ticks)
                    torch.cuda.synchronize()
                    times[name].append(time.perf_counter() - t0)
                    launches[name] = fl.opt.launch_count() - c0
                    ticks_run[name] = int(np.max(r["ticks"]))
                    last[name] = r
            fl.close()
            entry = {}
            for name in arms:
                best = min(times[name])
                entry[name] = {"robot_ticks_per_s": B * ticks_run[name] / best,
                               "ms_per_tick": 1e3 * best / ticks_run[name], "ticks_run": ticks_run[name],
                               "launches_per_tick": launches[name] / ticks_run[name],
                               "runs_s": [round(t, 4) for t in times[name]], "outcome": outcome(last[name])}
            entry["tracked_ms_per_tick_over_white"] = entry["tracked"]["ms_per_tick"] / entry["white"]["ms_per_tick"]
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
