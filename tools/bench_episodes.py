#!/usr/bin/env python
"""Closed-loop episodes on one GPU, two arms on the same scenes (scenarios.episodes), alternating within one run:
  episodes    FleetOptimizer.run_episodes: one C call, every tick enqueued on one stream, one upload, one download;
  host_loop   the same ticks stepped from Python: trajectorize_batch, filter_people_fov, optimize_batch(inplace=True)
              and a numpy world step, i.e. three host round trips per tick.
Per arm and B: robot ticks/s, ms per tick, kernel launches per tick (smpc_launch_count), goal and metric summary; the
card's name and power limit are read in the same run. Writes one JSON (stdout and --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nav2_social_mpc_controller_b200 import scenarios as sc  # noqa: E402
from nav2_social_mpc_controller_b200.fleet import FleetOptimizer  # noqa: E402


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        name, limit = [x.strip() for x in q[0].split(",")]
        return {"name": name, "power_limit": limit}
    except Exception as e:  # the numbers are still reported, without the card
        return {"error": repr(e)}


def _args(s):
    return {k: v for k, v in s.items() if k not in ("params", "ticks")}


def host_loop(fl, s, T, goal_tolerance=0.25):
    """The tick loop of run_episodes written with the per-stage Python entries and a numpy world."""
    fl.reset_memory()  # run_episodes starts from fresh warm-start memory too
    gp, pose, speed = s["global_path"], s["pose"].copy(), s["speed"].copy()
    people0, n_people, dt = s["people"], s["n_people"], s["control_period"]
    cms, morg, res, od, cidx = s["costmaps"], s["costmap_origin"], s["costmap_resolution"], s["od"], s["costmap_index"]
    B, K = pose.shape[0], people0.shape[1]
    H, W = cms.shape[1:]
    goal = gp[:, -1]
    done = np.zeros(B, bool)
    out = dict(reached=np.zeros(B, bool), ticks=np.full(B, T, np.int32), path_length=np.zeros(B),
               min_person_dist=np.full(B, np.inf), intimate_ticks=np.zeros(B, np.int32),
               personal_ticks=np.zeros(B, np.int32), collision_ticks=np.zeros(B, np.int32),
               not_optimized_ticks=np.zeros(B, np.int32), cmd_variation=np.zeros(B))
    valid = np.arange(K)[None, :] < n_people[:, None]
    for k in range(T):
        if done.all():
            break
        poses, cmds3, n_steps = fl.trajectorize_batch(gp, pose)
        cmds = np.zeros((B, poses.shape[1], 2))
        cmds[:, : cmds3.shape[1]] = cmds3[:, :, [0, 2]]
        ppl = people0.copy()
        ppl[:, :, 0] += ppl[:, :, 2] * (k * dt)
        ppl[:, :, 1] += ppl[:, :, 3] * (k * dt)
        if K > 0:
            fp, fn = fl.filter_people_fov(ppl, n_people, pose, morg, W, H, res, costmap_index=cidx)
        else:
            fp, fn = np.zeros((B, fl.A, 5)), np.zeros(B, np.int32)
        n_poses = np.where(done, 0, n_steps + 1).astype(np.int32)
        r = fl.optimize_batch(poses, cmds, fp, fn, speed, cms, morg, res, od, costmap_index=cidx, n_poses=n_poses,
                              want_people_proj=False, inplace=True)
        act = ~done
        v, w = cmds[:, 0, 0], cmds[:, 0, 1]
        x, y, th = pose[:, 0], pose[:, 1], pose[:, 2]
        x1, y1 = x + (v * np.cos(th)) * dt, y + (v * np.sin(th)) * dt
        yaw1 = sc.yaw_roundtrip(th + w * dt)
        t1 = (k + 1) * dt
        dx = people0[:, :, 0] + people0[:, :, 2] * t1 - x1[:, None]
        dy = people0[:, :, 1] + people0[:, :, 3] * t1 - y1[:, None]
        dmin = np.where(valid, np.sqrt(dx * dx + dy * dy), np.inf).min(axis=1) if K > 0 else np.full(B, np.inf)
        ox, oy = morg[cidx, 0], morg[cidx, 1]
        inside = (x1 >= ox) & (y1 >= oy)
        mx = np.where(inside, (x1 - ox) / res, -1).astype(np.int64)
        my = np.where(inside, (y1 - oy) / res, -1).astype(np.int64)
        inside &= (mx < W) & (my < H)
        cost = np.where(inside, cms[cidx, np.clip(my, 0, H - 1), np.clip(mx, 0, W - 1)], 255)
        out["path_length"][act] += np.sqrt((x1 - x) ** 2 + (y1 - y) ** 2)[act]
        out["min_person_dist"][act] = np.minimum(out["min_person_dist"], dmin)[act]
        out["intimate_ticks"][act] += (dmin < 0.45)[act]
        out["personal_ticks"][act] += (dmin < 1.2)[act]
        out["collision_ticks"][act] += (cost >= 253)[act]
        out["not_optimized_ticks"][act] += (~r["optimized"])[act]
        if k >= 1:
            out["cmd_variation"][act] += (np.abs(v - speed[:, 0]) + np.abs(w - speed[:, 1]))[act]
        pose[act] = np.stack([x1, y1, yaw1], axis=1)[act]
        speed[act] = np.stack([v, w], axis=1)[act]
        arrived = act & (np.sqrt((x1 - goal[:, 0]) ** 2 + (y1 - goal[:, 1]) ** 2) <= goal_tolerance)
        out["reached"][arrived] = True
        out["ticks"][arrived] = k + 1
        done |= arrived
    return out


def summary(r):
    return {"reached_fraction": float(np.mean(r["reached"])), "mean_ticks": float(np.mean(r["ticks"])),
            "mean_path_length_m": float(np.mean(r["path_length"])),
            "min_person_dist_p05_m": float(np.percentile(r["min_person_dist"], 5)),
            "intimate_ticks_per_episode": float(np.mean(r["intimate_ticks"])),
            "personal_ticks_per_episode": float(np.mean(r["personal_ticks"])),
            "collision_ticks_per_episode": float(np.mean(r["collision_ticks"])),
            "episodes_with_collision": float(np.mean(r["collision_ticks"] > 0)),
            "not_optimized_share": float(np.sum(r["not_optimized_ticks"]) / max(1, np.sum(r["ticks"]))),
            "mean_cmd_variation": float(np.mean(r["cmd_variation"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,64,4096,16384")
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--people", type=int, default=20)
    ap.add_argument("--reps", type=int, default=2, help="timed runs per arm and size, alternating the arms")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_episodes.py needs a CUDA device")
    result = {"card": _card(), "ticks": a.ticks, "people": a.people, "agents": 3, "param_set": "soc_work_obst",
              "control_period_s": 0.05, "timing": "wall clock of the whole run, ending in a device synchronise",
              "sizes": {}}
    for B in [int(x) for x in a.sizes.split(",")]:
        s = sc.episodes(B, a.people, ticks=a.ticks)
        fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
        arms = {"episodes": lambda T: fl.run_episodes(ticks=T, **_args(s)),
                "host_loop": lambda T: host_loop(fl, s, T)}
        for name, fn in arms.items():  # warm-up: module loads, allocations of this shape
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
                           "runs_s": [round(t, 4) for t in times[name]], "outcome": summary(last[name])}
        e, h = last["episodes"], last["host_loop"]
        entry["speedup_episodes_over_host_loop"] = entry["host_loop"]["ms_per_tick"] / entry["episodes"]["ms_per_tick"]
        entry["arms_agree"] = {"same_reached": float(np.mean(e["reached"] == h["reached"])),
                               "same_ticks": float(np.mean(e["ticks"] == h["ticks"])),
                               "max_abs_path_length_diff_m": float(np.max(np.abs(e["path_length"] - h["path_length"])))}
        result["sizes"][str(B)] = entry
        print(json.dumps({str(B): entry}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
