#!/usr/bin/env python
"""A/B of the closed-loop episode entries of two built trees of the package: FleetOptimizer.run_episodes and
run_crowd_episodes with every log on seeded scenes (scenarios.episodes, scenarios.crowd_episodes), dumped by each
tree's own package and libsmpc.so in a child process of its own and compared bit for bit. Each tree generates the
scenes with its own scenarios, which both must have unchanged. Writes one JSON (stdout and --out).
  python tools/ab_episodes.py --tree-a OLD_CHECKOUT --tree-b . --out ab.json"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

# (entry, B, K, seed, ticks, substeps)
CASES = [("episodes", 1024, 20, 1, 100, 0), ("crowd", 1024, 20, 2, 100, 1), ("crowd", 256, 9, 3, 120, 4),
         ("crowd", 64, 0, 4, 60, 1)]
OUTPUTS = ("reached", "ticks", "path_length", "min_person_dist", "intimate_ticks", "personal_ticks",
           "collision_ticks", "not_optimized_ticks", "cmd_variation", "pose_log", "cmd_log", "optimized_log",
           "people_disturbance", "people_log")


def _name(case):
    return "{}_B{}_K{}_s{}_T{}_n{}".format(*case)


def dump(out_dir, tree):
    sys.path.insert(0, os.path.abspath(tree))
    from nav2_social_mpc_controller_b200 import scenarios as sc
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    import nav2_social_mpc_controller_b200 as pkg
    assert os.path.dirname(os.path.dirname(os.path.abspath(pkg.__file__))) == os.path.abspath(tree)
    for case in CASES:
        entry, B, K, seed, T, substeps = case
        s = sc.episodes(B, K, seed=seed, ticks=T) if entry == "episodes" else \
            sc.crowd_episodes(B, K, seed=seed, ticks=T, substeps=substeps)
        args = {k: v for k, v in s.items() if k not in ("params", "ticks")}
        fl = FleetOptimizer(s["params"], n_robots=B, n_agents=3)
        fn = fl.run_episodes if entry == "episodes" else fl.run_crowd_episodes
        r = fn(ticks=T, want_logs=True, **args)
        fl.close()
        for k in OUTPUTS:
            if k in r:
                np.save(os.path.join(out_dir, f"{_name(case)}__{k}.npy"), np.asarray(r[k]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree-a")
    ap.add_argument("--tree-b")
    ap.add_argument("--dump", help=argparse.SUPPRESS)
    ap.add_argument("--tree", help=argparse.SUPPRESS)
    ap.add_argument("--out")
    a = ap.parse_args()
    if a.dump:
        dump(a.dump, a.tree)
        return
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from tools.bench_episodes import _card
    res = {"card": _card(), "cases": []}
    with tempfile.TemporaryDirectory() as tmp:
        dirs = {}
        for name, tree in (("a", a.tree_a), ("b", a.tree_b)):
            d = os.path.join(tmp, name)
            os.makedirs(d)
            env = {k: v for k, v in os.environ.items() if k != "SMPC_LIB_PATH"}
            subprocess.run([sys.executable, os.path.abspath(__file__), "--dump", d, "--tree", tree], check=True,
                           env=env)
            dirs[name] = d
        for case in CASES:
            files = sorted(f for f in os.listdir(dirs["a"]) if f.startswith(_name(case) + "__"))
            assert files == sorted(f for f in os.listdir(dirs["b"]) if f.startswith(_name(case) + "__"))
            same = {}
            for f in files:
                x, y = np.load(os.path.join(dirs["a"], f)), np.load(os.path.join(dirs["b"], f))
                same[f.split("__")[1][:-4]] = bool(x.dtype == y.dtype and x.shape == y.shape and
                                                   x.tobytes() == y.tobytes())
            res["cases"].append({"case": _name(case), "outputs": len(files), "bit_identical": all(same.values()),
                                 "differing": [k for k, v in same.items() if not v]})
    res["all_bit_identical"] = all(c["bit_identical"] for c in res["cases"])
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
