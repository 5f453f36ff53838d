#!/usr/bin/env python
"""A/B of the people projection of two built trees of the package: FleetOptimizer.optimize_batch(...,
want_people_proj=True) on seeded episode scenes (scenarios.episodes: corridor, trajectorizer seed, the people of each
scene as the A columns), dumped by each tree's own package and libsmpc.so in a child process of its own and compared
bit for bit. Each tree generates the scenes with its own scenarios.episodes, which both must have unchanged. Writes one JSON (stdout and --out).
  python tools/ab_people_proj.py --tree-a OLD_CHECKOUT --tree-b . --out ab.json"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

CASES = [(4096, 3, 1), (4096, 20, 2), (1024, 50, 3)]  # (B, A, seed)


def dump(out_dir, tree):
    sys.path.insert(0, os.path.abspath(tree))
    from nav2_social_mpc_controller_b200 import scenarios as sc
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    import nav2_social_mpc_controller_b200 as pkg
    assert os.path.dirname(os.path.dirname(os.path.abspath(pkg.__file__))) == os.path.abspath(tree)
    for B, A, seed in CASES:
        s = sc.episodes(B, A, seed=seed, ticks=40)
        p = s["params"]
        poses, cmds = sc.pure_pursuit_seed(s["global_path"], s["pose"], p)
        fl = FleetOptimizer(p, n_robots=B, n_agents=A)
        r = fl.optimize_batch(poses, cmds, s["people"], np.full(B, A, np.int32), s["speed"], s["costmaps"],
                              s["costmap_origin"], s["costmap_resolution"], s["od"], costmap_index=s["costmap_index"],
                              want_people_proj=True)
        fl.close()
        np.save(os.path.join(out_dir, f"proj_B{B}_A{A}_s{seed}.npy"), r["people_proj"])
        np.save(os.path.join(out_dir, f"status_B{B}_A{A}_s{seed}.npy"), r["project_status"])


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
        for B, A, seed in CASES:
            f = f"B{B}_A{A}_s{seed}.npy"
            pa, pb = np.load(os.path.join(dirs["a"], "proj_" + f)), np.load(os.path.join(dirs["b"], "proj_" + f))
            sa, sb = np.load(os.path.join(dirs["a"], "status_" + f)), np.load(os.path.join(dirs["b"], "status_" + f))
            res["cases"].append({"B": B, "A": A, "seed": seed, "values": int(pa.size),
                                 "bit_identical": bool(pa.tobytes() == pb.tobytes() and np.array_equal(sa, sb)),
                                 "max_abs_diff": float(np.nanmax(np.abs(pa - pb))) if pa.size else 0.0,
                                 "projected_problems": int(np.sum(sa == 0))})
    res["all_bit_identical"] = all(c["bit_identical"] for c in res["cases"])
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
