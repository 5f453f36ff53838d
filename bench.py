#!/usr/bin/env python
"""bench.py — MPC solves/sec of the batched social-MPC solver on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--legs all|none]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path (the whole bounded TR-LM solve of every problem) over one batch of synthetic
scenarios. Headline workload = BASELINE.json configs[2], the configuration the north star is quoted on ("full
social-MPC solves"): soc_work_obst parameters, 65536 crowd scenarios, 20 agents. Under torchrun every rank solves its
own 65536 scenarios (weak scaling, no collective on the solve path); the time is the max over ranks.

  value      solves/s with the batch already resident in HBM (CUDA events on the launching stream)
  e2e        solves/s through the host-buffer C-ABI call smpc_solve_batch: pinned host inputs, H2D, kernels, D2H
  roofline   FP64 CUDA-core roofline of the solve kernel (SURVEY §8d: the path is FP64-instruction bound, not HBM
             or tensor bound); the HBM side is reported next to it
  cpu_baseline / parity_vs_oracle   the CPU oracle (Ceres-algorithm restatement; Ceres itself is not installable
             here) on all host cores over a bounded sample of the same workload, and the GPU results checked against it
             (rank 0, at every N)
  legs       the other BASELINE configs measured in the same run: configs[1] obst_only x4096, configs[3] multi-start
             256 x 1024 sharded by robot with the per-robot arg-min and the host gather inside the timed region,
             configs[4] 10^6 problems x 50 agents STRONG scaling (10^6 / N per rank) with the final host gather, in the
             reference's unicycle model and in the omnidirectional extension,
             configs[0] single-solve latency
--impl reference times only the CPU restatement (the reference's own code needs Ceres + ROS and cannot build here).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from nav2_social_mpc_controller_b200 import abi, scenarios as sc  # noqa: E402

METRIC = "mpc_solves_per_sec"
UNIT = "solves/s"
HEADLINE = "soc_work_obst_x65536_A20"

WORKLOADS = {
    # name: (builder, description, unique costmap per problem)
    "obst_only_x4096": (lambda: sc.corridor(B=4096), "BASELINE configs[1]: obst_only params, 4096 corridor scenarios, "
                        "S=28, P=6, one 80x80 costmap per problem", True),
    "soc_work_obst_x65536_A20": (lambda: sc.crowd(B=65536, A=20), "BASELINE configs[2]: soc_work_obst params (full "
                                 "social + proxemics + obstacle critics), 65536 crowd scenarios, 20 agents, S=28, P=6, "
                                 "256 shared costmaps", False),
    "soc_work_obst_x16384_A3": (lambda: sc.crowd(B=16384, A=3, config_id=6), "soc_work_obst params, 16384 crowd "
                                "scenarios with the reference's 3 agents, S=28, P=6", False),
    "obst_only_x65536": (lambda: sc.corridor(B=65536, unique_maps=False, config_id=22), "obst_only params, 65536 corridor "
                         "scenarios, 256 shared costmaps (throughput-mode check)", False),
    "soc_work_obst_x65536_A3": (lambda: sc.crowd(B=65536, A=3, config_id=23), "soc_work_obst params, 65536 crowd "
                                "scenarios with the reference's 3 agents", False),
    "multistart_256x1024": (lambda: sc.multistart(256, 1024), "BASELINE configs[3]: 1024 perturbed starts x 256 robots, "
                            "A=3, per-robot arg-min", False),
    "crowd_x16384_A50": (lambda: sc.crowd(B=16384, A=50, config_id=5), "BASELINE configs[4] slice: 16384 problems, "
                         "50 agents, S=28, P=6 (a 1.1 GB slice of one GPU's shard of the 10^6 sweep)", False),
}
# Workloads whose device batch is larger than the generated one: the unique scenarios are tiled on the device up to
# this many problems IN TOTAL over all ranks (strong scaling: each rank takes total / world). 10^6 problems at A = 50
# are 70 GB of agent trajectories: resident in one B200's HBM, never materialised on the host.
TILED_TOTAL = {"crowd_x1M_A50": 1_000_000}
WORKLOADS["crowd_x1M_A50"] = (lambda: sc.crowd(B=16384, A=50, config_id=5), "BASELINE configs[4] (unicycle): 10^6 "
                              "problems, 50 agents, S=28, P=6 = 16384 unique crowd scenarios tiled on the device "
                              "(70 GB of agent trajectories resident in HBM); e2e and CPU arms use the unique 16384",
                              False)
# bounded CPU samples: roughly 10-30 s of single-core oracle work each (a solve costs ~7 ms without people,
# ~15 ms at A = 3, ~40 ms at A = 20, ~100 ms at A = 50)
CPU_SAMPLE = {"obst_only_x4096": 3072, "obst_only_x65536": 3072, "soc_work_obst_x16384_A3": 1536,
              "soc_work_obst_x65536_A3": 1536, "multistart_256x1024": 1536, "soc_work_obst_x65536_A20": 1024,
              "crowd_x16384_A50": 256, "crowd_x1M_A50": 256}
WANT = ("u", "cmds", "cost_initial", "cost_final", "iterations", "termination", "usable", "n_evals")
DUMP_BYTES = 60_000_000  # --dump-outputs: array data per directory, so that the files stay under 64 MB in all


def dump_outputs(path, outputs):
    """--dump-outputs: write every output of the timed path's last step (one row per problem) as PATH/<name>.npy in
    float64; integer outputs widen exactly. The inputs are seeded, so two builds run with the same arguments can be
    compared file by file. When all rows exceed DUMP_BYTES, every file holds the same fixed, seeded sample of rows, and
    PATH/problem_index.npy lists which."""
    n = len(next(iter(outputs.values())))
    row_bytes = sum(8 * (v.size // n) for v in outputs.values())
    rows = None
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))
    os.makedirs(path, exist_ok=True)
    for name, v in outputs.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(v if rows is None else v[rows], dtype=np.float64))
    if rows is not None:
        np.save(os.path.join(path, "problem_index.npy"), rows.astype(np.float64))


def flops_per_solve(S, P, A_eff, m, n_full, n_light, iters):
    """SURVEY §8d algorithmic FLOPs: F_solve = n_full F_jac + n_light F_grad + K F_lin. The per-agent term is 410 instead
    of SURVEY's a-priori 810: the social pair function is odd, so the minimal algorithm needs ONE pair interaction
    (~400 FLOPs with its 2x4 Jacobian) per agent and step, not two (DESIGN.md §3). n_full = evaluations that build
    J^T J, n_light = line-search samples that stop at cost + J^T r (F_grad = F_jac without the J^T J accumulation)."""
    f_res = S * (224 + 29 * P + 410 * A_eff)
    f_jac = f_res + 2 * m * (P * (P + 1) / 2 + P)
    f_grad = f_res + 2 * m * P
    f_lin = P ** 3 / 3 + 2 * P ** 2 + 4 * P
    return n_full * f_jac + n_light * f_grad + iters * f_lin


def n_residuals(batch):
    ch, bl, nb, nbd = batch.dims
    per_step = 8 if batch.arrays["has_people"].any() else 5
    return per_step * batch.n_steps + max(nbd - 1, 0)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed regions (B200_PROFILING.md recipe): one long-running
    `nvidia-smi -lms 50` process, every line time-stamped; summary() keeps the samples inside the marked windows."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.windows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append((time.perf_counter(), parts))
        except Exception:
            pass

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self):
        inside = [p for (t, p) in self.samples if any(a <= t <= b for a, b in self.windows)]
        used = inside if inside else [p for _, p in self.samples]
        if not used:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(x[0]) for x in used if x[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(x[3 + i].lower().startswith("active") for x in used)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(used[0][1]), "reasons": reasons,
                "samples_in_timed_regions": len(inside), "samples_total": len(self.samples)}


def load_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of the solve kernel, per launch, from the committed
    `ncu --set full` capture of this workload (profiles/r02_traffic.json); None when no capture exists."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                t = json.load(f).get(workload)
            if t:
                return dict(t, source=f"profiles/{name}")
    return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def parity_block(got, ref, n):
    us = ref["usable"][:n].astype(bool)
    du = np.abs(got["u"][:n] - ref["u"][:n]).reshape(n, -1).max(axis=1)
    dc = np.abs(got["cost_final"][:n] - ref["cost_final"][:n]) / np.maximum(np.abs(ref["cost_final"][:n]), 1e-300)
    ok = (~us & (got["usable"][:n] == 0)) | (us & (got["usable"][:n] == 1) & (du <= 1e-6) & (dc <= 1e-8))
    return {"problems": int(n), "within_1e-6_u_and_1e-8_cost": float(ok.mean()),
            "same_termination": float((got["termination"][:n] == ref["termination"][:n]).mean()),
            "same_iteration_count": float((got["iterations"][:n] == ref["iterations"][:n]).mean()),
            "max_du": float(du[us].max()) if us.any() else None,
            "max_rel_dcost": float(dc[us].max()) if us.any() else None,
            "note": "misses are iterate-path flips at decision thresholds: per-problem evidence in "
                    "profiles/r02_flip_log_*.json (tools/flip_log.py)"}


def cpu_baseline(batch, workload, threads):
    from tests import oracle_lib
    o = oracle_lib.load()
    n = min(CPU_SAMPLE.get(workload, 256), batch.n_problems)
    sub = batch.slice(0, n)
    t0 = time.perf_counter()
    out = o.solve_batch(sub, n_threads=threads, want=("u", "cost_final", "usable", "iterations", "termination"))
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"first {n} problems of {workload}, {threads} host threads, {dt:.2f} s wall; "
                      "oracle = Ceres-algorithm restatement built -O3 -ffp-contract=off without -march "
                      "(the reference's own flags; Ceres/ROS not installable here)"}, out, sub


def run_reference(args, rank, world):
    """--impl reference: the reference algorithm on the box's host cores (oracle port; rank 0 only)."""
    if rank != 0:
        return
    from tests import oracle_lib
    o = oracle_lib.load()
    builder, desc, _ = WORKLOADS[args.workload]
    batch = builder()
    threads = os.cpu_count() or 1
    n = min(CPU_SAMPLE.get(args.workload, 256), batch.n_problems)
    sub = batch.slice(0, n)
    want = ("u", "cost_final", "usable")
    for _ in range(args.warmup):
        o.solve_batch(sub.slice(0, min(n, 4 * threads)), n_threads=threads, want=want)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        out = o.solve_batch(sub, n_threads=threads, want=want)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    total = sum(times)
    value = n * args.steps / total
    sample = (f"each step = first {n} problems of {args.workload} on {threads} host threads "
              "(CPU oracle: Ceres-algorithm restatement with per-residual Jet<4> re-rollouts)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "description": desc, "problems_per_step": n},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


class Ctx:
    """Per-process benchmark context: device, stream, L2-flush buffer, distributed helpers."""

    def __init__(self, rank, local_rank, world):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.local_rank, self.world = rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.gloo = None
        if world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.gloo = dist.new_group(backend="gloo")  # host-side gathers of result tables (not on the solve path)
        self.stream = torch.cuda.Stream(device=self.dev)  # non-default stream: kernels and events share it
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
        self.tdt = {np.float64: torch.float64, np.int32: torch.int32, np.uint8: torch.uint8}

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def host_barrier(self):
        """Barrier on the gloo group: the waiting ranks sleep on the host. (An NCCL barrier keeps a spinning kernel on
        every waiting rank's GPU, and kernels of two PROCESSES time-slice a GPU: rank 0 driving all GPUs through the
        library would then get half of each.)"""
        if self.world > 1:
            self.torch.cuda.synchronize()
            self.dist.barrier(group=self.gloo)

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return vals
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return tuple(float(v) for v in t)

    def gather_host(self, arr: np.ndarray):
        """Concatenate per-rank host arrays on rank 0 (gloo; the 'final host gather' of the north star)."""
        if self.world == 1:
            return arr
        t = self.torch.from_numpy(np.ascontiguousarray(arr))
        parts = [self.torch.empty_like(t) for _ in range(self.world)] if self.rank == 0 else None
        self.dist.gather(t, parts, dst=0, group=self.gloo)
        return np.concatenate([p.numpy() for p in parts], axis=0) if self.rank == 0 else None


def device_batch(ctx, batch, B, tiled_total=None):
    """Device-resident copy of a host batch; with tiled_total the unique scenarios are tiled to B problems per rank."""
    torch = ctx.torch
    host_pinned = {k: (torch.from_numpy(v).pin_memory() if v is not None else None) for k, v in batch.arrays.items()}
    dev_arrays = {k: (t.to(ctx.dev, non_blocking=True) if t is not None else None) for k, t in host_pinned.items()}
    if tiled_total is not None:
        from nav2_social_mpc_controller_b200.sharding import tiled_source_index
        Bu = batch.n_problems
        src = torch.from_numpy(tiled_source_index(tiled_total, Bu, ctx.world, ctx.rank)).to(ctx.dev)
        for k, t in list(dev_arrays.items()):
            if t is None or k in ("costmaps", "costmap_origin"):
                continue
            big = torch.empty((B,) + tuple(t.shape[1:]), dtype=t.dtype, device=ctx.dev)
            for lo in range(0, B, Bu):  # gather piecewise: index_select on the whole batch would double the 70 GB
                n = min(Bu, B - lo)
                torch.index_select(t, 0, src[lo:lo + n], out=big[lo:lo + n])
            dev_arrays[k] = big
        del src
    torch.cuda.synchronize()
    return host_pinned, dev_arrays


def time_device(ctx, opt, dstruct, dev_out, steps, warmup, extra=None):
    """W warm-up + K timed device-resident solves; L2 flushed between steps; CUDA events on the launching stream."""
    torch = ctx.torch

    def step():
        opt.solve_batch_device(dstruct, dev_out, stream=ctx.stream.cuda_stream)
        if extra is not None:
            extra()

    with torch.cuda.stream(ctx.stream):
        for _ in range(warmup):
            step()
    torch.cuda.synchronize()
    ctx.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    launches0 = opt.launch_count()
    t0 = time.perf_counter()
    with torch.cuda.stream(ctx.stream):
        for s in range(steps):
            ctx.flush.fill_(s & 0xFF)  # L2 flush between timed iterations (outside the event pair)
            ev[s][0].record(ctx.stream)
            step()
            ev[s][1].record(ctx.stream)
    torch.cuda.synchronize()
    window = (t0, time.perf_counter())
    return [a.elapsed_time(b) for a, b in ev], opt.launch_count() - launches0, window


def time_e2e(ctx, fn, steps, warmup):
    """W warm-up + K timed host-buffer calls (wall clock around the call, which returns with the results on the host)."""
    for _ in range(warmup):
        fn()
    ctx.barrier()
    ts = []
    t_region0 = time.perf_counter()
    for s in range(steps):
        ctx.flush.fill_(s & 0xFF)
        ctx.torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts, (t_region0, time.perf_counter())


def measure(ctx, name, steps, warmup, sampler=None, with_cpu=False, threads=1, dump_dir=None):
    """Device-resident + end-to-end measurement of one workload on this rank. Returns a dict of raw pieces. With
    dump_dir, rank 0 writes the device-resident outputs of the last timed step there (dump_outputs)."""
    from nav2_social_mpc_controller_b200.optimizer import Optimizer
    torch = ctx.torch
    builder, desc, unique_map = WORKLOADS[name]
    batch = builder()
    if ctx.world > 1 and name not in TILED_TOTAL:  # weak scaling: every rank gets its own scenarios of the same shape
        rng = np.random.default_rng(1000 + ctx.rank)
        perm = rng.permutation(batch.n_problems)
        for k, v in batch.arrays.items():
            if v is not None and k not in ("costmaps", "costmap_origin"):
                batch.arrays[k] = np.ascontiguousarray(v[perm])
    Bu, S, A = batch.n_problems, batch.n_steps, batch.n_agents
    tiled = name in TILED_TOTAL
    B = TILED_TOTAL[name] // ctx.world if tiled else Bu
    nb = batch.dims[2]
    opt = Optimizer(ctx.local_rank)
    opt.initialize(batch.params)
    host_pinned, dev_arrays = device_batch(ctx, batch, B, TILED_TOTAL.get(name))
    shapes = abi.result_shapes(B, S, nb)
    dev_out = {k: torch.zeros(shapes[k][0], dtype=ctx.tdt[shapes[k][1]], device=ctx.dev) for k in WANT}
    dstruct = abi.make_batch_struct(dev_arrays, B, S, A, batch.n_costmaps, batch.size_x, batch.size_y,
                                    batch.resolution, batch.dt)
    step_ms, launches, win = time_device(ctx, opt, dstruct, dev_out, steps, warmup)
    if sampler:
        sampler.mark(*win)
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, {k: t.cpu().numpy() for k, t in dev_out.items()})
    # end to end: host-buffer C-ABI call, pinned host memory, H2D + kernels + D2H every step (the unique scenarios)
    host_np = {k: (t.numpy() if t is not None else None) for k, t in host_pinned.items()}
    hshapes = abi.result_shapes(Bu, S, nb)
    host_out_t = {k: torch.zeros(hshapes[k][0], dtype=ctx.tdt[hshapes[k][1]]).pin_memory() for k in WANT}
    host_out = {k: t.numpy() for k, t in host_out_t.items()}
    hbatch = sc.Batch(params=batch.params, n_problems=Bu, n_steps=S, n_agents=A, n_costmaps=batch.n_costmaps,
                      size_x=batch.size_x, size_y=batch.size_y, resolution=batch.resolution, dt=batch.dt, arrays=host_np)
    e2e_t, win = time_e2e(ctx, lambda: opt.solve_batch(hbatch, out=host_out), steps, warmup)
    if sampler:
        sampler.mark(*win)
    # the timed device run and the e2e run see the same inputs -> identical results
    dev_u = dev_out["u"][:Bu].cpu().numpy()
    if tiled and (ctx.rank * B) % Bu:
        dev_u = None  # this rank's device batch starts at another unique scenario
    if dev_u is not None and not np.array_equal(dev_u, host_out["u"]):
        raise SystemExit(f"{name}: device-resident and host-buffer solves disagree")
    res = dict(name=name, desc=desc, unique_map=unique_map, batch=batch, hbatch=hbatch, B=B, Bu=Bu, S=S, A=A, nb=nb,
               step_ms=step_ms, launches=launches, e2e_t=e2e_t, dev_out=dev_out, host_out=host_out, opt=opt,
               h2d=int(sum(v.nbytes for v in host_np.values() if v is not None)),
               d2h=int(sum(v.nbytes for v in host_out.values())), tiled=tiled)
    if with_cpu and ctx.rank == 0:
        cb, ref_out, sub = cpu_baseline(hbatch, name, threads)
        res["cpu_baseline"] = cb
        res["parity"] = parity_block(host_out, ref_out, sub.n_problems)
    return res


def roofline_block(ctx, res, k_ms):
    batch, S, A, nb = res["batch"], res["S"], res["A"], res["nb"]
    P = batch.dof * nb
    n_evals = res["dev_out"]["n_evals"].cpu().numpy().astype(np.float64)
    iters = res["dev_out"]["iterations"].cpu().numpy().astype(np.float64)
    term = res["dev_out"]["termination"].cpu().numpy()
    A_eff = A if batch.arrays["has_people"].any() else 0
    flops = float(sum(flops_per_solve(S, P, A_eff, n_residuals(batch), n_evals[:, 0], n_evals[:, 1], iters)))
    peaks, peak_kind = load_peaks()
    fp64_peak = res["opt"].measure_fp64_peak()
    achieved = flops / (k_ms * 1e-3) / 1e12
    alg_bytes = res["B"] * batch.algorithmic_bytes_per_problem(res["unique_map"])
    if not res["unique_map"]:
        alg_bytes += batch.n_costmaps * batch.size_x * batch.size_y
    tr = load_traffic(res["name"])
    roof = {"bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": achieved / fp64_peak if fp64_peak > 0 else None,
            "traffic": (tr or {}).get("bytes"), "traffic_detail": tr,
            "kernel": f"smpc_solve_kernel<{nb}>", "kernel_ms": k_ms,
            "peak_source": "DFMA microbenchmark measured in this run (smpc_measure_fp64_peak); "
                           "MEASURED_PEAKS.json has no FP64 entry",
            "algorithmic_flops_per_launch": flops,
            "hbm": {"achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                    "algorithmic_bytes_per_launch": int(alg_bytes), "peak_source": peak_kind}}
    solver = {"mean_iterations": float(iters.mean()), "mean_evaluations_with_JtJ": float(n_evals[:, 0].mean()),
              "mean_evaluations_gradient_only": float(n_evals[:, 1].mean()),
              "termination_histogram": {abi.TERMINATION_NAMES[int(k)]: int(v) for k, v in
                                        zip(*np.unique(term, return_counts=True))},
              "usable_fraction": float(res["dev_out"]["usable"].float().mean()),
              "ceres_compat": int(batch.params.ceres_compat)}
    return roof, solver


def leg_simple(ctx, name, steps, warmup):
    """A secondary workload: device-resident + e2e throughput, weak scaling like the headline."""
    res = measure(ctx, name, steps, warmup)
    tot_ms, tot_e2e = ctx.max_over_ranks(float(sum(res["step_ms"])), float(sum(res["e2e_t"])))
    out = None
    if ctx.rank == 0:
        roof, solver = roofline_block(ctx, res, tot_ms / steps)
        out = {"workload": name, "description": res["desc"], "scaling": "weak",
               "value": ctx.world * res["B"] * steps / (tot_ms * 1e-3), "unit": UNIT, "ms_per_step": tot_ms / steps,
               "e2e": {"value": ctx.world * res["Bu"] * steps / tot_e2e, "unit": UNIT, "ms_per_step": 1e3 * tot_e2e / steps,
                       "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"]},
               "steps": steps, "warmup": warmup, "roofline_frac": roof["frac"], "solver": solver}
    res["opt"].close()
    return out


def leg_multistart(ctx, steps, warmup, n_robots=256, n_starts=1024):
    """BASELINE configs[3]: multi-start MPC sharded BY ROBOT (n_robots / N robots per rank, so a robot's arg-min never
    crosses a rank). The timed region holds the solve, the per-robot arg-min kernel and the final host gather."""
    from nav2_social_mpc_controller_b200.optimizer import Optimizer
    from nav2_social_mpc_controller_b200.sharding import shard_bounds
    torch = ctx.torch
    # scenario sharing (smpc_batch.scenario_index): the scene of a robot is ONE row of the input arrays, read by its
    # 1024 starts; only the start controls u0 and the row index are per problem
    full = sc.multistart(n_robots, n_starts, shared=True)
    lo, hi = shard_bounds(full.n_problems, ctx.world, ctx.rank, granule=n_starts)
    batch = full.slice(lo, hi)
    R = (hi - lo) // n_starts
    B, S, A, nb = batch.n_problems, batch.n_steps, batch.n_agents, batch.dims[2]
    opt = Optimizer(ctx.local_rank)
    opt.initialize(batch.params)
    host_pinned, dev_arrays = device_batch(ctx, batch, B)
    shapes = abi.result_shapes(B, S, nb)
    want = ("u", "cost_final", "usable", "iterations", "termination", "n_evals")
    dev_out = {k: torch.zeros(shapes[k][0], dtype=ctx.tdt[shapes[k][1]], device=ctx.dev) for k in want}
    best_index = torch.empty(R, dtype=torch.int32, device=ctx.dev)
    best_cost = torch.empty(R, dtype=torch.float64, device=ctx.dev)
    best_u = torch.empty(R, nb, 2, dtype=torch.float64, device=ctx.dev)
    dstruct = abi.make_batch_struct(dev_arrays, B, S, A, batch.n_costmaps, batch.size_x, batch.size_y,
                                    batch.resolution, batch.dt)

    def argmin():
        opt.multistart_argmin_device(R, n_starts, nb, dev_out["cost_final"], dev_out["usable"], dev_out["u"], best_index,
                                     best_cost, best_u, stream=ctx.stream.cuda_stream)

    step_ms, launches, _ = time_device(ctx, opt, dstruct, dev_out, steps, warmup, extra=argmin)
    # end to end: pinned host inputs -> H2D -> solve -> arg-min on the device -> winners D2H -> gather on rank 0
    host_np = {k: (t.numpy() if t is not None else None) for k, t in host_pinned.items()}
    pin = {k: torch.zeros_like(v, device="cpu").pin_memory() for k, v in
           dict(best_index=best_index, best_cost=best_cost, best_u=best_u).items()}
    gathered = {}

    def e2e():
        with torch.cuda.stream(ctx.stream):
            for k, t in host_pinned.items():
                if t is not None:
                    dev_arrays[k].copy_(t, non_blocking=True)
            opt.solve_batch_device(dstruct, dev_out, stream=ctx.stream.cuda_stream)
            argmin()
            pin["best_index"].copy_(best_index, non_blocking=True)
            pin["best_cost"].copy_(best_cost, non_blocking=True)
            pin["best_u"].copy_(best_u, non_blocking=True)
        ctx.stream.synchronize()
        gathered["index"] = ctx.gather_host(pin["best_index"].numpy() + lo)
        gathered["cost"] = ctx.gather_host(pin["best_cost"].numpy())
        gathered["u"] = ctx.gather_host(pin["best_u"].numpy())

    e2e_t, _ = time_e2e(ctx, e2e, steps, warmup)
    tot_ms, tot_e2e = ctx.max_over_ranks(float(sum(step_ms)), float(sum(e2e_t)))
    out = None
    if ctx.rank == 0:
        # check the winners against a host arg-min of rank 0's own shard
        cf = dev_out["cost_final"].cpu().numpy().reshape(R, n_starts)
        us = dev_out["usable"].cpu().numpy().reshape(R, n_starts).astype(bool)
        want_idx = np.where(us, cf, np.inf).argmin(axis=1) + np.arange(R) * n_starts + lo
        ok = bool(np.array_equal(gathered["index"][:R], want_idx)) and gathered["index"].shape[0] == n_robots
        out = {"workload": "multistart_256x1024", "description": WORKLOADS["multistart_256x1024"][1],
               "scaling": "strong", "sharding": f"by robot: {R} robots x {n_starts} starts per rank",
               "inputs": "scenario sharing: one scene row per robot + per-start u0 (smpc_batch.scenario_index)",
               "value": full.n_problems * steps / (tot_ms * 1e-3), "unit": UNIT, "ms_per_step": tot_ms / steps,
               "robots_per_sec": n_robots * steps / (tot_ms * 1e-3),
               "timed_region": "solve kernel + per-robot arg-min kernel (CUDA events, max over ranks)",
               "e2e": {"value": full.n_problems * steps / tot_e2e, "unit": UNIT, "ms_per_step": 1e3 * tot_e2e / steps,
                       "robots_per_sec": n_robots * steps / tot_e2e,
                       "h2d_bytes_per_step": int(sum(v.nbytes for v in host_np.values() if v is not None)) * ctx.world,
                       "d2h_bytes_per_step": int(sum(t.numel() * t.element_size() for t in pin.values())) * ctx.world,
                       "how": "pinned host inputs H2D + solve + arg-min + winners D2H + gloo gather to rank 0, wall clock"},
               "argmin_matches_host": ok, "steps": steps, "warmup": warmup,
               "winner_cost_mean": float(np.mean(gathered["cost"][np.isfinite(gathered["cost"])]))}
    opt.close()
    return out


def leg_scaling_sweep(ctx, steps, warmup, name="crowd_x1M_A50", omni=False):
    """BASELINE configs[4]: 10^6 problems x 50 agents, STRONG scaling: every rank solves 10^6 / N problems (inputs
    resident in HBM: 70 GB of agent trajectories cannot come from the host every step), then the result table
    (u, cost_final, iterations, termination, usable) goes D2H and is gathered on rank 0: the north star's 'final host
    gather' is inside value_with_gather."""
    from nav2_social_mpc_controller_b200.optimizer import Optimizer
    torch = ctx.torch
    builder, desc, _ = WORKLOADS[name]
    batch = builder()
    if omni:  # (vx, vy, w) blocks: the extension of BASELINE configs[4]; no reference solve exists for it
        batch = sc.omni(batch)
        desc = desc.replace("(unicycle)", "(OMNIDIRECTIONAL blocks vx, vy, w: extension, checked against this repo's "
                            "own oracle functors only — the reference has no omnidirectional solve)")
    total = TILED_TOTAL[name]
    B = total // ctx.world
    S, A, nb = batch.n_steps, batch.n_agents, batch.dims[2]
    opt = Optimizer(ctx.local_rank)
    opt.initialize(batch.params)
    _, dev_arrays = device_batch(ctx, batch, B, total)
    shapes = abi.result_shapes(B, S, nb, batch.dof)
    want = ("u", "cost_final", "iterations", "termination", "usable", "n_evals")
    dev_out = {k: torch.zeros(shapes[k][0], dtype=ctx.tdt[shapes[k][1]], device=ctx.dev) for k in want}
    dstruct = abi.make_batch_struct(dev_arrays, B, S, A, batch.n_costmaps, batch.size_x, batch.size_y,
                                    batch.resolution, batch.dt)
    step_ms, launches, _ = time_device(ctx, opt, dstruct, dev_out, steps, warmup)
    pin = {k: torch.zeros_like(dev_out[k], device="cpu").pin_memory() for k in ("u", "cost_final", "iterations",
                                                                                "termination", "usable")}
    got = {}

    def with_gather():
        with torch.cuda.stream(ctx.stream):
            opt.solve_batch_device(dstruct, dev_out, stream=ctx.stream.cuda_stream)
            for k, t in pin.items():
                t.copy_(dev_out[k], non_blocking=True)
        ctx.stream.synchronize()
        for k, t in pin.items():
            got[k] = ctx.gather_host(t.numpy())

    g_t, _ = time_e2e(ctx, with_gather, steps, 1)
    tot_ms, tot_g = ctx.max_over_ranks(float(sum(step_ms)), float(sum(g_t)))
    out = None
    if ctx.rank == 0:
        res = dict(batch=batch, S=S, A=A, nb=nb, dev_out=dev_out, opt=opt, B=B, unique_map=False, name=name)
        roof, solver = roofline_block(ctx, res, tot_ms / steps)
        # parity of a prefix of the unique scenarios against the oracle (rank 0's shard starts at unique scenario 0)
        from tests import oracle_lib
        n = min(CPU_SAMPLE[name], batch.n_problems)
        ref = oracle_lib.load().solve_batch(batch.slice(0, n), n_threads=os.cpu_count() or 1,
                                            want=("u", "cost_final", "usable", "iterations", "termination"))
        mine = {k: got[k][:n] for k in ("u", "cost_final", "usable", "iterations", "termination")}
        out = {"workload": name, "description": desc, "scaling": "strong", "problems_total": total,
               "problems_per_gpu": B, "model": "omnidirectional" if omni else "unicycle",
               "value": total * steps / (tot_ms * 1e-3), "unit": UNIT,
               "ms_per_step": tot_ms / steps,
               "value_with_gather": total * steps / tot_g, "ms_per_step_with_gather": 1e3 * tot_g / steps,
               "gathered_bytes_per_step": int(sum(t.numel() * t.element_size() for t in pin.values())) * ctx.world,
               "gather": "per-rank D2H of the result table into pinned memory + gloo gather to rank 0 (wall clock)",
               "gathered_rows": int(got["cost_final"].shape[0]), "steps": steps, "warmup": warmup,
               "roofline_frac": roof["frac"], "solver": solver, "parity_vs_oracle": parity_block(mine, ref, n)}
    opt.close()
    del dev_arrays, dev_out
    torch.cuda.empty_cache()
    return out


def leg_library_multi(ctx, steps, warmup, per_gpu=16384, A=20):
    """SURVEY §8e through the LIBRARY: smpc_solve_batch_multi — one process (rank 0), one host thread + handle per GPU,
    contiguous shards of one pinned host batch, results gathered into one pinned host table by the shards' own D2H
    copies. The other ranks idle at a barrier while rank 0 drives all N GPUs."""
    from nav2_social_mpc_controller_b200.optimizer import MultiGpuOptimizer
    torch = ctx.torch
    ctx.host_barrier()
    out = None
    if ctx.rank == 0:
        base = sc.crowd(B=per_gpu, A=A)
        n = per_gpu * ctx.world
        arr = {}
        for k, v in base.arrays.items():
            if v is None or k in ("costmaps", "costmap_origin"):
                arr[k] = v
            else:
                arr[k] = np.ascontiguousarray(np.tile(v, (ctx.world,) + (1,) * (v.ndim - 1)))
        pinned = {k: (torch.from_numpy(v).pin_memory() if v is not None else None) for k, v in arr.items()}
        host_np = {k: (t.numpy() if t is not None else None) for k, t in pinned.items()}
        batch = sc.Batch(params=base.params, n_problems=n, n_steps=base.n_steps, n_agents=A, n_costmaps=base.n_costmaps,
                         size_x=base.size_x, size_y=base.size_y, resolution=base.resolution, dt=base.dt, arrays=host_np)
        shapes = abi.result_shapes(n, base.n_steps, base.dims[2])
        host_out_t = {k: torch.zeros(shapes[k][0], dtype=ctx.tdt[shapes[k][1]]).pin_memory() for k in WANT}
        host_out = {k: t.numpy() for k, t in host_out_t.items()}
        multi = MultiGpuOptimizer(base.params, list(range(ctx.world)))
        for _ in range(warmup):
            multi.solve_batch(batch, out=host_out)
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            multi.solve_batch(batch, out=host_out)
            ts.append(time.perf_counter() - t0)
        multi.close()
        same = all(np.array_equal(host_out["u"][:per_gpu], host_out["u"][r * per_gpu:(r + 1) * per_gpu])
                   for r in range(ctx.world))
        out = {"workload": f"soc_work_obst A={A}, {per_gpu} problems per GPU, one host batch of {n}",
               "entry": "smpc_solve_batch_multi (one process, one host thread + handle per GPU, pinned host buffers)",
               "n_gpus": ctx.world, "value": n * steps / sum(ts), "unit": UNIT, "ms_per_step": 1e3 * sum(ts) / steps,
               "h2d_bytes_per_step": int(sum(v.nbytes for v in host_np.values() if v is not None)),
               "d2h_bytes_per_step": int(sum(v.nbytes for v in host_out.values())),
               "shards_identical": bool(same), "usable_fraction": float(host_out["usable"].mean()),
               "steps": steps, "warmup": warmup}
    ctx.host_barrier()
    return out


def leg_fleet_tick(ctx, steps, warmup, robots=16384, A=20):
    """SURVEY §8f / VERDICT item 5-6: the whole Optimizer::optimize tick for a fleet through ONE C call
    (smpc_optimize_batch): host buffers hold what the controller has — seed path and cmds, RAW people (x, y, vx, vy,
    vz), speed — and the SFM crowd projection, the solve with per-robot horizons, the post-solve expansion and the
    warm-start memory update run on the device; costmaps and obstacle grids stay resident. Compared with the level-1
    e2e arm (which ships the PROJECTED agent trajectories, 6 x (S+1) doubles per agent) the tick moves ~14x fewer
    bytes per robot. Every rank runs its own fleet (weak scaling); wall clock per tick, max over ranks."""
    from nav2_social_mpc_controller_b200.fleet import FleetOptimizer
    rng = np.random.default_rng(20261018 + 77 + ctx.rank)
    p = sc.make_params("soc_work_obst")
    B = robots
    pose = np.stack([rng.uniform(0.5, 1.0, B), 2.0 + rng.uniform(-0.3, 0.3, B), rng.uniform(-0.3, 0.3, B)], axis=1)
    gp = sc._straight_path(B, np.full(B, 0.6), np.full(B, 2.0))
    poses_h, cmds_h = sc.pure_pursuit_seed(gp, pose, p)
    people = np.zeros((B, A, 5))
    people[:, :, 0] = rng.uniform(1.0, 3.0, (B, A))  # nobody leaves the 4 m obstacle grid within the horizon
    people[:, :, 1] = rng.uniform(1.0, 3.0, (B, A))
    people[:, :, 2:4] = rng.uniform(-0.5, 0.5, (B, A, 2))
    n_people = np.full(B, A, dtype=np.int32)
    speed = np.tile([0.3, 0.0], (B, 1))
    costmap = sc.wall_costmap(80, 80, 0.05, walls_y=(0.6, 3.4))[None]
    rows = np.arange(80)[:, None] * np.ones((1, 80), dtype=int)
    cols = np.ones((80, 1), dtype=int) * np.arange(80)[None, :]
    near = np.where(np.abs(rows - 12) <= np.abs(rows - 68), 12, 68)
    od = dict(width=80, height=80, resolution=0.05, origins=[[0.0, 0.0]], indexes=(near * 80 + cols).astype(np.uint32).ravel())
    fl = FleetOptimizer(p, n_robots=B, n_agents=A, device=ctx.local_rank)
    n = poses_h.shape[1]
    # in/out buffers as the controller holds them: the trajectorizer's fresh seed of every tick goes in, the optimised
    # path / cmds come back in place (one pre-filled buffer pair per tick, so no copy sits in the timed region)
    seeds = []
    for _ in range(warmup + steps):
        c = np.zeros((B, n, 2))
        c[:, :cmds_h.shape[1]] = cmds_h[:, :, :2]
        seeds.append((np.ascontiguousarray(poses_h, dtype=np.float64).copy(), c))
    origin = np.zeros((1, 2))

    def tick(i):
        return fl.optimize_batch(seeds[i][0], seeds[i][1], people, n_people, speed, costmap, origin, 0.05, od,
                                 want_people_proj=False, inplace=True)
    for i in range(warmup):
        r = tick(i)
    ctx.barrier()
    ts = []
    for i in range(steps):
        t0 = time.perf_counter()
        r = tick(warmup + i)
        ts.append(time.perf_counter() - t0)
    fl.close()
    (tot,) = ctx.max_over_ranks(float(sum(ts)))
    h2d = B * (n * 3 * 8 + n * 2 * 8 + A * 5 * 8 + 4 + 2 * 8 + 4)
    d2h = B * (n * 3 * 8 + n * 2 * 8 + 4 + 1 + 4 + 4 + 8 + 8 + 4)
    level1 = B * 8 * (3 + 6 + 2 * n + 1 + 6 * A * n)
    if ctx.rank != 0:
        return None
    return {"workload": f"fleet tick: {B} robots per GPU x {A} people, soc_work_obst params, seed paths of {n} poses",
            "entry": "smpc_optimize_batch (host buffers in / out; people projection, solve, post-solve and warm-start "
                     "memory on the device; maps resident)",
            "scaling": "weak", "value": ctx.world * B * steps / tot, "unit": "robot ticks/s",
            "ms_per_step": 1e3 * tot / steps, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "level1_e2e_h2d_bytes_for_the_same_fleet": int(level1), "h2d_reduction": round(level1 / h2d, 1),
            "optimized_fraction": float(r["optimized"].mean()), "mean_iterations": float(r["iterations"].mean()),
            "steps": steps, "warmup": warmup}


def leg_latency(ctx, calls):
    """BASELINE configs[0]: p50 / p99 of ONE solve through the host-buffer C-ABI (H2D + kernel + D2H), rank 0."""
    from nav2_social_mpc_controller_b200.optimizer import Optimizer
    out = {}
    for pname in ("readme", "params_yaml", "soc_work_obst"):
        b = sc.single(pname, n_people=3)
        opt = Optimizer(ctx.local_rank)
        opt.initialize(b.params)
        for _ in range(30):
            r = opt.solve_batch(b)
        lat = []
        for _ in range(calls):
            t0 = time.perf_counter()
            r = opt.solve_batch(b)
            lat.append(time.perf_counter() - t0)
        lat = np.sort(np.array(lat)) * 1e3
        out[pname] = {"S": b.n_steps, "P": 2 * b.n_blocks, "agents": 3, "p50_ms": float(lat[len(lat) // 2]),
                      "p99_ms": float(lat[int(len(lat) * 0.99)]), "iterations": int(r["iterations"][0]),
                      "evaluations": int(r["n_evals"][0].sum()), "calls": calls}
        opt.close()
    out["what"] = "smpc_solve_batch, B = 1, host buffers in / out; budget = one 20 Hz controller period (50 ms)"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=HEADLINE, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--legs", default="all", help="all | none | comma list of obst_only,multistart,scaling_sweep,scaling_sweep_omni,library_multi,fleet_tick,latency")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--latency-calls", type=int, default=300)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the headline workload as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libsmpc has no CPU path")
    ctx = Ctx(rank, local_rank, world)
    legs = ("obst_only", "multistart", "scaling_sweep", "scaling_sweep_omni", "library_multi", "fleet_tick", "latency") \
        if args.legs == "all" else \
        tuple(x for x in args.legs.split(",") if x and x != "none")
    if args.latency_calls <= 0:
        legs = tuple(x for x in legs if x != "latency")

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.15)
    threads = os.cpu_count() or 1
    res = measure(ctx, args.workload, args.steps, args.warmup, sampler=sampler,
                  with_cpu=not args.no_cpu_baseline, threads=threads, dump_dir=args.dump_outputs)
    time.sleep(0.06)
    sampler.stop()
    sampler.join(timeout=2)
    tot_ms, tot_e2e = ctx.max_over_ranks(float(sum(res["step_ms"])), float(sum(res["e2e_t"])))
    line = None
    if rank == 0:
        k_ms = tot_ms / args.steps
        roof, solver = roofline_block(ctx, res, k_ms)
        line = {
            "metric": METRIC, "value": world * res["B"] * args.steps / (tot_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": k_ms, "higher_is_better": True,
            "scaling": "strong" if res["tiled"] else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "description": res["desc"], "problems_per_gpu": res["B"],
                       "n_steps": res["S"], "e2e_problems_per_gpu": res["Bu"], "n_params": 2 * res["nb"],
                       "n_agents": res["A"], "l2": "flushed between timed steps (256 MiB write)",
                       "timing": "CUDA events per step on the launching stream, max over ranks"},
            "e2e": {"value": world * res["Bu"] * args.steps / tot_e2e, "unit": UNIT, "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": res["d2h"], "ms_per_step": 1e3 * tot_e2e / args.steps,
                    "how": "smpc_solve_batch(host pinned buffers): H2D + solve kernel + D2H + sync, wall clock"},
            "gpu_launches": int(res["launches"]),
            "clocks": sampler.summary(),
            "roofline": roof, "solver": solver,
        }
        if "cpu_baseline" in res:
            line["cpu_baseline"] = res["cpu_baseline"]
            line["parity_vs_oracle"] = res["parity"]
    res["opt"].close()
    del res
    torch.cuda.empty_cache()

    leg_out = {}
    if "obst_only" in legs and args.workload != "obst_only_x4096":
        leg_out["obst_only_x4096"] = leg_simple(ctx, "obst_only_x4096", min(args.steps, 10), args.warmup)
    if "multistart" in legs:
        leg_out["multistart_256x1024"] = leg_multistart(ctx, min(args.steps, 3), 3)
    if "scaling_sweep" in legs:
        leg_out["crowd_x1M_A50"] = leg_scaling_sweep(ctx, min(args.steps, 2), 2)
    if "scaling_sweep_omni" in legs:
        leg_out["crowd_x1M_A50_omni"] = leg_scaling_sweep(ctx, min(args.steps, 2), 2, omni=True)
    if "library_multi" in legs:
        leg_out["library_multi_gpu"] = leg_library_multi(ctx, min(args.steps, 3), 2)
    if "fleet_tick" in legs:
        leg_out["fleet_tick_A20"] = leg_fleet_tick(ctx, min(args.steps, 5), 2)
    if "latency" in legs and rank == 0:
        leg_out["single_solve_latency"] = leg_latency(ctx, args.latency_calls)
    if rank == 0:
        if leg_out:
            line["legs"] = leg_out
            if "single_solve_latency" in leg_out:
                line["latency_ms"] = {"p50": leg_out["single_solve_latency"]["params_yaml"]["p50_ms"],
                                      "p99": leg_out["single_solve_latency"]["params_yaml"]["p99_ms"],
                                      "what": "BASELINE configs[0]: smpc_solve_batch, B=1, params.yaml set, 3 people"}
        print(json.dumps(line))
    if world > 1:
        ctx.dist.barrier()
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
