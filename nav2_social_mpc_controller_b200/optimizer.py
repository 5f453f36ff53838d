"""Host-side mirror of the reference optimizer interface for the solve path, over libsmpc.so.

Reference interface mirrored (include/nav2_social_mpc_controller/optimizer.hpp):
  struct OptimizerParams (:59-101)          -> OptimizerParams (defaults of src/optimizer.cpp:26-84, from_yaml)
  Optimizer::initialize(params) (:152)      -> Optimizer.initialize(params)
  ceres::Solve inside Optimizer::optimize   -> Optimizer.solve_batch / solve_batch_device (level-1 C-ABI)
All compute happens in the CUDA library; this file only marshals buffers. No CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib, abi


class OptimizerParams:
    """Same fields and defaults as the reference OptimizerParams (+ trajectorizer.* the optimizer reads)."""

    def __init__(self, **overrides):
        self.c = abi.SmpcParams()
        _lib.lib().smpc_params_default(C.byref(self.c))
        for k, v in overrides.items():
            self.set(k, v)

    def set(self, key, value):
        if key in ("linear_solver_type", "base_frame") and isinstance(value, str):
            value = value.encode()
        setattr(self.c, key, value)

    def __getattr__(self, key):
        if key == "c":
            raise AttributeError(key)
        v = getattr(self.c, key)
        return v.decode() if isinstance(v, bytes) else v

    @classmethod
    def from_yaml(cls, path: str, plugin_name: str = "FollowPath") -> "OptimizerParams":
        """OptimizerParams::get (reference src/optimizer.cpp:16-85): reads `<plugin>.optimizer.*`,
        `<plugin>.optimizer.weights.*` and `<plugin>.trajectorizer.*`. Raises on an invalid linear_solver_type
        like the reference's std::runtime_error (:44)."""
        self = cls.__new__(cls)
        self.c = abi.SmpcParams()
        _lib.check(_lib.lib().smpc_params_from_yaml(path.encode(), plugin_name.encode(), C.byref(self.c)))
        return self

    @classmethod
    def from_struct(cls, c: abi.SmpcParams) -> "OptimizerParams":
        self = cls.__new__(cls)
        self.c = c
        return self


def weight_sets(params_list, base) -> np.ndarray:
    """The [P][9] weight table (abi.WEIGHT_NAMES columns) of P params structs that may differ from `base`, the handle's
    params, in their critic weights only: every other field is the handle's in a weighted call, so a params that
    differs elsewhere would not be computed as written. Raises ValueError naming the first such field."""
    def fields(p):
        c = p.c if isinstance(p, OptimizerParams) else p
        return {k: getattr(c, k) for k, _ in abi.SmpcParams._fields_}
    ref = fields(base)
    rows = []
    for i, p in enumerate(params_list):
        f = fields(p)
        for k, v in f.items():
            if k not in abi.WEIGHT_NAMES and v != ref[k]:
                raise ValueError(f"weight_sets: params {i} differs from the handle's params in {k} "
                                 f"({v!r} vs {ref[k]!r}); only the critic weights may differ")
        rows.append(abi.weight_row(p))
    if not rows:
        raise ValueError("weight_sets: no params given")
    return np.array(rows, dtype=np.float64)


class Optimizer:
    """Batched drop-in for the solve inside nav2_social_mpc_controller::Optimizer. One instance per GPU."""

    def __init__(self, device: int = 0):
        self.device = device
        self._h = None
        self.params = None

    def initialize(self, params) -> None:
        """Optimizer::initialize (reference src/optimizer.cpp:98-132)."""
        if isinstance(params, abi.SmpcParams):
            params = OptimizerParams.from_struct(params)
        self.close()
        h = C.c_void_p()
        _lib.check(_lib.lib().smpc_create(C.byref(params.c), self.device, C.byref(h)))
        self._h = h
        self.params = params

    def close(self):
        if self._h is not None:
            _lib.lib().smpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _need(self):
        if self._h is None:
            raise RuntimeError("Optimizer.initialize(params) has not been called")

    def dims(self, n_steps: int):
        ch, bl, nb, nbd = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        _lib.check(_lib.lib().smpc_problem_dims(C.byref(self.params.c), n_steps, C.byref(ch), C.byref(bl), C.byref(nb),
                                                C.byref(nbd)))
        return ch.value, bl.value, nb.value, nbd.value

    # ---- level-1 solve, host buffers (numpy or pinned torch CPU tensors) --------------------------------
    def solve_batch(self, batch, out: dict | None = None,
                    want=("u", "cmds", "cost_initial", "cost_final", "iterations", "termination", "usable",
                          "n_evals"), trace_rows: int = 0) -> dict:
        """H2D copy of the batch, one solve launch, D2H copy of the results (all inside the C call).
        trace_rows > 0 adds out["trace"] [B][trace_rows][8] (per-evaluation solver trace, include/smpc.h)."""
        self._need()
        nb = self.dims(batch.n_steps)[2]
        if out is None:
            shapes = abi.result_shapes(batch.n_problems, batch.n_steps, nb, 3 if int(self.params.omni_solve) else 2)
            out = {k: np.zeros(shapes[k][0], dtype=shapes[k][1]) for k in want}
            if trace_rows > 0:
                out["trace"] = np.full((batch.n_problems, trace_rows, 8), np.nan)
        st = batch.struct()
        rs = abi.make_result_struct(out)
        _lib.check(_lib.lib().smpc_solve_batch(self._h, C.byref(st), C.byref(rs)))
        return out

    # ---- level-1 solve, device buffers (torch CUDA tensors), asynchronous on `stream` -------------------
    def solve_batch_device(self, batch_struct: abi.SmpcBatch, out: dict, stream: int | None = None) -> None:
        self._need()
        rs = abi.make_result_struct(out)
        _lib.check(_lib.lib().smpc_solve_batch_device(self._h, C.byref(batch_struct), C.byref(rs),
                                                      C.c_void_p(stream) if stream else None))

    # ---- level-2 entry: bool Optimizer::optimize(path, people_proj, costmap, obstacles, cmds, people, speed, dt) ----
    def optimize(self, path: np.ndarray, cmds: np.ndarray, people: np.ndarray, speed, time_step: float,
                 costmap: np.ndarray, costmap_origin, costmap_resolution: float, od: dict):
        """Mirror of the reference call (include/nav2_social_mpc_controller/optimizer.hpp:167-170).
        path [n][3] (x, y, yaw) and cmds [m][2] are the trajectorizer's seed and come back optimised (in-out like
        the reference); people [k][5] = position.x/y, velocity.x/y/z; speed = (linear.x, angular.z); od = dict(width,
        height, resolution, origin_x, origin_y, distances f32[], indexes u32[]).
        Returns (ok, path, cmds, people_proj[P][3][6], info). ok == False <=> the reference returns false."""
        self._need()
        path = np.ascontiguousarray(path, dtype=np.float64).reshape(-1, 3)
        cmds = np.ascontiguousarray(cmds, dtype=np.float64).reshape(-1, 2)
        people = np.ascontiguousarray(people, dtype=np.float64).reshape(-1, 5)
        costmap = np.ascontiguousarray(costmap, dtype=np.uint8)
        cap = max(path.shape[0], cmds.shape[0]) + 2
        poses_buf = np.zeros((cap, 3))
        poses_buf[: path.shape[0]] = path
        cmds_buf = np.zeros((cap, 2))
        cmds_buf[: cmds.shape[0]] = cmds
        proj = np.zeros((cap, 3, 6))
        dist = np.ascontiguousarray(od["distances"], dtype=np.float32)
        idx = np.ascontiguousarray(od["indexes"], dtype=np.uint32)
        io = abi.SmpcOptimizeIo()
        io.capacity, io.n_poses, io.n_cmds, io.n_people = cap, path.shape[0], cmds.shape[0], people.shape[0]
        io.poses, io.cmds, io.people = poses_buf.ctypes.data, cmds_buf.ctypes.data, people.ctypes.data
        io.speed_v, io.speed_w, io.time_step = float(speed[0]), float(speed[1]), float(time_step)
        io.costmap, io.size_x, io.size_y = costmap.ctypes.data, costmap.shape[1], costmap.shape[0]
        io.origin_x, io.origin_y, io.resolution = float(costmap_origin[0]), float(costmap_origin[1]), float(
            costmap_resolution)
        io.od.width, io.od.height, io.od.resolution = int(od["width"]), int(od["height"]), float(od["resolution"])
        io.od.origin_x, io.od.origin_y = float(od["origin_x"]), float(od["origin_y"])
        io.od.distances = dist.ctypes.data if dist.size else None
        io.od.indexes = idx.ctypes.data if idx.size else None
        io.people_proj = proj.ctypes.data
        _lib.check(_lib.lib().smpc_optimize(self._h, C.byref(io)))
        info = dict(termination=io.termination, iterations=io.iterations, cost_initial=io.cost_initial,
                    cost_final=io.cost_final)
        return (bool(io.optimized), poses_buf[: io.n_poses].copy(), cmds_buf[: io.n_cmds].copy(),
                proj[: io.n_proj_steps].copy(), info)

    def project_people_batch(self, robot: np.ndarray, people_init: np.ndarray, od: dict, max_time: float,
                             time_step: float, od_index: np.ndarray | None = None):
        """Batched GPU project_people (reference src/optimizer.cpp:554-671): robot [B][S+1][6], people_init [B][A][6]
        (t == -1: padded), od = dict(width, height, resolution, origins [M][2], indexes u32 [M][h*w]).
        Returns (agents [B][A][6][S+1] in the level-1 layout, status [B])."""
        self._need()
        robot = np.ascontiguousarray(robot, dtype=np.float64)
        people_init = np.ascontiguousarray(people_init, dtype=np.float64)
        B, S1, _ = robot.shape
        A = people_init.shape[1]
        origins = np.ascontiguousarray(od["origins"], dtype=np.float64).reshape(-1, 2)
        idx = np.ascontiguousarray(od["indexes"], dtype=np.uint32).reshape(origins.shape[0], -1)
        out = np.zeros((B, A, 6, S1))
        status = np.zeros(B, dtype=np.int32)
        a = abi.SmpcProjectArgs()
        a.n_problems, a.n_steps, a.n_agents, a.n_grids = B, S1 - 1, A, origins.shape[0]
        a.od_width, a.od_height, a.od_resolution = int(od["width"]), int(od["height"]), float(od["resolution"])
        a.max_time, a.time_step = float(max_time), float(time_step)
        a.od_origin, a.od_indexes = origins.ctypes.data, idx.ctypes.data
        oi = None if od_index is None else np.ascontiguousarray(od_index, dtype=np.int32)
        a.od_index = None if oi is None else oi.ctypes.data
        a.robot, a.people_init, a.agents, a.status = (robot.ctypes.data, people_init.ctypes.data, out.ctypes.data,
                                                      status.ctypes.data)
        _lib.check(_lib.lib().smpc_project_people_batch(self._h, C.byref(a)))
        return out, status

    def reset_memory(self) -> None:
        """Forget the previous path / cmds (fresh TrajectoryMemory)."""
        self._need()
        _lib.check(_lib.lib().smpc_reset_memory(self._h))

    def eval_batch(self, batch, x: np.ndarray) -> dict:
        """cost, J^T r, J^T J at block values x [B][NB][2] (host buffers)."""
        self._need()
        nb = self.dims(batch.n_steps)[2]
        P = (3 if int(self.params.omni_solve) else 2) * nb
        B = batch.n_problems
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(B, P)
        out = dict(cost=np.zeros(B), grad=np.zeros((B, P)), hess=np.zeros((B, P * (P + 1) // 2)),
                   ok=np.zeros(B, dtype=np.uint8), cost_plain=np.zeros(B))
        eo = abi.SmpcEvalOut()
        for k in ("cost", "grad", "hess", "ok", "cost_plain"):
            setattr(eo, k, out[k].ctypes.data)
        st = batch.struct()
        _lib.check(_lib.lib().smpc_eval_batch(self._h, C.byref(st), x.ctypes.data, C.byref(eo)))
        return out

    def multistart_argmin_device(self, n_robots, n_starts, n_blocks, cost_final, usable, u, best_index, best_cost,
                                 best_u, stream: int | None = None):
        self._need()
        p = abi._ptr
        _lib.check(_lib.lib().smpc_multistart_argmin_device(
            self._h, n_robots, n_starts, n_blocks, p(cost_final), p(usable), p(u), p(best_index), p(best_cost),
            p(best_u), C.c_void_p(stream) if stream else None))

    def set_group(self, lanes_per_problem: int) -> None:
        """Lanes per problem (0 = auto, 4, 8, 16, 32): throughput vs latency mapping of the solve kernel."""
        self._need()
        _lib.check(_lib.lib().smpc_set_group(self._h, lanes_per_problem))

    def last_kernel_ms(self) -> float:
        self._need()
        return float(_lib.lib().smpc_last_kernel_ms(self._h))

    def debug_polymin(self, rows: np.ndarray) -> np.ndarray:
        """Line-search polynomial minimiser on rows of (lo, hi, f0, g0, t1, f1, g1, t2, f2, g2) (unit tests)."""
        self._need()
        rows = np.ascontiguousarray(rows, dtype=np.float64).reshape(-1, 10)
        out = np.zeros(rows.shape[0])
        _lib.check(_lib.lib().smpc_debug_polymin(self._h, rows.shape[0], rows.ctypes.data, out.ctypes.data))
        return out

    def debug_math(self, kind: int, a: np.ndarray, b: np.ndarray | None = None) -> np.ndarray:
        """The kernel's own exp_nonpos (kind 0) / rsqrt_pos (1) / atan2_unit(a, b) (2) on arrays (unit tests)."""
        self._need()
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        rows = np.stack([a, np.zeros_like(a) if b is None else np.ascontiguousarray(b, dtype=np.float64).ravel()], axis=1)
        rows = np.ascontiguousarray(rows)
        out = np.zeros(a.shape[0])
        _lib.check(_lib.lib().smpc_debug_math(self._h, int(kind), a.shape[0], rows.ctypes.data, out.ctypes.data))
        return out

    def measure_fp64_peak(self) -> float:
        """TFLOP/s of a DFMA-saturating microbenchmark on this GPU (roofline denominator)."""
        self._need()
        v = C.c_double(0.0)
        _lib.check(_lib.lib().smpc_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    def launch_count(self) -> int:
        self._need()
        return int(_lib.lib().smpc_launch_count(self._h))


class MultiGpuOptimizer:
    """smpc_solve_batch_multi: one host batch solved across several GPUs inside the library (one host thread + handle
    per GPU, contiguous shards at multiples of `granule`, results land in the caller's host arrays). `devices` may name
    a GPU more than once."""

    def __init__(self, params, devices):
        if isinstance(params, abi.SmpcParams):
            params = OptimizerParams.from_struct(params)
        self.params = params
        devs = (C.c_int * len(devices))(*devices)
        h = C.c_void_p()
        _lib.check(_lib.lib().smpc_multi_create(C.byref(params.c), len(devices), devs, C.byref(h)))
        self._m = h

    def close(self):
        if self._m is not None:
            _lib.lib().smpc_multi_destroy(self._m)
            self._m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve_batch(self, batch, out: dict | None = None, granule: int = 1,
                    want=("u", "cmds", "cost_initial", "cost_final", "iterations", "termination", "usable", "n_evals")):
        ch, bl, nb, nbd = abi.problem_dims(self.params.control_horizon, self.params.parameter_block_length, batch.n_steps)
        if out is None:
            shapes = abi.result_shapes(batch.n_problems, batch.n_steps, nb, 3 if int(self.params.omni_solve) else 2)
            out = {k: np.zeros(shapes[k][0], dtype=shapes[k][1]) for k in want}
        st = batch.struct()
        rs = abi.make_result_struct(out)
        _lib.check(_lib.lib().smpc_solve_batch_multi(self._m, C.byref(st), C.byref(rs), int(granule)))
        return out


def hess_to_dense(h_packed: np.ndarray, P: int) -> np.ndarray:
    """Row-major lower-triangle packing of include/smpc.h -> dense symmetric [.., P, P]."""
    out = np.zeros(h_packed.shape[:-1] + (P, P))
    e = 0
    for a in range(P):
        for b in range(a + 1):
            out[..., a, b] = h_packed[..., e]
            out[..., b, a] = h_packed[..., e]
            e += 1
    return out
