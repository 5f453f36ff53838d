"""CPU tests of per-robot critic weights: the ctypes mirror of smpc_weight_sets against include/smpc.h, the exported
entries, the weight order of a table row, weight_sets and the checks of the `weights=` keyword."""
import os
import re

import numpy as np
import pytest

from nav2_social_mpc_controller_b200 import _lib, abi, scenarios as sc
from nav2_social_mpc_controller_b200.fleet import weight_sets_arg
from nav2_social_mpc_controller_b200.optimizer import OptimizerParams, weight_sets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = open(os.path.join(ROOT, "include", "smpc.h")).read()


def _fields(struct):
    body = re.search(r"typedef struct " + struct + r" \{(.*?)\} " + struct + ";", HDR, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [re.sub(r"\[.*\]", "", d.strip().split()[-1].lstrip("*")) for d in body.split(";") if d.strip()]


def test_weight_sets_struct_matches_header_and_entries_are_exported():
    assert _fields("smpc_weight_sets") == [f[0] for f in abi.SmpcWeightSets._fields_]
    L = _lib.lib()
    for name in ("smpc_optimize_batch_weighted", "smpc_run_weighted_episodes"):
        assert re.search(r"\bint " + name + r"\(", HDR)
        assert hasattr(L, name) and name in _lib.EXPORTED_SYMBOLS


def test_weight_row_order_is_smpc_params_order():
    names = _fields("smpc_params")
    i = names.index("distance_w")
    assert tuple(names[i:i + 9]) == abi.WEIGHT_NAMES
    p = sc.make_params("soc_work_obst")
    assert np.array_equal(abi.weight_row(p), [20.0, 120.0, 10.0, 250.0, 40.0, 90.0, 5.0, 0.13, 10.0])
    assert np.array_equal(abi.weight_row(OptimizerParams.from_struct(p)), abi.weight_row(p))


def test_weight_sets_of_the_two_benchmark_configurations():
    base = sc.make_params("soc_work_obst")
    t = weight_sets([sc.make_params("obst_only"), sc.make_params("soc_work_obst")], base)
    assert t.shape == (2, 9) and t.dtype == np.float64
    diff = [abi.WEIGHT_NAMES[j] for j in np.nonzero(t[0] != t[1])[0]]
    assert diff == ["socialwork_w", "agent_angle_w"]
    assert np.array_equal(t[1], abi.weight_row(base))


@pytest.mark.parametrize("field,value", [("control_horizon", 12), ("time_step", 0.1), ("fov_angle", 1.0),
                                         ("current_cmds_w", 1.0), ("param_tol", 1e-6), ("base_frame", b"odom")])
def test_weight_sets_rejects_a_differing_non_weight_field(field, value):
    base = sc.make_params("soc_work_obst")
    other = sc.make_params("obst_only")
    setattr(other, field, value)
    with pytest.raises(ValueError, match=field):
        weight_sets([base, other], base)
    with pytest.raises(ValueError):
        weight_sets([], base)


def test_weights_keyword_checks_shapes_and_indices():
    t = np.ones((3, 9))
    ws, keep = weight_sets_arg((t, [0, 2, 1, 2]), 4)
    assert ws.n_sets == 3 and keep[1].dtype == np.int32 and list(keep[1]) == [0, 2, 1, 2]
    assert ws.weights == keep[0].ctypes.data and ws.set_index == keep[1].ctypes.data
    for bad in ((np.ones((3, 8)), [0, 0, 0, 0]), (np.ones((0, 9)), np.zeros(4, int)), (np.ones(9), [0, 0, 0, 0]),
                (t, [0, 1, 2]), (t, [[0, 1], [2, 0]]), (t, [0.0, 1.0, 2.0, 0.0]),
                (t, [0, 3, 1, 2]), (t, [0, -1, 1, 2])):
        with pytest.raises(ValueError):
            weight_sets_arg(bad, 4)
