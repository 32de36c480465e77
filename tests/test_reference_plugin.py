"""GPU (-m gpu): the batched entry of examples/reference_plugin/b200_solverwrapper.py (pure ctypes over the C-ABI, no
torch, none of this repo's Python package), the routine that gives the reference the solver-wrapper name "b200", must
return what the UNMODIFIED reference computes path by path with its own TOPPRA(..., solver_wrapper="seidel").  The
reference's results are stored in tests/golden/plugin_batch.npz (tests/golden/make_golden.py plugin_batch, whose
PLUGIN_SINGLE_CASES are the parameters below)."""
import importlib.util
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def plugin():
    spec = importlib.util.spec_from_file_location(
        "b200_solverwrapper", os.path.join(ROOT, "examples", "reference_plugin", "b200_solverwrapper.py"))
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


@pytest.mark.parametrize("seed,G,vel_active,s0,s1,scheme", [(1000, 200, False, 0.0, 0.0, 1), (1003, 100, True, 0.0, 0.0, 1),
                                                           (1005, 150, False, 0.1, 0.1, 1), (1007, 64, False, 0.0, 0.0, 0),
                                                           (1002, 100, False, 30.0, 0.0, 1)])
def test_plugin_single_paths_equal_reference(plugin, golden, seed, G, vel_active, s0, s1, scheme):
    """One path per call, with boundary velocities, the collocation scheme and an inadmissible start: controllable sets,
    velocities, accelerations and return code of the reference's TOPPRA(..., solver_wrapper="seidel")."""
    from problems import make_path
    way, vlim, alim = make_path(seed, vel_active=vel_active)
    ref = golden("plugin_batch")
    u, sd, K, status = plugin.solve_velacc(np.linspace(0, 1, 5), way[None], np.linspace(0, 1, G), vlim, alim, sd_start=s0,
                                           sd_end=s1, interpolation=bool(scheme))
    key = "single%d_" % seed
    assert status[0] == ref[key + "status"]
    assert np.array_equal(K[0], ref[key + "K"], equal_nan=True)
    if status[0] != 0:
        assert status[0] == 3 and s0 == 30.0   # inadmissible start: FailUncontrollable on both
    else:
        assert np.array_equal(sd[0], ref[key + "sd"]) and np.array_equal(u[0], ref[key + "sdd"])


def test_plugin_batched_entry_equals_reference(plugin, golden):
    """solve_velacc(B paths) == the reference solved path by path."""
    from problems import make_batch
    B, G = 24, 120
    ss, way, vlim, alim = make_batch(B, 1000)
    grid = np.linspace(0, 1, G)
    ref = golden("plugin_batch")
    u, sd, K, status = plugin.solve_velacc(ss, way, grid, vlim, alim)
    for b in range(B):
        assert ref["status"][b] == 0
        assert status[b] == 0 and np.array_equal(K[b], ref["K"][b]) and np.array_equal(sd[b], ref["sd"][b])
        assert np.array_equal(u[b], ref["sdd"][b])
