"""The oracle's C restatement must reproduce the committed golden vectors bit for bit."""
import numpy as np
import pytest

import golden_cases as gc


def test_port_reproduces_config1(oracle_mod):
    g, o = gc.replay_config1(oracle_mod.Port)
    assert np.array_equal(o["obstacle"], g["obstacle"])
    assert np.array_equal(o["cost"], g["cost"])
    assert np.array_equal(o["slope"], g["slope"])          # node_field(1), as the reference taps it
    assert np.array_equal(o["raw_cost"], g["raw_cost"])    # node_field(2)
    assert np.array_equal(o["total_cost_early"], g["total_cost_early"])
    assert np.array_equal(o["state_early"], g["state_early"])
    assert np.array_equal(o["path_early"], g["path_early"])
    assert np.array_equal(o["total_cost_full"], g["total_cost_full"])
    assert np.array_equal(o["path_full"], g["path_full"])


@pytest.mark.parametrize("approach,name", [(1, "repair_120_sweeping.npz"),
                                           (0, "repair_120_conservative.npz")])
def test_port_reproduces_repair(oracle_mod, approach, name):
    g, o = gc.replay_repair(oracle_mod.Port, approach, name)
    assert o["repaired"]
    for k in ("path", "traj", "risk", "deviation", "hazard", "traff", "has_local"):
        assert np.array_equal(o[k], g[k]), k
    assert o["reconnecting_index"] == int(g["reconnecting_index"])


def test_reference_still_reproduces_golden(ref_lib):
    """Guards against a stale fixture: the compiled reference regenerates it exactly."""
    g, o = gc.replay_config1(ref_lib.DyMuPathPlanner)
    assert np.array_equal(o["total_cost_early"], g["total_cost_early"])
    assert np.array_equal(o["path_full"], g["path_full"])
