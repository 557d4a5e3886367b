"""Replays the committed golden fixtures (tests/golden/*.npz, outputs of the unmodified
reference) on any planner factory."""
import os

import numpy as np

import scenarios as sc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LOCS = ["DRIVING"]


def load(name):
    return np.load(os.path.join(GOLDEN, name))


def replay_config1(factory):
    g = load("config1_100.npz")
    p = sc.make_planner(factory, 1, 100, 100)
    assert p.computeCostMap(g["lut"], g["slopes"], LOCS, g["elevation"], g["terrain"])
    gi, gj = (int(v) for v in g["goal"])
    si, sj = (int(v) for v in g["start"])
    assert p.setGoal(gi, gj)
    assert p.computeTotalCostMap(si, sj)
    out = dict(obstacle=sc.obstacle_plane(p), total_cost_early=p.getTotalCostMatrix())
    out["state_early"] = (p.node_field(5) if hasattr(p, "node_field")
                          else p.plane("state").astype(np.float64))
    out["cost"] = (p.node_field(3) if hasattr(p, "node_field") else p.plane("cost"))
    if hasattr(p, "node_field"):
        out["slope"], out["raw_cost"] = p.node_field(1), p.node_field(2)
    out["path_early"] = p.getPath(si, sj)
    assert p.computeEntireTotalCostMap()
    out["total_cost_full"] = p.getTotalCostMatrix()
    out["path_full"] = p.getPath(si, sj)
    return g, out


def replay_repair(factory, approach, name):
    g = load(name)
    p = sc.make_planner(factory, approach, 120, 120)
    assert p.computeCostMap(g["lut"], g["slopes"], LOCS, g["elevation"], g["terrain"])
    gi, gj = (int(v) for v in g["goal"])
    si, sj = (int(v) for v in g["start"])
    assert p.setGoal(gi, gj) and p.computeEntireTotalCostMap()
    path = p.getPath(si, sj)
    c = g["centre"]
    repaired, traj, _ = p.computeLocalPlanning(float(c[0]), float(c[1]), g["image"], 0.1)
    out = dict(path=path, repaired=repaired, traj=traj, risk=p.getRiskMatrix(c[0], c[1]),
               deviation=p.getDeviationMatrix(c[0], c[1]), hazard=p.getHazardDensityMatrix(),
               traff=p.getTrafficabilityMatrix(), reconnecting_index=p.getReconnectingIndex())
    if hasattr(p, "node_field"):
        out["has_local"] = p.node_field(6)
    return g, out
