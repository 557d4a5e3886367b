"""GPU parity through the reference-facing class interface: the same call sequence
(tests/scenarios.py) is issued to the reference (tests/conftest.py::ref_planner: the compiled
UNMODIFIED reference, or its bit-exact C restatement where that is not built) and to the B200 drop-in (libdymu_b200.so -> libdymu_cuda.so).

Bars (BASELINE.json north_star): obstacle / risk masks and indices bit-exact; total-cost,
risk and deviation planes <= 1e-9 relative; waypoints <= 1e-3 cell."""
import numpy as np
import pytest

import scenarios as sc
from conftest import rel_err

pytestmark = pytest.mark.gpu

TOL_PLANE = 1e-9
TOL_WP = 1e-3


def _pair(pkg, ref, approach, nx, ny, **kw):
    return (sc.make_planner(ref, approach, nx, ny, **kw),
            sc.make_planner(pkg.DyMuPathPlanner, approach, nx, ny, **kw))


def _closed(p):
    return p.node_field(pkg_state := 5) > 0


@pytest.mark.parametrize("ny,nx,seed", [(100, 100, 1), (129, 257, 2), (300, 300, 3)])
def test_entire_total_cost_map_and_path(pkg, ref_planner, ny, nx, seed):
    """computeEntireTotalCostMap + getPath (config 1 shape, full solve)."""
    ref, dut = _pair(pkg, ref_planner, 1, nx, ny)
    a = sc.global_scenario(ref, pkg.synthetic, nx, ny, seed, entire=True)
    b = sc.global_scenario(dut, pkg.synthetic, nx, ny, seed, entire=True)
    assert a["ok"] and b["ok"]
    assert np.array_equal(a["obstacle"], b["obstacle"])
    assert np.array_equal(a["T"] < 0, b["T"] < 0)
    assert rel_err(b["T"], a["T"]) <= TOL_PLANE
    assert rel_err(b["cost"], a["cost"]) <= 1e-14
    assert a["path"].shape == b["path"].shape
    assert np.max(np.abs(a["path"][:, :2] - b["path"][:, :2])) <= TOL_WP
    assert np.max(np.abs(a["path"][:, 2] - b["path"][:, 2])) <= 1e-6   # z
    assert np.max(np.abs(np.angle(np.exp(1j * (a["path"][:, 3] - b["path"][:, 3]))))) <= 1e-3


def test_config1_early_stop(pkg, ref_planner):
    """Config 1: 100x100, goal (75,75), start (20,25), computeTotalCostMap(start) + getPath.
    The reference stops once the start node and its 4 neighbours are CLOSED; parity is
    defined on the CLOSED set (SURVEY.md section 7, 'early-stop semantics')."""
    nx = ny = 100
    ref, dut = _pair(pkg, ref_planner, 1, nx, ny)
    a = sc.global_scenario(ref, pkg.synthetic, nx, ny, 1, goal_frac=(0.75, 0.75),
                           start_frac=(0.20, 0.25))
    b = sc.global_scenario(dut, pkg.synthetic, nx, ny, 1, goal_frac=(0.75, 0.75),
                           start_frac=(0.20, 0.25))
    assert a["ok"] and b["ok"]
    ca, cb = ref.node_field(5) > 0, dut.node_field(5) > 0
    assert np.array_equal(ca, cb), "CLOSED sets differ"
    assert rel_err(np.where(ca, b["T"], 0), np.where(ca, a["T"], 0)) <= TOL_PLANE
    # every cell the reference reached is reached here too
    assert np.all(b["T"][a["T"] >= 0] >= 0)
    assert a["path"].shape == b["path"].shape
    # the whole early-stop path, start waypoint included, at north_star's bound
    d = np.abs(a["path"][:, :2] - b["path"][:, :2]).max(axis=1)
    assert d.max() <= TOL_WP
    assert ref.getTotalCost(30.3, 40.6) == pytest.approx(dut.getTotalCost(30.3, 40.6), rel=1e-9)


def test_offset_and_locomotion_modes(pkg, ref_lib):
    nx, ny, off = 120, 90, (12.0, -7.0)
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(ny, nx, seed=6)
    lut, slopes, locs = syn.default_lut(n_loc=3)
    out = []
    for p in _pair(pkg, ref_lib.DyMuPathPlanner, 0, nx, ny, offset=off):
        assert p.computeCostMap(lut, slopes, locs, elev, terr)
        ob = sc.obstacle_plane(p)
        gi, gj = syn.free_interior_cell_near(ob, 90, 60)
        si, sj = syn.free_interior_cell_near(ob, 25, 25)
        assert p.setGoal(gi + off[0], gj + off[1])
        assert p.computeEntireTotalCostMap()
        out.append((p.getTotalCostMatrix(), p.getPath(si + off[0], sj + off[1]),
                    [p.getLocomotionMode(x + off[0], y + off[1]) for x, y in
                     ((30, 30), (60, 45), (100, 70), (0, 0))], p.node_field(2)))
    (Ta, pa, la, ra), (Tb, pb, lb, rb) = out
    assert rel_err(Tb, Ta) <= TOL_PLANE and np.array_equal(Ta < 0, Tb < 0)
    assert rel_err(rb, ra) <= 1e-14
    assert la == lb
    assert pa.shape == pb.shape and np.max(np.abs(pa[:, :2] - pb[:, :2])) <= TOL_WP


def test_invalid_goals_and_starts(pkg, ref_planner):
    nx = ny = 64
    cost = np.ones((ny, nx))
    cost[30:34, 30:34] = 0.0
    for p in _pair(pkg, ref_planner, 1, nx, ny):
        assert p.setCostMap(cost)
        assert not p.setGoal(-3.0, 5.0)
        assert not p.setGoal(0.0, 10.0)         # border
        assert not p.setGoal(63.0, 10.0)
        assert not p.setGoal(200.0, 10.0)       # outside
        assert not p.setGoal(31.0, 31.0)        # obstacle
        assert not p.setGoal(29.0, 31.0)        # next to an obstacle
        assert not p.computeEntireTotalCostMap()  # no goal yet
        assert p.setGoal(10.0, 10.0)
        assert not p.computeTotalCostMap(34.0, 34.0)  # start touches an obstacle
        assert p.computeTotalCostMap(50.0, 50.0)
        assert not p.setCostMap(np.ones((10, 10)))    # size mismatch


@pytest.mark.parametrize("approach", [1, 0])
def test_local_repair(pkg, ref_planner, approach):
    """Config 2 shape at 200x200: global plan, obstacle frame, computeLocalPlanning."""
    n, syn = 200, pkg.synthetic
    res = []
    for p in _pair(pkg, ref_planner, approach, n, n):
        g = sc.global_scenario(p, syn, n, n, seed=3, entire=True)
        r = sc.repair_scenario(p, syn, g["path"])
        res.append((g, r, p.node_field(6)))
    (ga, ra, ha), (gb, rb, hb) = res
    assert ra["repaired"] and rb["repaired"]
    assert np.array_equal(ra["risk"] > 0, rb["risk"] > 0), "risk mask"
    assert np.array_equal(ra["risk"] == 1.0, rb["risk"] == 1.0), "obstacle mask"
    assert np.max(np.abs(ra["risk"] - rb["risk"])) <= 1e-12
    assert np.array_equal(ra["deviation"] < 0, rb["deviation"] < 0), "propagated set"
    assert rel_err(rb["deviation"], ra["deviation"]) <= TOL_PLANE
    assert np.max(np.abs(ra["hazard"] - rb["hazard"])) <= 1e-12
    assert np.max(np.abs(ra["traff"] - rb["traff"])) <= 1e-9
    assert ra["reconnecting_index"] == rb["reconnecting_index"]
    assert ra["traj"].shape == rb["traj"].shape
    assert np.max(np.abs(ra["traj"][:, :2] - rb["traj"][:, :2])) <= TOL_WP
    assert np.array_equal(ha, hb), "hasLocalMap"


@pytest.mark.parametrize("approach", [1, 0])
def test_config2_1000(pkg, ref_planner, approach):
    """Config 2 at full size (SURVEY.md section 8d): 1000x1000, goal (800,800), start (200,200),
    computeTotalCostMap(start) + getPath, then a 120x120 px frame with an obstacle disc on
    path[10] (+3 random discs, seed 7) -> computeLocalPlanning, SWEEPING and CONSERVATIVE."""
    n, syn = 1000, pkg.synthetic
    res = []
    for p in _pair(pkg, ref_planner, approach, n, n):
        g = sc.global_scenario(p, syn, n, n, seed=20261018)
        r = sc.repair_scenario(p, syn, g["path"], disc_wp=10)
        res.append((g, r, p.node_field(5), p.node_field(6)))
    (ga, ra, ca, ha), (gb, rb, cb, hb) = res
    assert ga["ok"] and gb["ok"]
    closed = ca > 0
    assert np.array_equal(closed, cb > 0), "CLOSED set"
    assert rel_err(np.where(closed, gb["T"], 0), np.where(closed, ga["T"], 0)) <= TOL_PLANE
    assert ga["path"].shape == gb["path"].shape
    assert np.max(np.abs(ga["path"][:, :2] - gb["path"][:, :2])) <= TOL_WP
    assert ra["repaired"] and rb["repaired"]
    assert np.array_equal(ra["risk"] > 0, rb["risk"] > 0), "risk mask"
    assert np.array_equal(ra["risk"] == 1.0, rb["risk"] == 1.0), "obstacle mask"
    assert np.max(np.abs(ra["risk"] - rb["risk"])) <= 1e-12
    assert np.array_equal(ra["deviation"] < 0, rb["deviation"] < 0), "propagated set"
    assert rel_err(rb["deviation"], ra["deviation"]) <= TOL_PLANE
    assert np.max(np.abs(ra["hazard"] - rb["hazard"])) <= 1e-12
    assert np.max(np.abs(ra["traff"] - rb["traff"])) <= 1e-9
    assert ra["reconnecting_index"] == rb["reconnecting_index"]
    assert np.array_equal(ha, hb), "hasLocalMap"
    assert ra["traj"].shape == rb["traj"].shape
    assert np.max(np.abs(ra["traj"][:, :2] - rb["traj"][:, :2])) <= TOL_WP


def test_cora_loop_rebuilds_cost_map_on_device(pkg, ref_lib):
    """SURVEY.md section 8 row f4: traverse feedback -> updateCost (G.cpp:956-993) -> new table
    -> cost map -> total cost.  The reference is handed both maps again; the B200 build
    rebuilds from the elevation and terrain planes already resident in HBM.  getTerrain
    (G.cpp:941-950) is read from the device terrain plane."""
    nx, ny = 160, 120
    ref, dut = _pair(pkg, ref_lib.DyMuPathPlanner, 1, nx, ny)
    a = sc.global_scenario(ref, pkg.synthetic, nx, ny, 4, entire=True)
    b = sc.global_scenario(dut, pkg.synthetic, nx, ny, 4, entire=True)
    # the transformed read-backs above reuse the staging plane the terrain map was uploaded
    # through: the rebuild below must not depend on it
    for x, y in ((10.2, 20.7), (80.0, 60.0), (150.4, 100.6), (0.0, 0.0)):
        assert ref.getTerrain(x, y) == dut.getTerrain(x, y)
    taps_a = sc.cora_feed(ref, rounds=40, tap_every=40)
    taps_b = sc.cora_feed(dut, rounds=40, tap_every=40)
    assert np.array_equal(taps_a[-1][1], taps_b[-1][1])
    lut0, _, _ = pkg.synthetic.default_lut()
    assert not np.array_equal(taps_a[-1][1], np.asarray(lut0, dtype=np.float64))
    assert ref.recomputeCostMap() and dut.recomputeCostMap()
    assert np.array_equal(ref.node_field(4), dut.node_field(4))            # isObstacle
    assert rel_err(dut.node_field(2), ref.node_field(2)) <= 1e-14          # raw_cost
    ca, cb = ref.getGlobalCostMatrix(), dut.getGlobalCostMatrix()
    assert rel_err(cb, ca) <= 1e-14
    assert not np.array_equal(ca, a["cost"]), "the new table did not change the cost map"
    gx, gy = a["goal"]
    assert ref.setGoal(gx, gy) and dut.setGoal(gx, gy)
    assert ref.computeEntireTotalCostMap() and dut.computeEntireTotalCostMap()
    Ta, Tb = ref.getTotalCostMatrix(), dut.getTotalCostMatrix()
    assert np.array_equal(Ta < 0, Tb < 0)
    assert rel_err(Tb, Ta) <= TOL_PLANE
    assert rel_err(Tb, b["T"]) > 1e-6                                      # and it matters


def test_streamed_cost_map_and_matrix_delivery(pkg, ref_planner):
    """The copy-free flow of the drop-in -- setCostMap(const double*, ld) with the upload hidden
    behind the solve, total-cost matrix delivered into a caller buffer while getPath runs --
    against the reference driven through the same flat calls (by-value underneath)."""
    nx, ny = 640, 480
    syn = pkg.synthetic
    cost1 = syn.smooth_cost_map(ny, nx, seed=8)
    cost2 = syn.smooth_cost_map(ny, nx, seed=9)
    ob = (cost1 <= 0) | (cost2 <= 0)             # setCostMap only ever adds obstacles (G.cpp:118-123)
    gi, gj = syn.free_interior_cell_near(ob, 500, 300)
    si, sj = syn.free_interior_cell_near(ob, 60, 70)
    out = []
    for p in _pair(pkg, ref_planner, 1, nx, ny):
        T = np.full((ny, nx), 7.0)
        assert p.setCostMapFlat(cost1)           # no goal yet: plain upload
        assert p.setGoal(gi, gj)
        assert p.setTotalCostMatrixTarget(T)
        assert p.computeEntireTotalCostMap()
        path1 = p.getPath(si, sj)
        assert p.getTotalCostMatrixFlat(T)
        T1 = T.copy()
        assert p.setCostMapFlat(cost2)           # goal in place: streamed behind the solve
        assert p.computeEntireTotalCostMap()
        path2 = p.getPath(si, sj)
        assert p.getTotalCostMatrixFlat(T)
        T2 = T.copy()
        other = np.empty((ny, nx))
        assert p.getTotalCostMatrixFlat(other)   # a different buffer: plain download
        assert np.array_equal(other, T2)
        assert np.array_equal(p.getTotalCostMatrix(), T2)
        # a streamed upload that is consumed by something else than the solve
        assert p.setCostMapFlat(cost1)
        c = p.getGlobalCostMatrix()
        out.append((T1, path1, T2, path2, c, p.node_field(4)))
        assert p.setTotalCostMatrixTarget(None)
    a, b = out
    for k in (0, 2):
        assert np.array_equal(a[k] < 0, b[k] < 0)
        assert rel_err(b[k], a[k]) <= TOL_PLANE
    assert rel_err(b[2], b[0]) > 1e-3            # the second map did change the result
    for k in (1, 3):
        assert a[k].shape == b[k].shape and np.max(np.abs(a[k][:, :2] - b[k][:, :2])) <= TOL_WP
    assert rel_err(b[4], a[4]) <= 1e-14 and np.array_equal(a[5], b[5])


def test_streamed_cost_map_invalid_goal(pkg):
    """A cost map that turns the goal into an obstacle while its upload is streamed: the solve
    reports it (G.cpp:447-451) instead of propagating from an obstacle."""
    n = 256
    cost = np.ones((n, n))
    p = sc.make_planner(pkg.DyMuPathPlanner, 1, n, n)
    assert p.setCostMap(cost) and p.setGoal(100, 120) and p.computeEntireTotalCostMap()
    bad = cost.copy()
    bad[118:123, 98:103] = 0.0
    assert p.setCostMapFlat(bad)
    assert not p.computeEntireTotalCostMap()
    assert not p.computeEntireTotalCostMap()     # and again through the settled (non-streamed) path


def _repair_at(p, syn, path, k0, seed):
    """A frame centred on path[k0] with an obstacle disc on the path 1.2 m ahead (+2 random discs)."""
    c = path[k0, :2]
    d = path[min(k0 + 12, len(path) - 2), :2]
    rng = np.random.default_rng(seed)
    discs = [(d[0], d[1], 0.8)] + [(c[0] + rng.uniform(-4, 4), c[1] + rng.uniform(-4, 4), rng.uniform(0.2, 0.5))
                                   for _ in range(2)]
    img = syn.obstacle_frame(120, 120, 0.1, c, discs)
    repaired, traj, _ = p.computeLocalPlanning(c[0], c[1], img, 0.1)
    return dict(repaired=repaired, traj=traj, centre=c, risk=p.getRiskMatrix(c[0], c[1]),
                deviation=p.getDeviationMatrix(c[0], c[1]), reconnecting_index=p.getReconnectingIndex())


@pytest.mark.parametrize("approach", [1, 0])
def test_local_window_grows_and_keeps_obstacles(pkg, ref_planner, approach, monkeypatch):
    """The reference's local layer is unbounded and never forgets (L.cpp:150-156, G.cpp:36).  With a
    device window of only 16 global nodes the first frame does not fit (the window is re-created
    larger), the local wave runs into its border (it is doubled and the march repeated), and a
    second repair 40 m further along the path makes it grow to the union -- the obstacles and the
    risk of the first repair must still be there, as in the reference."""
    monkeypatch.setenv("DYMU_LOCAL_WINDOW", "16")
    n, syn = 300, pkg.synthetic
    res = []
    for p in _pair(pkg, ref_planner, approach, n, n):
        g = sc.global_scenario(p, syn, n, n, seed=5, entire=True)
        r1 = _repair_at(p, syn, g["path"], 0, seed=21)
        path = p.current_path
        k1 = int(np.argmax(np.hypot(path[:, 0] - r1["centre"][0], path[:, 1] - r1["centre"][1]) > 40.0))
        assert k1 > 0
        r2 = _repair_at(p, syn, path, k1, seed=22)
        back = p.getRiskMatrix(r1["centre"][0], r1["centre"][1])      # first site, after the second repair
        res.append((r1, r2, back, p.node_field(6), p.getHazardDensityMatrix(), p.getTrafficabilityMatrix()))
    (a1, a2, aback, ha, hza, tra), (b1, b2, bback, hb, hzb, trb) = res
    for a, b in ((a1, b1), (a2, b2)):
        assert a["repaired"] and b["repaired"]
        assert np.array_equal(a["risk"] > 0, b["risk"] > 0) and np.array_equal(a["risk"] == 1.0, b["risk"] == 1.0)
        assert np.max(np.abs(a["risk"] - b["risk"])) <= 1e-12
        assert np.array_equal(a["deviation"] < 0, b["deviation"] < 0)
        assert rel_err(b["deviation"], a["deviation"]) <= TOL_PLANE
        assert a["reconnecting_index"] == b["reconnecting_index"]
        assert a["traj"].shape == b["traj"].shape
        assert np.max(np.abs(a["traj"][:, :2] - b["traj"][:, :2])) <= TOL_WP
    assert (aback == 1.0).any(), "the first site's obstacles are inside the tap"
    assert np.array_equal(aback > 0, bback > 0) and np.max(np.abs(aback - bback)) <= 1e-12
    assert np.array_equal(ha, hb), "hasLocalMap"
    assert np.max(np.abs(hza - hzb)) <= 1e-12 and np.max(np.abs(tra - trb)) <= 1e-9


def test_two_repairs_with_incremental_resolve(pkg, ref_planner):
    """SURVEY.md section 8 row f2: repair -> trafficability / hazard feedback -> total-cost map
    again -> new path -> second repair.  The reference solves from scratch each time; the drop-in
    re-propagates only the dependency cone of the changed nodes (dymu_solve_incremental)."""
    n, syn = 400, pkg.synthetic
    res = []
    for p in _pair(pkg, ref_planner, 1, n, n):
        g = sc.global_scenario(p, syn, n, n, seed=9, entire=True)
        r1 = _repair_at(p, syn, g["path"], 0, seed=31)
        assert p.computeEntireTotalCostMap()                   # feedback -> re-solve
        T1 = p.getTotalCostMatrix()
        path = p.getPath(*g["path"][0, :2])
        k1 = int(np.argmax(np.hypot(path[:, 0] - path[0, 0], path[:, 1] - path[0, 1]) > 25.0))
        r2 = _repair_at(p, syn, path, k1, seed=32)
        assert p.computeTotalCostMap(*path[k1, :2])
        res.append((r1, T1, path, r2, p.getTotalCostMatrix(), p.node_field(5), p.getTrafficabilityMatrix()))
    a, b = res
    assert rel_err(b[6], a[6]) <= 1e-9 and (a[6] < 1.0).any(), "trafficability feedback"
    assert np.array_equal(a[1] < 0, b[1] < 0) and rel_err(b[1], a[1]) <= TOL_PLANE
    assert a[2].shape == b[2].shape and np.max(np.abs(a[2][:, :2] - b[2][:, :2])) <= TOL_WP
    closed = a[5] > 0                                          # early stop: parity on the CLOSED set
    assert np.array_equal(closed, b[5] > 0), "CLOSED set after the second re-solve"
    assert rel_err(np.where(closed, b[4], 0), np.where(closed, a[4], 0)) <= TOL_PLANE
    for k in (0, 3):
        assert a[k]["repaired"] == b[k]["repaired"]
        assert a[k]["traj"].shape == b[k]["traj"].shape
        assert np.max(np.abs(a[k]["traj"][:, :2] - b[k]["traj"][:, :2])) <= TOL_WP
