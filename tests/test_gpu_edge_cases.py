"""Edge cases of the class interface, each run on the reference (tests/conftest.py::ref_planner) and
on the B200 drop-in with identical calls."""
import numpy as np
import pytest

import scenarios as sc
from conftest import rel_err

pytestmark = pytest.mark.gpu


def _both(pkg, ref, approach=1, nx=64, ny=64, gres=1.0, lres=0.1, offset=(0.0, 0.0)):
    out = []
    for f in (ref, pkg.DyMuPathPlanner):
        p = f(1.0, 1.5, 2.0, approach)
        assert p.initGlobalLayer(gres, lres, nx, ny, offset)
        out.append(p)
    return out


def test_non_unit_global_resolution(pkg, ref_planner):
    """global_res = 2.5 m: goal/start conversion, C = res*cost, path step res*tau (G.cpp:326-333,
    527, 706)."""
    nx, ny, gres = 90, 70, 2.5
    cost = pkg.synthetic.smooth_cost_map(ny, nx, seed=3)
    res = []
    for p in _both(pkg, ref_planner, nx=nx, ny=ny, gres=gres, lres=0.25):
        assert p.setCostMap(cost)
        ob = sc.obstacle_plane(p)
        gi, gj = pkg.synthetic.free_interior_cell_near(ob, 70, 50)
        si, sj = pkg.synthetic.free_interior_cell_near(ob, 15, 15)
        assert p.setGoal(gi * gres, gj * gres)
        assert p.computeEntireTotalCostMap()
        res.append((p.getTotalCostMatrix(), p.getPath(si * gres, sj * gres)))
    (Ta, pa), (Tb, pb) = res
    assert np.array_equal(Ta < 0, Tb < 0) and rel_err(Tb, Ta) <= 1e-9
    assert pa.shape == pb.shape
    assert np.max(np.abs(pa[:, :2] - pb[:, :2])) <= 1e-3 * gres


@pytest.mark.parametrize("nx,ny", [(5, 7), (33, 31), (32, 32), (65, 3 + 32)])
def test_small_and_ragged_grids(pkg, ref_planner, nx, ny):
    cost = 1.0 + np.arange(nx * ny, dtype=np.float64).reshape(ny, nx) % 7 * 0.25
    res = []
    for p in _both(pkg, ref_planner, nx=nx, ny=ny):
        assert p.setCostMap(cost)
        assert p.setGoal(nx // 2, ny // 2)
        assert p.computeEntireTotalCostMap()
        res.append(p.getTotalCostMatrix())
    assert np.array_equal(res[0] < 0, res[1] < 0)
    assert rel_err(res[1], res[0]) <= 1e-9


def test_replanning_with_a_new_goal_resets_the_map(pkg, ref_planner):
    nx = ny = 96
    cost = pkg.synthetic.smooth_cost_map(ny, nx, seed=12)
    res = []
    for p in _both(pkg, ref_planner, nx=nx, ny=ny):
        assert p.setCostMap(cost)
        ob = sc.obstacle_plane(p)
        g1 = pkg.synthetic.free_interior_cell_near(ob, 20, 20)
        g2 = pkg.synthetic.free_interior_cell_near(ob, 75, 70)
        assert p.setGoal(*g1) and p.computeEntireTotalCostMap()
        T1 = p.getTotalCostMatrix()
        assert p.setGoal(*g2) and p.computeEntireTotalCostMap()
        res.append((T1, p.getTotalCostMatrix()))
    for k in (0, 1):
        assert np.array_equal(res[0][k] < 0, res[1][k] < 0)
        assert rel_err(res[1][k], res[0][k]) <= 1e-9


def test_walled_in_start_is_unreachable(pkg, ref_planner):
    """computeTotalCostMap returns false when the wave cannot close the start (G.cpp:399-403)."""
    nx = ny = 64
    cost = np.ones((ny, nx))
    cost[20:41, 20] = cost[20:41, 40] = cost[20, 20:41] = cost[40, 20:41] = 0.0   # closed box
    for p in _both(pkg, ref_planner, nx=nx, ny=ny):
        assert p.setCostMap(cost)
        assert p.setGoal(10.0, 10.0)
        assert not p.computeTotalCostMap(30.0, 30.0)   # inside the box
        assert p.computeTotalCostMap(50.0, 50.0)
        T = p.getTotalCostMatrix()
        assert np.all(T[22:39, 22:39] == -1.0)


def test_frame_without_obstacles_and_frame_partly_outside(pkg, ref_planner):
    nx = ny = 80
    syn = pkg.synthetic
    res = []
    for p in _both(pkg, ref_planner, nx=nx, ny=ny):
        g = sc.global_scenario(p, syn, nx, ny, seed=4, entire=True, goal_frac=(0.8, 0.8),
                               start_frac=(0.1, 0.1))
        path = g["path"]
        empty = np.zeros((100, 100), dtype=np.uint8)
        rep0, traj0, _ = p.computeLocalPlanning(path[0, 0], path[0, 1], empty, 0.1)
        # a frame centred near the map corner: most pixels fall outside the map (L.cpp:239-241)
        img = np.zeros((120, 120), dtype=np.uint8)
        img[40:60, 40:60] = 1
        rep1, traj1, _ = p.computeLocalPlanning(2.0, 2.0, img, 0.1)
        res.append((rep0, len(traj0), rep1, p.getRiskMatrix(2.0, 2.0), p.getHazardDensityMatrix(),
                    p.node_field(6)))
    a, b = res
    assert a[0] == b[0] and a[1] == b[1] and a[2] == b[2]
    assert np.array_equal(a[3] > 0, b[3] > 0)
    assert np.max(np.abs(a[3] - b[3])) <= 1e-12
    assert np.max(np.abs(a[4] - b[4])) <= 1e-12
    assert np.array_equal(a[5], b[5])


@pytest.mark.parametrize("approach", [1, 0])
def test_two_consecutive_frames(pkg, ref_planner, approach):
    """Obstacles seen first off the path (no repair, expansion deferred: L.cpp:278), then a
    second frame that blocks the path: the deferred obstacles must be dilated too."""
    n, syn = 160, pkg.synthetic
    res = []
    for p in _both(pkg, ref_planner, approach=approach, nx=n, ny=n):
        g = sc.global_scenario(p, syn, n, n, seed=9, entire=True)
        path = g["path"]
        c = path[0, :2]
        off = syn.obstacle_frame(120, 120, 0.1, c, [(c[0] - 4.0, c[1] + 4.5, 0.4)])
        rep0, _, _ = p.computeLocalPlanning(c[0], c[1], off, 0.1)
        d = path[14, :2]
        blk = syn.obstacle_frame(120, 120, 0.1, c, [(d[0], d[1], 0.7)])
        rep1, traj, _ = p.computeLocalPlanning(c[0], c[1], blk, 0.1)
        res.append((rep0, rep1, traj, p.getRiskMatrix(c[0], c[1]), p.getDeviationMatrix(c[0], c[1]),
                    p.getReconnectingIndex()))
    a, b = res
    assert a[0] == b[0] and a[1] == b[1] and a[5] == b[5]
    assert np.array_equal(a[3] > 0, b[3] > 0) and np.max(np.abs(a[3] - b[3])) <= 1e-12
    assert np.array_equal(a[4] < 0, b[4] < 0) and rel_err(b[4], a[4]) <= 1e-9
    assert a[2].shape == b[2].shape
    if len(a[2]):
        assert np.max(np.abs(a[2][:, :2] - b[2][:, :2])) <= 1e-3


def test_total_cost_queries_and_node_views(pkg, ref_planner):
    nx = ny = 72
    cost = pkg.synthetic.smooth_cost_map(ny, nx, seed=6)
    vals = []
    for p in _both(pkg, ref_planner, nx=nx, ny=ny, offset=(3.0, -2.0)):
        assert p.setCostMap(cost)
        ob = sc.obstacle_plane(p)
        gi, gj = pkg.synthetic.free_interior_cell_near(ob, 50, 50)
        assert p.setGoal(gi + 3.0, gj - 2.0) and p.computeEntireTotalCostMap()
        vals.append([p.getTotalCost(x + 3.0, y - 2.0) for x, y in
                     ((10.2, 11.7), (35.5, 20.25), (60.9, 66.1), (gi + 0.3, gj + 0.4))])
    a, b = np.array(vals[0]), np.array(vals[1])
    fin = np.isfinite(a)
    assert np.array_equal(fin, np.isfinite(b))
    assert np.max(np.abs(a[fin] - b[fin]) / np.maximum(1e-300, np.abs(a[fin]))) <= 1e-9


def test_node_level_forwards(pkg, ref_lib):
    """gradientNode, computeNextGlobalWaypoint and propagateGlobalNode (H.hpp:520-536) called from
    outside, on the reference's pointer graph and on the drop-in's node views."""
    nx, ny = 96, 80
    elev, terr = pkg.synthetic.mars_dem(ny, nx, seed=7)      # (setCostMap alone leaves the reference's
    lut, slopes, locs = pkg.synthetic.default_lut()          #  elevation uninitialised, H.hpp:95)
    out = []
    for p in _both(pkg, ref_lib.DyMuPathPlanner, nx=nx, ny=ny):
        assert p.computeCostMap(lut, slopes, locs, elev, terr)
        ob = sc.obstacle_plane(p)
        gi, gj = pkg.synthetic.free_interior_cell_near(ob, 70, 60)
        assert p.setGoal(gi, gj) and p.computeEntireTotalCostMap()
        T = p.getTotalCostMatrix()
        rec = []
        # (the reference dereferences a missing neighbour when the other one is unreached,
        # G.cpp:729-731: border nodes next to the obstacle rim cannot be asked there)
        for (i, j) in ((40, 30), (gi, gj), (gi + 1, gj), (17, 63), (3, 3), (nx - 4, ny - 4)):
            rec.append(p.gradientNode(i, j))
        # next to an unreached / obstacle cell: one-sided differences
        jj, ii = np.nonzero(T < 0)
        for k in range(0, len(ii), max(1, len(ii) // 6)):
            if 1 < ii[k] < nx - 3 and 1 < jj[k] < ny - 2:
                rec.append(p.gradientNode(int(ii[k]) + 1, int(jj[k])))
        steps = [p.computeNextGlobalWaypoint(x, y, 0.4) for x, y in ((20.3, 15.8), (60.0, 40.0), (gi - 3.2, gj + 2.1))]
        # a converged node cannot be improved; a node whose value is raised by hand comes back down
        same = p.propagateGlobalNode(40, 30)
        out.append((rec, steps, same, T[30, 40]))
        assert p.gradientNode(nx + 5, 3) is None
    (ra, sa, ta, Ta), (rb, sb, tb, Tb) = out
    assert len(ra) == len(rb)
    for a, b in zip(ra, rb):
        assert np.allclose(a, b, rtol=0, atol=1e-9, equal_nan=True), (a, b)
    for a, b in zip(sa, sb):
        assert np.max(np.abs(a[:2] - b[:2])) <= 1e-9 and abs(a[3] - b[3]) <= 1e-9
        assert abs(np.angle(np.exp(1j * (a[2] - b[2])))) <= 1e-9
    assert ta == pytest.approx(Ta, rel=1e-12) and tb == pytest.approx(Tb, rel=1e-12)
