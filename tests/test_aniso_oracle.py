"""The plain-C restatement of the slope-anisotropic solve (oracle/dymu_oracle_aniso.c) against
closed forms and against the isotropic restatement.  No GPU needed."""
import math

import numpy as np
import pytest

TABLE = ([-20.0, 0.0, 20.0], [0.5, 1.0, 3.0])


@pytest.fixture(scope="module")
def orc_aniso():
    """The plain-C restatement of the anisotropic model (built on first use)."""
    import oracle_aniso
    return oracle_aniso


def _ceff(port, gres=1.0):
    """C_eff of G.cpp:527-528 from the restatement's planes, +inf on obstacles."""
    cost = port.plane("cost")
    haz, traff = port.plane("hazard_density"), port.plane("trafficability")
    c = gres * cost * (2 + haz - traff)
    c[port.plane("isObstacle") != 0] = np.inf
    return c


@pytest.mark.parametrize("seed", [3, 11])
def test_flat_table_equals_isotropic_heap(oracle_mod, orc_aniso, pkg, seed):
    syn = pkg.synthetic
    nx, ny = 97, 61
    p = oracle_mod.Port(1.0, 1.5, 2.0, 0)
    assert p.initGlobalLayer(1.0, 0.1, nx, ny)
    elev, terr = syn.mars_dem(ny, nx, seed=seed)
    lut, slopes, locs = syn.default_lut()
    assert p.computeCostMap(lut, slopes, locs, elev, terr)
    ob = p.plane("isObstacle")
    gi, gj = syn.free_interior_cell_near(ob, nx // 3, ny // 2)
    assert p.setGoal(float(gi), float(gj))
    assert p.computeEntireTotalCostMap(heap=True)
    T_iso = p.plane("total_cost")
    A = orc_aniso.aniso_dircost(elev, _ceff(p), 1.0, [-90.0, 90.0], [1.0, 1.0])
    assert np.array_equal(np.isinf(A[0]), np.isinf(_ceff(p)) | (np.arange(nx) == 0)[None, :])
    T = orc_aniso.aniso_march(A, (gi, gj))
    assert np.array_equal(np.isinf(T), np.isinf(T_iso))
    r = np.isfinite(T) & (T_iso > 0)
    assert np.max(np.abs(T[r] - T_iso[r]) / T_iso[r]) <= 1e-13


def _corridor(n=41, slope_deg=10.0, c=0.7):
    """A one-cell-wide corridor along x (row 1) between two obstacle rows on a uniform incline."""
    elev = np.tile(np.arange(n, dtype=np.float64) * math.tan(math.radians(slope_deg)), (3, 1))
    ceff = np.full((3, n), np.inf)
    ceff[1, :] = c
    return elev, ceff


def _f(theta):
    return float(np.interp(theta, TABLE[0], TABLE[1]))


def test_corridor_is_the_running_sum(orc_aniso):
    n, c, goal = 41, 0.7, 20
    elev, ceff = _corridor(n, 10.0, c)
    A = orc_aniso.aniso_dircost(elev, ceff, 1.0, *TABLE)
    th = math.degrees(math.atan(math.tan(math.radians(10.0))))
    up, down = c * _f(th), c * _f(-th)
    assert A[1, 1, 5] == pytest.approx(up, rel=1e-14) and A[0, 1, 5] == pytest.approx(down, rel=1e-14)
    assert np.isinf(A[:, 0, :]).all() and np.isinf(A[:, 2, :]).all()
    assert np.isinf(A[0, 1, 0]) and np.isinf(A[1, 1, n - 1])
    T = orc_aniso.aniso_march(A, (goal, 1))
    assert np.isinf(T[0]).all() and np.isinf(T[2]).all()
    expect = np.zeros(n)
    for i in range(goal + 1, n):      # above the goal the rover drives downhill toward it
        expect[i] = expect[i - 1] + down
    for i in range(goal - 1, -1, -1):  # below it, uphill
        expect[i] = expect[i + 1] + up
    r = expect > 0
    assert np.max(np.abs(T[1, r] - expect[r]) / expect[r]) <= 1e-12
    for d in (1, 7, 20):
        assert T[1, goal - d] / T[1, goal + d] == pytest.approx(_f(th) / _f(-th), rel=1e-12)


def test_march_is_a_fixed_point(orc_aniso, pkg):
    syn = pkg.synthetic
    nx, ny = 83, 77
    elev, _ = syn.mars_dem(ny, nx, seed=5)
    cost = syn.smooth_cost_map(ny, nx, seed=5)
    ceff = np.where(cost > 0, cost * 2.0, np.inf)
    A = orc_aniso.aniso_dircost(elev, ceff, 1.0, *TABLE)
    goal = syn.free_interior_cell_near(cost <= 0, nx // 2, ny // 2)
    T = orc_aniso.aniso_march(A, goal)
    assert np.isfinite(T).mean() > 0.8
    assert orc_aniso.aniso_improvable(A, T, goal, 1e-14) == 0
    # a perturbed plane is not: lowering one reached cell makes its neighbours improvable
    T2 = T.copy()
    j, i = np.argwhere(np.isfinite(T) & (T > 5))[0]
    T2[j, i] *= 0.5
    assert orc_aniso.aniso_improvable(A, T2, goal, 1e-14) > 0


def test_descent_reaches_the_goal(orc_aniso, pkg):
    syn = pkg.synthetic
    nx, ny = 90, 70
    elev, _ = syn.mars_dem(ny, nx, seed=4)
    cost = syn.smooth_cost_map(ny, nx, seed=4)
    ceff = np.where(cost > 0, cost * 2.0, np.inf)
    A = orc_aniso.aniso_dircost(elev, ceff, 1.0, [-30.0, 0.0, 30.0], [0.8, 1.0, 1.6])
    goal = syn.free_interior_cell_near(cost <= 0, 70, 50)
    start = syn.free_interior_cell_near(cost <= 0, 12, 10)
    T = orc_aniso.aniso_march(A, goal)
    wps, status = orc_aniso.aniso_path(A, T, elev, 1.0, start, 0.4, goal)
    assert status == 0 and len(wps) > 10 and np.isfinite(wps).all()
    assert np.hypot(wps[-1, 0] - goal[0], wps[-1, 1] - goal[1]) < 3.0
