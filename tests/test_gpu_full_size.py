"""Parity at BASELINE.json's full sizes through properties that do not need the (hours-long)
reference run:

* the converged plane is the fixed point of propagateGlobalNode (G.cpp:500-546): evaluated in
  numpy in the reference's operation order on all 16.7 M cells, the update expression improves
  no cell (exactly), and reproduces every reached cell from its four current neighbours to
  within rounding (a neighbour that decreased after a cell's last update can move the
  expression by an ulp or two -- floating-point evaluation is not exactly monotone -- which is
  also true of the reference's own result);
* re-activating every tile changes nothing (idempotence);
* the result does not depend on the schedule beyond rounding: a goal solved inside a batch of
  goals agrees with the same goal solved alone to 1e-13 with the same reached set;
* the total cost decreases strictly along the extracted path and the path ends at the goal."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _update_expression(T, C):
    """G.cpp:527-535 on whole planes: Tn(i,j) from the 4 neighbours, +inf outside the grid."""
    P = np.pad(T, 1, constant_values=np.inf)
    Tx = np.minimum(P[1:-1, :-2], P[1:-1, 2:])
    Ty = np.minimum(P[:-2, 1:-1], P[2:, 1:-1])
    del P
    with np.errstate(invalid="ignore", over="ignore"):
        d = Tx - Ty
        two = np.abs(d) < C
        t2 = (Tx + Ty + np.sqrt(np.where(two, 2 * (C * C) - d * d, 1.0))) / 2
        t1 = np.minimum(Tx, Ty) + C
    return np.where(two, t2, t1)


def _plan(pkg, n, seed=20261018):
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(n, n, seed=seed)
    lut, slopes, locs = syn.default_lut()
    dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    dev.compute_cost_map(lut, slopes, len(locs), elev, terr)
    ob = dev.download_plane_u8("obstacle")
    return dev, ob


def test_plan4096_is_the_exact_fixed_point(pkg):
    n = 4096
    dev, ob = _plan(pkg, n)
    goal = pkg.synthetic.free_interior_cell_near(ob, n // 2, n // 2)
    st = dev.solve_total_cost([goal])
    assert st["converged"]
    T = dev.download_total_cost()
    C = dev.download_plane("ceff")
    assert np.array_equal(np.isinf(C), ob != 0)
    reached = np.isfinite(T)
    assert 0.9 <= reached.mean() <= 1.0 and not reached[ob != 0].any()
    assert T[goal[1], goal[0]] == 0.0 and (T[reached] >= 0).all()
    Tn = _update_expression(T, C)
    interior = reached.copy()
    interior[goal[1], goal[0]] = False
    # no target cell can still be improved: exact (the kernel's update is bit-identical to this one)
    target = np.isfinite(C)
    with np.errstate(invalid="ignore"):
        assert not (Tn[target] < T[target]).any()
    # and every reached cell is reproduced by its current neighbours up to rounding
    gap = (Tn[interior] - T[interior]) / T[interior]
    print("cells off by rounding: %d of %d, largest relative gap %.3e" %
          (np.count_nonzero(gap), gap.size, gap.max()))
    assert gap.min() >= 0.0 and gap.max() <= 1e-14
    assert np.count_nonzero(gap) <= 0.02 * gap.size
    del Tn
    # idempotence: waking every tile again leaves the plane bit-identical
    again = dev.solve_advance([(0, n)], 0.0, 1 << 20)
    assert again["converged"] and again["tile_activations"] >= (n // 32) ** 2
    assert np.array_equal(dev.download_total_cost(), T)
    # the path descends strictly and arrives
    start = pkg.synthetic.free_interior_cell_near(ob, n // 16, n // 16)
    wps, status = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, goal[0], goal[1])
    assert status == 0 and len(wps) > n // 2
    ij = np.rint(wps[:, :2]).astype(np.int64)
    t_along = T[ij[:, 1], ij[:, 0]]
    assert np.isfinite(t_along).all()
    assert t_along[-1] <= 4 * C[np.isfinite(C)].max()          # within two cells of the goal
    coarse = t_along[::25]
    assert (np.diff(coarse) < 0).all()
    assert np.hypot(wps[-1, 0] - goal[0], wps[-1, 1] - goal[1]) <= 2.0 + 0.4


def test_queries2048_batch_is_schedule_independent(pkg):
    n = 2048
    dev, ob = _plan(pkg, n)
    rng = np.random.default_rng(11)
    goals = [pkg.synthetic.free_interior_cell_near(ob, int(rng.uniform(0.1, 0.9) * n),
                                                   int(rng.uniform(0.1, 0.9) * n)) for _ in range(8)]
    dev.reserve_slots(8)
    st = dev.solve_total_cost(goals)
    assert st["converged"]
    batch = [dev.download_total_cost(slot=q) for q in (0, 3, 7)]
    for q, Tb in zip((0, 3, 7), batch):
        dev.solve_total_cost([goals[q]])
        Ts = dev.download_total_cost(slot=0)
        assert np.array_equal(np.isinf(Ts), np.isinf(Tb)), "goal %d" % q
        fin = np.isfinite(Tb) & (Tb > 0)
        assert np.max(np.abs(Ts[fin] - Tb[fin]) / Tb[fin]) <= 1e-13, "goal %d" % q


def _heap_port(oracle_mod, pkg, n, goal, seed=20261018):
    """The pinned C port (bit-exact against the unmodified reference at <= 1000^2,
    tests/test_oracle_vs_reference.py) with a binary heap instead of the reference's linear
    narrow-band scan: same update expression, same values, seconds instead of an hour."""
    syn = pkg.synthetic
    elev, terr = syn.mars_dem(n, n, seed=seed)
    lut, slopes, locs = syn.default_lut()
    po = oracle_mod.Port(1.0, 1.5, 2.0, 1)
    assert po.initGlobalLayer(1.0, 0.1, n, n)
    assert po.computeCostMap(lut, slopes, locs, elev, terr)
    assert po.setGoal(*goal)
    assert po.computeEntireTotalCostMap(heap=True)
    T = po.plane("total_cost").copy()
    ob = po.plane("isObstacle").copy()
    po.close()
    return T, ob


def test_plan4096_matches_heap_port(pkg, oracle_mod):
    """The headline configuration (bench.py's map, goal and seed) compared cell by cell."""
    n = 4096
    dev, ob = _plan(pkg, n)
    goal = pkg.synthetic.free_interior_cell_near(ob, n // 2, n // 2)
    assert dev.solve_total_cost([goal])["converged"]
    T = dev.download_total_cost()
    To, obo = _heap_port(oracle_mod, pkg, n, goal)
    assert np.array_equal(obo != 0, ob != 0), "obstacle mask"
    assert np.array_equal(np.isinf(T), np.isinf(To)), "unreached set"
    fin = np.isfinite(To) & (To > 0)
    err = np.max(np.abs(T[fin] - To[fin]) / To[fin])
    print("4096^2 vs heap port: max rel err %.3e, bit-equal cells %.4f" % (err, (T == To).mean()))
    assert err <= 1e-9


def test_query2048_matches_heap_port(pkg, oracle_mod):
    """One query of config 4 (2048^2 map, goal drawn like bench.py draws them, solved inside a
    batch of 8) against the heap port."""
    n = 2048
    dev, ob = _plan(pkg, n)
    rng = np.random.default_rng(11)
    goals = [pkg.synthetic.free_interior_cell_near(ob, int(rng.uniform(0.03, 0.97) * n),
                                                   int(rng.uniform(0.03, 0.97) * n)) for _ in range(8)]
    dev.reserve_slots(8)
    assert dev.solve_total_cost(goals)["converged"]
    T = dev.download_total_cost(slot=5)
    To, _ = _heap_port(oracle_mod, pkg, n, goals[5])
    assert np.array_equal(np.isinf(T), np.isinf(To))
    fin = np.isfinite(To) & (To > 0)
    assert np.max(np.abs(T[fin] - To[fin]) / To[fin]) <= 1e-9
