"""Batches of independent cost maps (dymu_reserve_maps / dymu_set_maps / dymu_solve_maps /
dymu_batch_solve_maps): each map of a batch against a freshly created context solving that map alone,
against the reference, the fixed point, paths, device input, isolation from the context's own state,
errors and the multi-context driver."""
import numpy as np
import pytest

import scenarios as sc
from conftest import rel_err

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -2, -3


def _ceff(cost, g=1.0):
    """The model: C_eff of a fresh context after dymu_set_cost_map(cost)."""
    with np.errstate(over="ignore"):
        return np.where(cost <= 0, np.inf, g * cost * (2 + 0.0 - 1.0))


def _goal(pkg, cost, fi, fj):
    ny, nx = cost.shape
    return pkg.synthetic.free_interior_cell_near(cost <= 0, int(fi * nx), int(fj * ny))


def _batch(pkg, ny, nx, n, seed):
    """n maps with different crater layouts and goals; map 1 is scaled x100 (a mixed band), map 2 has
    its goal on an obstacle, map 3 walls its goal into a pocket."""
    rng = np.random.default_rng(seed)
    costs = np.stack([pkg.synthetic.smooth_cost_map(ny, nx, seed=seed * 100 + q) for q in range(n)])
    goals = [_goal(pkg, costs[q], rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8)) for q in range(n)]
    costs[1] *= 100.0
    gi, gj = goals[2]
    costs[2, gj, gi] = 0.0
    gi, gj = goals[3]
    r = max(3, min(nx, ny) // 8)
    i0, i1, j0, j1 = max(gi - r, 0), min(gi + r, nx - 1), max(gj - r, 0), min(gj + r, ny - 1)
    costs[3, j0, i0:i1 + 1] = costs[3, j1, i0:i1 + 1] = 0.0
    costs[3, j0:j1 + 1, i0] = costs[3, j0:j1 + 1, i1] = 0.0
    pocket = np.zeros((ny, nx), bool)
    pocket[j0 + 1:j1, i0 + 1:i1] = True
    return costs, goals, pocket


def _solo(pkg, cost, goal, start=None, g=1.0):
    ny, nx = cost.shape
    dev = pkg.cuda_api.DeviceLayer(nx, ny, g, 0.1)
    try:
        dev.set_cost_map(cost)
        st = dev.solve_total_cost([goal])
        T = dev.download_total_cost()
        path = None
        if start is not None:
            path = dev.extract_global_path(float(start[0]), float(start[1]), 0.4, goal[0], goal[1], cap=1 << 14)
        return T, st, path
    finally:
        dev.close()


def _same(Tb, Ts, tol=1e-12):
    assert np.array_equal(np.isfinite(Tb), np.isfinite(Ts))
    assert rel_err(Tb, Ts) <= tol


def _snake(ny, nx, rng):
    """A one-cell-wide serpentine corridor: every cell has one upstream neighbour, so the total cost
    is the running sum of C_eff along it, whatever the order of updates (exact, bit for bit)."""
    cost = np.zeros((ny, nx))
    cost[0::2, :] = rng.uniform(0.05, 3.0, (len(range(0, ny, 2)), nx))
    for j in range(1, ny - 1, 2):
        i = nx - 1 if (j // 2) % 2 == 0 else 0
        cost[j, i] = rng.uniform(0.05, 3.0)
    if ny % 2 == 0:
        cost[ny - 1, :] = 0.0
    return cost


def _snake_T(cost, g):
    """Running sum of C_eff along the snake from cell (0, 0) in the expression order of the update."""
    ny, nx = cost.shape
    C = _ceff(cost, g)
    T = np.full((ny, nx), np.inf)
    t = 0.0
    order = []
    for j in range(ny):
        if j % 2 == 0:
            row = range(nx) if (j // 2) % 2 == 0 else range(nx - 1, -1, -1)
            order += [(j, i) for i in row if cost[j, i] > 0]
        else:
            order += [(j, i) for i in range(nx) if cost[j, i] > 0]
    for k, (j, i) in enumerate(order):
        t = 0.0 if k == 0 else t + C[j, i]
        T[j, i] = t
    return T


# ---- 1. batch equals solo --------------------------------------------------------------------------
@pytest.mark.parametrize("ny,nx,n", [(129, 257, 10), (100, 100, 8), (512, 512, 16)])
def test_batch_equals_solo(pkg, ny, nx, n):
    costs, goals, pocket = _batch(pkg, ny, nx, n, seed=ny + nx)
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.reserve_maps(n)
    dev.set_maps(costs)
    st = dev.solve_maps(goals)
    assert st["converged"] and st["goal_obstacle"] == 1
    for q in range(n):
        Tb = dev.download_total_cost(slot=q)
        Ts, sts, _ = _solo(pkg, costs[q], goals[q])
        _same(Tb, Ts)
        if q == 2:
            assert sts["goal_obstacle"] == 1 and not np.isfinite(Tb).any()
        else:
            assert Tb[goals[q][1], goals[q][0]] == 0.0 and dev.count_reached(slot=q) == np.isfinite(Ts).sum()
        if q == 3:
            assert np.isfinite(Tb).any() and not np.isfinite(Tb[~pocket]).any()


# ---- 2. against the reference ---------------------------------------------------------------------
def test_maps_match_reference(pkg, ref_planner):
    n = 100
    costs = np.stack([pkg.synthetic.smooth_cost_map(n, n, seed=s) for s in (1, 5, 9)])
    goals = [_goal(pkg, costs[0], 0.8, 0.8), _goal(pkg, costs[1], 0.3, 0.7), _goal(pkg, costs[2], 0.5, 0.2)]
    dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    dev.reserve_maps(3)
    dev.set_maps(costs)
    assert dev.solve_maps(goals)["converged"]
    for q in range(3):
        ref = sc.make_planner(ref_planner, 1, n, n)
        assert ref.setCostMap(costs[q]) and ref.setGoal(*goals[q]) and ref.computeEntireTotalCostMap()
        Tr = ref.getTotalCostMatrix()
        Tb = dev.download_total_cost(slot=q, xform=pkg.cuda_api.XFORM_INF_TO_MINUS1)
        assert np.array_equal(Tb < 0, Tr < 0)
        fin = Tr > 0
        assert float(np.max(np.abs(Tb[fin] - Tr[fin]) / Tr[fin])) <= 1e-9


# ---- 3. fixed point --------------------------------------------------------------------------------
def _update_expression(T, C):
    """G.cpp:527-535 on whole planes: Tn(i,j) from the 4 neighbours, +inf outside the grid."""
    P = np.pad(T, 1, constant_values=np.inf)
    Tx = np.minimum(P[1:-1, :-2], P[1:-1, 2:])
    Ty = np.minimum(P[:-2, 1:-1], P[2:, 1:-1])
    with np.errstate(invalid="ignore", over="ignore"):
        d = Tx - Ty
        two = np.abs(d) < C
        t2 = (Tx + Ty + np.sqrt(np.where(two, 2 * (C * C) - d * d, 1.0))) / 2
        t1 = np.minimum(Tx, Ty) + C
    return np.where(two, t2, t1)


def test_slot_is_the_exact_fixed_point(pkg):
    n = 512
    costs = np.stack([pkg.synthetic.smooth_cost_map(n, n, seed=s) for s in (31, 32, 33, 34)])
    goals = [_goal(pkg, c, f, 1 - f) for c, f in zip(costs, (0.2, 0.4, 0.6, 0.8))]
    dev = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    dev.reserve_maps(4)
    dev.set_maps(costs)
    assert dev.solve_maps(goals)["converged"]
    q = 2
    T, C = dev.download_total_cost(slot=q), _ceff(costs[q])
    ref = pkg.cuda_api.DeviceLayer(n, n, 1.0, 0.1)
    ref.set_cost_map(costs[q])
    assert np.array_equal(ref.download_plane("ceff"), C)  # the model is the fresh context's C_eff
    Tn = _update_expression(T, C)
    target = np.isfinite(C)
    with np.errstate(invalid="ignore"):
        assert not (Tn[target] < T[target]).any()
    reached = np.isfinite(T)
    reached[goals[q][1], goals[q][0]] = False
    gap = (Tn[reached] - T[reached]) / T[reached]
    assert reached.mean() > 0.5 and gap.min() >= 0.0 and gap.max() <= 1e-14


# ---- 4. paths ---------------------------------------------------------------------------------------
def test_paths_on_map_slots(pkg):
    ny, nx, n = 300, 200, 6
    costs, goals, _ = _batch(pkg, ny, nx, n, seed=7)
    starts = [_goal(pkg, costs[q], 0.1 + 0.15 * q, 0.9 - 0.1 * q) for q in range(n)]
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.reserve_maps(n)
    dev.set_maps(costs)
    dev.solve_maps(goals)
    paths, status = dev.extract_global_path_batch(list(range(n)), [(float(i), float(j)) for i, j in starts], 0.4,
                                                  goals, cap=1 << 14)
    for q in range(n):
        _, _, (ps, ss) = _solo(pkg, costs[q], goals[q], starts[q])
        assert status[q] == ss and paths[q].shape == ps.shape, q
        if len(ps):
            assert np.max(np.abs(paths[q][:, :2] - ps[:, :2])) <= 1e-3


# ---- 5. device input equals host input ----------------------------------------------------------
def test_device_input_equals_host_input(pkg):
    torch = pytest.importorskip("torch")
    ny, nx, n, g = 97, 131, 5, 0.7
    rng = np.random.default_rng(5)
    snakes = np.stack([_snake(ny, nx, rng) for _ in range(n)])
    snakes[1] *= 100.0
    ld, rows = nx + 5, ny + 3
    big = torch.full((n, rows, ld), float("nan"), dtype=torch.float64, device="cuda:0")
    big[:, :ny, :nx] = torch.from_numpy(snakes).to("cuda:0")
    torch.cuda.synchronize()
    a = pkg.cuda_api.DeviceLayer(nx, ny, g, 0.1, device=0)
    b = pkg.cuda_api.DeviceLayer(nx, ny, g, 0.1, device=0)
    for d in (a, b):
        d.reserve_maps(n)
    a.set_maps(snakes)
    b.set_maps_device(big.data_ptr(), n, ld, rows * ld)
    goals = [(0, 0)] * n
    for d in (a, b):
        assert d.solve_maps(goals)["converged"]
    for q in range(n):
        Ta, Tb = a.download_total_cost(slot=q), b.download_total_cost(slot=q)
        assert np.array_equal(Ta, Tb), q
        assert np.array_equal(Ta, _snake_T(snakes[q], g)), q
    # a general map: the same to rounding (the update order of the solver varies from run to run)
    costs, goals, _ = _batch(pkg, ny, nx, n, seed=3)
    big[:, :ny, :nx] = torch.from_numpy(costs).to("cuda:0")
    torch.cuda.synchronize()
    a.set_maps(costs)
    b.set_maps_device(big.data_ptr(), n, ld, rows * ld)
    for d in (a, b):
        d.solve_maps(goals)
    for q in range(n):
        _same(b.download_total_cost(slot=q), a.download_total_cost(slot=q), 1e-13)
    # a host pointer announced as device memory is refused
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        b.set_maps_device(costs.ctypes.data, n, nx, ny * nx)
    assert e.value.code == ERR_ARG


# ---- 6. isolation ---------------------------------------------------------------------------------
def test_context_state_is_untouched(pkg):
    torch = pytest.importorskip("torch")
    ny, nx, n = 160, 224, 4
    own = pkg.synthetic.smooth_cost_map(ny, nx, seed=77)
    goal = _goal(pkg, own, 0.5, 0.5)
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.set_cost_map(own)
    dev.solve_total_cost([goal])
    ceff, ob = dev.download_plane("ceff"), dev.download_plane_u8("obstacle")
    pinned = torch.empty((ny, nx), dtype=torch.float64).pin_memory()
    buf = pinned.numpy()
    assert dev.set_total_cost_export(buf)
    costs, goals, _ = _batch(pkg, ny, nx, n, seed=8)
    dev.reserve_maps(n)
    dev.set_maps(costs)
    for m in (1, n):
        buf[:] = 12345.0
        dev.solve_maps(goals[:m])
        dev.synchronize()
        assert (buf == 12345.0).all()
        _same(dev.download_total_cost(slot=0), _solo(pkg, costs[0], goals[0])[0], 1e-12)
    assert np.array_equal(dev.download_plane("ceff"), ceff)
    assert np.array_equal(dev.download_plane_u8("obstacle"), ob)
    st, inv = dev.solve_incremental(goal)
    assert inv is None and st["converged"]
    T_inc = dev.download_total_cost()
    dev.set_total_cost_export(None)
    dev.solve_total_cost([goal])
    _same(T_inc, dev.download_total_cost(), 1e-13)
    _same(T_inc, _solo(pkg, own, goal)[0], 1e-13)


# ---- 7. errors ---------------------------------------------------------------------------------------
def _code(pkg, call):
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        call()
    return e.value.code


def test_errors(pkg):
    ny, nx = 64, 80
    costs, goals, _ = _batch(pkg, ny, nx, 4, seed=2)
    dev = pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1)
    dev.reserve_maps(3)
    for bad in (np.nan, np.inf):
        c = costs[0].copy()
        c[10, 20] = bad
        assert _code(pkg, lambda: dev.set_maps(c[None], first=1)) == ERR_ARG
    over = pkg.cuda_api.DeviceLayer(nx, ny, 1e10, 0.1)   # global_res * cost overflows
    over.reserve_maps(1)
    c = costs[0].copy()
    c[5, 5] = 1e300
    assert _code(pkg, lambda: over.set_maps(c)) == ERR_ARG
    over.close()
    assert _code(pkg, lambda: dev.set_maps(costs[:1], first=3)) == ERR_ARG
    assert _code(pkg, lambda: dev.set_maps(costs[:2], first=2)) == ERR_ARG
    assert _code(pkg, lambda: dev.solve_maps(goals[:4])) == ERR_ARG
    dev.set_maps(costs[:1])
    assert _code(pkg, lambda: dev.solve_maps(goals[:2])) == ERR_STATE   # map 1: NaN above, never set
    dev.set_maps(costs[1:3], first=1)
    assert dev.solve_maps(goals[:3])["converged"]
    dev.set_anisotropy([-10.0, 10.0], [0.8, 1.5])
    assert _code(pkg, lambda: dev.solve_maps(goals[:3])) == ERR_STATE
    dev.set_anisotropy([], [])
    dev.set_obstacle_clearance(1.0, 2.0, 1.0)
    assert _code(pkg, lambda: dev.solve_maps(goals[:3])) == ERR_STATE
    assert _code(pkg, lambda: pkg.cuda_api.batch_solve_maps([dev], costs[:3], goals[:3])) == ERR_STATE
    dev.set_obstacle_clearance(0.0, 0.0, 0.0)
    assert dev.solve_maps(goals[:3])["converged"]
    dev.reserve_maps(0)
    assert _code(pkg, lambda: dev.solve_maps(goals[:1])) == ERR_ARG


# ---- 8. several contexts ------------------------------------------------------------------------
def _check_batch(pkg, layers, n_maps, ny, nx, seed):
    costs, goals, _ = _batch(pkg, ny, nx, n_maps, seed=seed)
    starts = [_goal(pkg, costs[q], 0.15, 0.85) for q in range(n_maps)]
    paths, T, ms = pkg.cuda_api.batch_solve_maps(layers, costs, goals, starts=starts, total_cost=True)
    assert len(ms) == len(layers) and (ms > 0).all()
    for q in range(n_maps):
        Ts, _, (ps, ss) = _solo(pkg, costs[q], goals[q], starts[q])
        _same(T[q], Ts)
        p, s = paths[q]
        assert s == ss and p.shape == ps.shape, q
        if len(ps):
            assert np.max(np.abs(p[:, :2] - ps[:, :2])) <= 1e-3


def test_batch_solve_maps_three_contexts(pkg):
    ny, nx = 140, 150
    layers = [pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1) for _ in range(3)]
    for d, r in zip(layers, (2, 3, 1)):
        d.reserve_maps(r)
    _check_batch(pkg, layers, 11, ny, nx, seed=12)   # blocks 4/4/3 in chunks of 2, 3 and 1


def test_batch_solve_maps_two_gpus(pkg):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ny, nx = 200, 180
    layers = [pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1, device=k) for k in range(2)]
    for d in layers:
        d.reserve_maps(4)
    _check_batch(pkg, layers, 9, ny, nx, seed=13)
