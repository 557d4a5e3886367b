"""Map batches under obstacle clearance and slope anisotropy (dymu_set_maps_clearance /
dymu_set_maps_anisotropy): every map of a batch against a freshly created context that solves that map
alone with the same settings, against the plain-C anisotropic restatement and exact corridors, paths on
anisotropic map slots, the lifecycle of the settings, isolation, errors and the multi-context driver."""
import math

import numpy as np
import pytest

import clearance_model as cm
from conftest import rel_err

pytestmark = pytest.mark.gpu

ERR_ARG, ERR_STATE = -2, -3
TABLE = ([-20.0, -5.0, 0.0, 10.0, 25.0], [0.6, 0.8, 1.0, 1.8, 3.5])   # DESIGN.md section 10
NEAR, FAR = (1.0, 2.0, 1.5), (3.0, 37.0, 2.0)    # R = 3 / 40 cells at global_res 1


@pytest.fixture(scope="module")
def orc_aniso():
    """The plain-C restatement of the anisotropic model (built on first use)."""
    import oracle_aniso
    return oracle_aniso


def _ceff(cost, g=1.0):
    """C_eff of a fresh context after dymu_set_cost_map(cost)."""
    with np.errstate(over="ignore"):
        return np.where(cost <= 0, np.inf, g * cost * (2 + 0.0 - 1.0))


def _goal(pkg, cost, fi, fj):
    ny, nx = cost.shape
    return pkg.synthetic.free_interior_cell_near(cost <= 0, int(fi * nx), int(fj * ny))


def _maps(pkg, ny, nx, n, seed):
    """n maps and goals: map 1 scaled x100, map 2 with its goal on an obstacle, map 3 with an obstacle
    next to its goal (the goal lies inside the lethal ring of any radius >= global_res)."""
    rng = np.random.default_rng(seed)
    costs = np.stack([pkg.synthetic.smooth_cost_map(ny, nx, seed=seed * 100 + q) for q in range(n)])
    goals = [_goal(pkg, costs[q], rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8)) for q in range(n)]
    costs[1] *= 100.0
    gi, gj = goals[2]
    costs[2, gj, gi] = 0.0
    gi, gj = goals[3]
    costs[3, gj, gi + 1] = 0.0
    return costs, goals


def _layer(pkg, nx, ny, g, elev=None, clear=None, table=None, n_maps=0, device=-1):
    dev = pkg.cuda_api.DeviceLayer(nx, ny, g, 0.1, device=device)
    if elev is not None:
        dev.upload_plane("elevation", elev)
    if clear is not None:
        dev.set_maps_clearance(*clear)
    if table is not None:
        dev.set_maps_anisotropy(*table)
    if n_maps:
        dev.reserve_maps(n_maps)
    return dev


def _solo(pkg, cost, goal, g=1.0, elev=None, clear=None, table=None, start=None):
    """The equivalence: elevation, dymu_set_cost_map, clearance, anisotropy, dymu_solve_total_cost."""
    ny, nx = cost.shape
    dev = pkg.cuda_api.DeviceLayer(nx, ny, g, 0.1)
    try:
        if elev is not None:
            dev.upload_plane("elevation", elev)
        dev.set_cost_map(cost)
        if clear is not None:
            dev.set_obstacle_clearance(*clear)
        if table is not None:
            dev.set_anisotropy(*table)
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


def _same_path(a, b, tol=1e-3):
    (pa, sa), (pb, sb) = a, b
    assert sa == sb and pa.shape == pb.shape
    if len(pb):
        assert np.max(np.abs(pa[:, :2] - pb[:, :2])) <= tol


def _check_against_solo(pkg, dev, costs, goals, g, elev, clear, table):
    for q in range(len(costs)):
        Tb = dev.download_total_cost(slot=q)
        Ts, sts, _ = _solo(pkg, costs[q], goals[q], g, elev, clear, table)
        _same(Tb, Ts)
        if q == 2:
            assert sts["goal_obstacle"] == 1 and not np.isfinite(Tb).any()
        else:
            assert Tb[goals[q][1], goals[q][0]] == 0.0
        if q == 3:
            assert sts["goal_obstacle"] == 0   # next to an obstacle, inside any lethal ring: seeded


SHAPES = [(129, 257, 1.0, NEAR), (129, 257, 0.7, NEAR), (129, 257, 1.0, FAR), (512, 512, 1.0, NEAR),
          (512, 512, 0.7, (2.0, 26.0, 2.0))]


# ---- 1. clearance --------------------------------------------------------------------------------
@pytest.mark.parametrize("ny,nx,g,clear", SHAPES)
def test_clearance_batch_equals_solo(pkg, ny, nx, g, clear):
    n = 6
    costs, goals = _maps(pkg, ny, nx, n, seed=ny + nx + int(10 * g))
    dev = _layer(pkg, nx, ny, g, clear=clear, n_maps=n)
    dev.set_maps(costs)
    st = dev.solve_maps(goals)
    assert st["converged"] and st["goal_obstacle"] == 1
    _check_against_solo(pkg, dev, costs, goals, g, None, clear, None)


# ---- 2. anisotropy ---------------------------------------------------------------------------------
@pytest.mark.parametrize("ny,nx,g", [(129, 257, 1.0), (129, 257, 0.7), (512, 512, 1.0)])
def test_anisotropy_batch_equals_solo(pkg, ny, nx, g):
    n = 6
    costs, goals = _maps(pkg, ny, nx, n, seed=ny + 3 * nx + int(10 * g))
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=ny + nx)
    dev = _layer(pkg, nx, ny, g, elev=elev, table=TABLE, n_maps=n)
    dev.set_maps(costs)
    st = dev.solve_maps(goals)
    assert st["converged"] and st["goal_obstacle"] == 1
    _check_against_solo(pkg, dev, costs, goals, g, elev, None, TABLE)


def test_anisotropy_against_oracle(pkg, orc_aniso):
    ny, nx, n = 129, 257, 4
    costs, goals = _maps(pkg, ny, nx, n, seed=21)
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=22)
    dev = _layer(pkg, nx, ny, 1.0, elev=elev, table=TABLE, n_maps=n)
    dev.set_maps(costs)
    assert dev.solve_maps(goals)["converged"]
    q = 1
    A = orc_aniso.aniso_dircost(elev, _ceff(costs[q]), 1.0, *TABLE)
    T_orc = orc_aniso.aniso_march(A, goals[q])
    _same(dev.download_total_cost(slot=q), T_orc, 1e-9)


# ---- 3. both ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("ny,nx,g,clear", [(129, 257, 0.7, NEAR), (300, 200, 1.0, (4.0, 6.0, 1.0))])
def test_clearance_and_anisotropy_batch_equals_solo(pkg, ny, nx, g, clear):
    n = 5
    costs, goals = _maps(pkg, ny, nx, n, seed=nx + 7)
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=nx + 8)
    dev = _layer(pkg, nx, ny, g, elev=elev, clear=clear, table=TABLE, n_maps=n)
    dev.set_maps(costs)
    st = dev.solve_maps(goals)
    assert st["converged"] and st["goal_obstacle"] == 1
    _check_against_solo(pkg, dev, costs, goals, g, elev, clear, TABLE)


# ---- 4. exact corridors ---------------------------------------------------------------------------
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


def _snake_T(cost, C):
    """Running sum of the cost term C along the snake from cell (0, 0) in the order of the update."""
    ny, nx = cost.shape
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


def test_margin_corridor_is_exact(pkg):
    torch = pytest.importorskip("torch")
    ny, nx, n, g = 97, 131, 4, 0.7
    margin, penalty = 2.5, 1.75      # radius 0: only the penalty margin, which covers every corridor cell
    rng = np.random.default_rng(9)
    snakes = np.stack([_snake(ny, nx, rng) for _ in range(n)])
    snakes[1] *= 100.0
    ld, rows = nx + 3, ny + 2
    big = torch.full((n, rows, ld), float("nan"), dtype=torch.float64, device="cuda:0")
    big[:, :ny, :nx] = torch.from_numpy(snakes).to("cuda:0")
    torch.cuda.synchronize()
    a = _layer(pkg, nx, ny, g, clear=(0.0, margin, penalty), n_maps=n, device=0)
    b = _layer(pkg, nx, ny, g, clear=(0.0, margin, penalty), n_maps=n, device=0)
    a.set_maps(snakes)
    b.set_maps_device(big.data_ptr(), n, ld, rows * ld)
    goals = [(0, 0)] * n
    for d in (a, b):
        assert d.solve_maps(goals)["converged"]
    for q in range(n):
        ob = snakes[q] <= 0
        dist = cm.clearance(ob, 0.0, margin, g)
        C = cm.ceff(cm.plain_ceff(snakes[q], np.zeros_like(dist), np.ones_like(dist), ob, g), dist, 0.0, margin, penalty)
        assert (C[~ob] > _ceff(snakes[q], g)[~ob]).all()   # the margin scaled every corridor cell
        Ta, Tb = a.download_total_cost(slot=q), b.download_total_cost(slot=q)
        assert np.array_equal(Ta, Tb), q
        assert np.array_equal(Ta, _snake_T(snakes[q], C)), q


def test_anisotropic_corridor_is_exact_and_asymmetric(pkg):
    n, slope = 64, 10.0
    table = ([-20.0, 0.0, 20.0], [0.5, 1.0, 3.0])
    cs, goals = (0.7, 1.3), [(30, 1), (18, 1)]
    costs = np.zeros((2, 3, n))
    for q, c in enumerate(cs):
        costs[q, 1, :] = c
    elev = np.tile(np.arange(n, dtype=np.float64) * math.tan(math.radians(slope)), (3, 1))
    dev = _layer(pkg, n, 3, 1.0, elev=elev, table=table, n_maps=2)
    dev.set_maps(costs)
    assert dev.solve_maps(goals)["converged"]
    th = math.degrees(math.atan(math.tan(math.radians(slope))))
    for q, c in enumerate(cs):
        up, down = c * np.interp(th, *table), c * np.interp(-th, *table)
        goal = goals[q][0]
        expect = np.zeros(n)
        for i in range(goal + 1, n):
            expect[i] = expect[i - 1] + down
        for i in range(goal - 1, -1, -1):
            expect[i] = expect[i + 1] + up
        T = dev.download_total_cost(slot=q)
        assert rel_err(T[1], expect) <= 1e-12
        Ts, _, _ = _solo(pkg, costs[q], goals[q], 1.0, elev, None, table)
        assert np.array_equal(T, Ts), q   # the same directional costs, summed in the same order


# ---- 5. paths ---------------------------------------------------------------------------------------
def test_paths_on_anisotropic_map_slots(pkg):
    ny, nx, n = 300, 200, 6
    costs, goals = _maps(pkg, ny, nx, n, seed=7)
    starts = [_goal(pkg, costs[q], 0.1 + 0.15 * q, 0.9 - 0.1 * q) for q in range(n)]
    xy = [(float(i), float(j)) for i, j in starts]
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=5)
    clear = (1.0, 2.0, 1.0)
    dev = _layer(pkg, nx, ny, 1.0, elev=elev, clear=clear, table=TABLE, n_maps=n)
    dev.set_maps(costs)
    dev.solve_maps(goals)
    paths, status = dev.extract_global_path_batch(list(range(n)), xy, 0.4, goals, cap=1 << 14)
    solo = [_solo(pkg, costs[q], goals[q], 1.0, elev, clear, TABLE, starts[q])[2] for q in range(n)]
    for q in range(n):
        _same_path((paths[q], status[q]), solo[q])
        _same_path(dev.extract_global_path(*xy[q], 0.4, *goals[q], slot=q, cap=1 << 14), solo[q])
    # isotropic map solves of all six, then an anisotropic one of the first three: one batch call on
    # marked (0, 1) and unmarked (3, 4) slots
    dev.set_maps_anisotropy([], [])
    dev.solve_maps(goals)
    dev.set_maps_anisotropy(*TABLE)
    dev.solve_maps(goals[:3])
    mixed = [0, 3, 1, 4]
    paths, status = dev.extract_global_path_batch(mixed, [xy[s] for s in mixed], 0.4, [goals[s] for s in mixed],
                                                  cap=1 << 14)
    for k, s in enumerate(mixed):
        want = solo[s] if s < 3 else _solo(pkg, costs[s], goals[s], 1.0, elev, clear, None, starts[s])[2]
        _same_path((paths[k], status[k]), want)
    # map 1 set again: its slot no longer matches the planes the descent would read
    dev.set_maps(costs[1:2], first=1)
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        dev.extract_global_path(*xy[1], 0.4, *goals[1], slot=1)
    assert e.value.code == ERR_STATE
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        dev.extract_global_path_batch([0, 1], xy[:2], 0.4, goals[:2])
    assert e.value.code == ERR_STATE
    _same_path(dev.extract_global_path(*xy[0], 0.4, *goals[0], slot=0, cap=1 << 14), solo[0])
    # the context's own solve takes slot 0 back, with the context's own (isotropic) descent
    own = pkg.synthetic.smooth_cost_map(ny, nx, seed=70)
    dev.set_cost_map(own)
    g0, s0 = _goal(pkg, own, 0.7, 0.3), _goal(pkg, own, 0.2, 0.8)
    dev.solve_total_cost([g0])
    _same_path(dev.extract_global_path(float(s0[0]), float(s0[1]), 0.4, *g0, cap=1 << 14),
               _solo(pkg, own, g0, 1.0, elev, None, None, s0)[2])


# ---- 6. lifecycle of the settings ---------------------------------------------------------------
def test_settings_apply_at_solve_time(pkg):
    ny, nx, n, g = 160, 224, 4, 1.0
    costs, goals = _maps(pkg, ny, nx, n, seed=31)
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=32)

    def fresh(clear, table):
        d = _layer(pkg, nx, ny, g, elev=elev, clear=clear, table=table, n_maps=n)
        d.set_maps(costs)
        launches = d.launches
        d.solve_maps(goals)
        return [d.download_total_cost(slot=q) for q in range(n)], d.launches - launches

    dev = _layer(pkg, nx, ny, g, elev=elev, clear=NEAR, n_maps=n)
    dev.set_maps(costs)
    dev.solve_maps(goals)
    for clear, table in (((2.0, 3.0, 0.5), None), ((2.0, 3.0, 0.5), TABLE), (None, TABLE), (None, None)):
        dev.set_maps_clearance(*(clear or (0.0, 0.0, 0.0)))
        dev.set_maps_anisotropy(*(table or ([], [])))
        launches = dev.launches
        dev.solve_maps(goals)
        used = dev.launches - launches
        want, want_used = fresh(clear, table)
        for q in range(n):
            _same(dev.download_total_cost(slot=q), want[q], 1e-13)
        if clear is None and table is None:
            assert used == want_used      # both off: the launches of a context that never had them
    # a clearance change rebuilds every map; a map set again is rebuilt without touching the others
    dev.set_maps_clearance(*FAR)
    dev.solve_maps(goals)
    costs2 = costs.copy()
    costs2[2] = pkg.synthetic.smooth_cost_map(ny, nx, seed=99)
    dev.set_maps(costs2[2:3], first=2)
    dev.solve_maps(goals)
    for q in range(n):
        _same(dev.download_total_cost(slot=q), _solo(pkg, costs2[q], goals[q], g, None, FAR, None)[0])


# ---- 7. isolation ---------------------------------------------------------------------------------
def test_context_state_is_untouched(pkg):
    torch = pytest.importorskip("torch")
    ny, nx, n = 160, 224, 4
    own = pkg.synthetic.smooth_cost_map(ny, nx, seed=77)
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=78)
    goal = _goal(pkg, own, 0.5, 0.5)
    dev = _layer(pkg, nx, ny, 1.0, elev=elev)
    dev.set_cost_map(own)
    dev.solve_total_cost([goal])
    before = {p: dev.download_plane(p) for p in ("elevation", "cost", "ceff", "hazard_density", "trafficability")}
    ob = dev.download_plane_u8("obstacle")
    pinned = torch.empty((ny, nx), dtype=torch.float64).pin_memory()
    buf = pinned.numpy()
    assert dev.set_total_cost_export(buf)
    costs, goals = _maps(pkg, ny, nx, n, seed=8)
    dev.set_maps_clearance(*NEAR)
    dev.set_maps_anisotropy(*TABLE)
    dev.reserve_maps(n)
    dev.set_maps(costs)
    buf[:] = 12345.0
    dev.solve_maps(goals)
    dev.synchronize()
    assert (buf == 12345.0).all()
    for p, v in before.items():
        assert np.array_equal(dev.download_plane(p), v), p
    assert np.array_equal(dev.download_plane_u8("obstacle"), ob)
    for p in ("clearance", "dircost_xm"):   # the context's own planes of those features stay off
        with pytest.raises(pkg.cuda_api.DymuError):
            dev.download_plane(p)
    dev.set_total_cost_export(None)
    dev.solve_total_cost([goal])
    _same(dev.download_total_cost(), _solo(pkg, own, goal, 1.0, elev)[0], 1e-13)


# ---- 8. errors ---------------------------------------------------------------------------------------
def _code(pkg, call):
    with pytest.raises(pkg.cuda_api.DymuError) as e:
        call()
    return e.value.code


def test_errors(pkg):
    ny, nx = 64, 80
    dev = _layer(pkg, nx, ny, 1.0, n_maps=2)
    for bad in ((-1.0, 1.0, 1.0), (1.0, np.nan, 1.0), (1.0, 1.0, np.inf), (1.0, 1.0, -0.5), (100.0, 29.0, 1.0)):
        assert _code(pkg, lambda: dev.set_maps_clearance(*bad)) == ERR_ARG
    for t, f in (([0.0], [1.0]), ([0.0, 0.0], [1.0, 1.0]), ([-1.0, 1.0], [1.0, 0.0]), ([-1.0, 1.0], [1.0, np.inf]),
                 ([-1.0, np.nan], [1.0, 1.0]), (list(range(65)), [1.0] * 65)):
        assert _code(pkg, lambda: dev.set_maps_anisotropy(t, f)) == ERR_ARG
    with pytest.raises(ValueError):
        dev.set_maps_anisotropy([0.0, 1.0], [1.0])
    # a refused setting leaves the batch settings as they were (off)
    costs, goals = _maps(pkg, ny, nx, 4, seed=2)
    dev.set_maps(costs[:2])
    assert dev.solve_maps(goals[:2])["converged"]
    _same(dev.download_total_cost(slot=1), _solo(pkg, costs[1], goals[1])[0])
    # contexts of one driver call solve with the same batch settings
    other = _layer(pkg, nx, ny, 1.0, n_maps=2)
    dev.set_maps_clearance(*NEAR)
    assert _code(pkg, lambda: pkg.cuda_api.batch_solve_maps([dev, other], costs, goals)) == ERR_ARG
    other.set_maps_clearance(1.0, 2.0, 1.25)
    assert _code(pkg, lambda: pkg.cuda_api.batch_solve_maps([dev, other], costs, goals)) == ERR_ARG
    other.set_maps_clearance(*NEAR)
    other.set_maps_anisotropy(*TABLE)
    assert _code(pkg, lambda: pkg.cuda_api.batch_solve_maps([dev, other], costs, goals)) == ERR_ARG
    dev.set_maps_anisotropy(TABLE[0], TABLE[1][:-1] + [3.0])
    assert _code(pkg, lambda: pkg.cuda_api.batch_solve_maps([dev, other], costs, goals)) == ERR_ARG
    dev.set_maps_anisotropy(*TABLE)
    pkg.cuda_api.batch_solve_maps([dev, other], costs, goals)
    # the context's own clearance still refuses map solves, whatever the batch settings
    dev.set_obstacle_clearance(1.0, 2.0, 1.0)
    assert _code(pkg, lambda: dev.solve_maps(goals[:2])) == ERR_STATE


# ---- 9. several contexts ------------------------------------------------------------------------
def _check_driver(pkg, layers, n_maps, ny, nx, elev, seed):
    clear = (1.0, 2.0, 1.0)
    for d in layers:
        d.upload_plane("elevation", elev)
        d.set_maps_clearance(*clear)
        d.set_maps_anisotropy(*TABLE)
    costs, goals = _maps(pkg, ny, nx, n_maps, seed=seed)
    starts = [_goal(pkg, costs[q], 0.15, 0.85) for q in range(n_maps)]
    paths, T, ms = pkg.cuda_api.batch_solve_maps(layers, costs, goals, starts=starts, total_cost=True)
    assert len(ms) == len(layers) and (ms > 0).all()
    for q in range(n_maps):
        Ts, _, path = _solo(pkg, costs[q], goals[q], 1.0, elev, clear, TABLE, starts[q])
        _same(T[q], Ts)
        _same_path(paths[q], path)


def test_batch_solve_maps_three_contexts(pkg):
    ny, nx = 140, 150
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=12)
    layers = [pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1) for _ in range(3)]
    for d, r in zip(layers, (2, 3, 1)):
        d.reserve_maps(r)
    _check_driver(pkg, layers, 11, ny, nx, elev, seed=12)   # blocks 4/4/3 in chunks of 2, 3 and 1


def test_batch_solve_maps_two_gpus(pkg):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ny, nx = 200, 180
    elev, _ = pkg.synthetic.mars_dem(ny, nx, seed=13)
    layers = [pkg.cuda_api.DeviceLayer(nx, ny, 1.0, 0.1, device=k) for k in range(2)]
    for d in layers:
        d.reserve_maps(4)
    _check_driver(pkg, layers, 9, ny, nx, elev, seed=13)
